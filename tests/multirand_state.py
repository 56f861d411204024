"""Whole-state access to the oracle's multirand generator (oracle/oracle.py MultiRand) for the device-stream tests, and
the helpers those tests share.

The oracle exposes only multirand_seeds(0:3) (KISS64).  SuperKISS64 and MT19937-64 need all of multirand_seeds and the
table / block position, and the Maxwellian loaders the one-slot buffer of gaussian_array, so this reads and writes them
in the oracle's generator object directly: `struct orc_multirand` (oracle/multirand_oracle.c) is
`uint64_t seeds[20635]; int iseed; int al_int; int gauss_filled; double gauss_buf`.  `_check_layout` and
`_check_spare_layout` pin that layout against the oracle's own accessor, its default seeding and gaussian_array before
any test relies on it."""
import ctypes as C
import subprocess

import numpy as np

from oracle import oracle as O

NSEED = 20635
_ISEED_OFFSET = NSEED * 8
_AL_OFFSET = NSEED * 8 + 4
_FILLED_OFFSET = NSEED * 8 + 8
_BUF_OFFSET = NSEED * 8 + 16
_checked = False
_spare_checked = False


def _check_layout():
    global _checked
    if _checked:
        return
    for al, iseed in ((3, 20632), (2, 312), (1, 0)):   # default seeding leaves these table positions (:476-518)
        g = O.MultiRand()
        g.seed_default(al)
        addr = g.g.value
        words = np.ctypeslib.as_array((C.c_uint64 * NSEED).from_address(addr))
        assert [int(w) for w in words[:4]] == g.seeds4(), "orc_multirand no longer starts with seeds[]"
        assert C.c_int.from_address(addr + _ISEED_OFFSET).value == iseed, "orc_multirand.iseed moved"
    _checked = True


def _check_spare_layout():
    global _spare_checked
    if _spare_checked:
        return
    for al in (1, 2, 3):
        g = O.MultiRand()
        g.seed_default(al)
        addr = g.g.value
        assert C.c_int.from_address(addr + _AL_OFFSET).value == al, "orc_multirand.al_int moved"
        assert C.c_int.from_address(addr + _FILLED_OFFSET).value == 0
        ref = O.MultiRand()
        ref.seed_default(al)
        pair = ref.gaussian_array(2)
        g.gaussian_array(1)   # odd length: the second value of the pair stays buffered
        assert C.c_int.from_address(addr + _FILLED_OFFSET).value == 1, "orc_multirand.gauss_filled moved"
        assert C.c_double.from_address(addr + _BUF_OFFSET).value == pair[1], "orc_multirand.gauss_buf moved"
    _spare_checked = True


def get_state(g: "O.MultiRand"):
    """(multirand_seeds(0:20634) as a uint64 array, table position)."""
    _check_layout()
    addr = g.g.value
    seeds = np.ctypeslib.as_array((C.c_uint64 * NSEED).from_address(addr)).copy()
    return seeds, C.c_int.from_address(addr + _ISEED_OFFSET).value


def set_state(g: "O.MultiRand", seeds, iseed: int):
    """Overwrite the state; the engine chosen by seed_default / init_const stays."""
    _check_layout()
    a = np.ascontiguousarray(seeds, dtype=np.uint64)
    assert a.size == NSEED
    addr = g.g.value
    C.memmove(addr, a.ctypes.data, NSEED * 8)
    C.c_int.from_address(addr + _ISEED_OFFSET).value = int(iseed)


def get_spare(g: "O.MultiRand"):
    """(gauss_filled, gauss_buf): the one-slot buffer of gaussian_array."""
    _check_spare_layout()
    addr = g.g.value
    return C.c_int.from_address(addr + _FILLED_OFFSET).value, C.c_double.from_address(addr + _BUF_OFFSET).value


def to_real(i):
    """INT2REAL64 of a 64-bit generator output (the reference's known-answer vectors hold the integers)."""
    return float(np.int64(i)) / 18446744073709551615.0 + 0.5


def ulps(a, b):
    """Elementwise distance in units in the last place (as ordered integers)."""
    def key(x):
        i = np.asarray(x, dtype=np.float64).view(np.int64)
        return np.where(i < 0, np.int64(-0x8000000000000000) - i, i)
    return np.abs(key(a) - key(b))


def run_host(exe, tmp_path, tag, args):
    """Run the C++ host driver with markers_out: (stdout, marker count, {x, v, p, w})."""
    mk = tmp_path / f"markers_{tag}.bin"
    r = subprocess.run([exe, *args, f"out={tmp_path / f'energy_{tag}.txt'}", f"markers_out={mk}"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    raw = np.fromfile(mk, dtype=np.float64)
    n = int(np.frombuffer(raw[:1].tobytes(), dtype=np.int64)[0])
    return r.stdout, n, dict(zip(("x", "v", "p", "w"), raw[1:].reshape(4, n)))
