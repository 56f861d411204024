"""Whole-state access to the oracle's multirand generator (oracle/oracle.py MultiRand) for the SuperKISS64 tests.

The oracle exposes only multirand_seeds(0:3) (KISS64).  SuperKISS64 needs all of multirand_seeds(0:20634) and the table
position, so this reads and writes them in the oracle's generator object directly: `struct orc_multirand`
(oracle/multirand_oracle.c) starts with `uint64_t seeds[20635]` followed by `int iseed`.  `_check_layout` pins that
layout against the oracle's own accessor and its default seeding before any test relies on it."""
import ctypes as C

import numpy as np

from oracle import oracle as O

NSEED = 20635
_ISEED_OFFSET = NSEED * 8
_checked = False


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
