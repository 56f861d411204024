"""The product's MT19937-64 jump (pic1dp_b200/csrc/rng_kernels.cuh, the window-XOR jump the device runs, here through
its host entry point) and the jump tables the build generates (tools_py3/gen_mt_jump.py into the build directory)
against the KAT-pinned oracle's sequential generator (/root/reference/src/multirand.F90:952-997)."""
import os
import sys

import numpy as np
import pytest

from multirand_state import get_state, set_state
from oracle import oracle as O
from pic1dp_b200 import build as B
from pic1dp_b200 import host as H

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools_py3"))
import gen_mt_jump  # noqa: E402

NN = 312


BUILT_TABLES = os.path.join(B.OBJDIR, B.MT_TABLES)


def test_library_is_built_from_the_generated_tables():
    with open(BUILT_TABLES) as f:
        assert f.read() == gen_mt_jump.render()


def _phi():
    with open(BUILT_TABLES) as f:
        text = f.read()
    body = text[text.index("mt_phi["):text.index("mt_jump_poly[")]
    words = [int(t.rstrip(",").rstrip("ULL"), 16) for t in body.split() if t.startswith("0x")]
    assert len(words) == NN
    return sum(w << (64 * q) for q, w in enumerate(words))


def test_phi_annihilates_the_oracle_stream():
    """sum over the set bits i of phi of output k + i is 0 for every k: the tempered outputs obey the recurrence the
    jump relies on (tempering is linear and invertible), from the first twisted block of the default seeding and from a
    rank's post-warm-up state."""
    phi = _phi()
    assert phi.bit_length() == 19938
    idx = np.array([i for i in range(19938) if (phi >> i) & 1])
    K = 3000
    for setup in (lambda g: g.seed_default(2), lambda g: g.init_const(2, 1, 5)):
        g = O.MultiRand()
        setup(g)
        y = np.array([g.int64() for _ in range(19938 + K)], dtype=np.int64).view(np.uint64)
        for k in range(K):
            assert np.bitwise_xor.reduce(y[idx + k]) == 0, k


def _start(kind):
    g = O.MultiRand()
    if kind == "default":
        g.seed_default(2)                # the raw seed block, iseed = 312
    elif kind.startswith("rank"):
        g.init_const(2, int(kind[4:]), 5)   # multirand_init as particle_load calls it (iseed = 312 after the warm-up)
    else:
        g.init_const(2, 2, 5)
        g.skip(int(kind[3:]))            # a part-used block
    return g


@pytest.mark.parametrize("kind", ["default", "rank0", "rank3", "mid1", "mid100", "mid311"])
def test_host_jump_lands_where_the_sequential_generator_does(kind):
    """pic1dp_host_mt19937_64_jump by n equals n sequential draws: the whole state (multirand_seeds(0:311), iseed)
    bitwise, then the same stream from both."""
    for n in (0, 1, 311, 312, 313, 1_000_003, 100_000_000):
        g = _start(kind)
        seeds, iseed = get_state(g)
        mt = seeds[:NN].copy()
        pos = H.host_mt19937_64_jump(mt, iseed, n)
        g.skip(n)
        want, want_pos = get_state(g)
        assert pos == want_pos and np.array_equal(mt, want[:NN]), (kind, n)
        if n == 0:
            assert pos == iseed and np.array_equal(mt, seeds[:NN])
        h = O.MultiRand()
        h.seed_default(2)
        full = want.copy()
        full[:NN] = mt
        set_state(h, full, pos)
        assert [h.int64() for _ in range(700)] == [g.int64() for _ in range(700)], (kind, n)


def test_host_jump_refuses_bad_state():
    g = _start("rank0")
    seeds, _ = get_state(g)
    mt = seeds[:NN].copy()
    for pos, n in ((-1, 5), (NN + 1, 5), (0, -1)):
        with pytest.raises(H.Pic1dpError):
            H.host_mt19937_64_jump(mt, pos, n)
    assert np.array_equal(mt, seeds[:NN])
