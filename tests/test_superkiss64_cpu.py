"""The product's SuperKISS64 (pic1dp_b200/csrc/rng_kernels.cuh, the code the device runs, here through its host entry
points) against the reference's known-answer vectors (/root/reference/src/multirand.F90:414-425) and the KAT-pinned
oracle's sequential stream, and the device's refill algorithm -- a scan over the 2-bit carry maps of chunks of the
table, then an element-wise rewrite -- against the sequential refill, bit for bit."""
import json
import os

import numpy as np
import pytest

from multirand_state import get_state, set_state
from oracle import oracle as O
from pic1dp_b200 import host as H

GOLD = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "multirand_kat.json")))
N = 20632
M64 = (1 << 64) - 1


def _to_real(i):
    return float(np.int64(i)) / 18446744073709551615.0 + 0.5   # INT2REAL64, :49


def _default_state():
    g = O.MultiRand()
    g.seed_default(3)          # the self test's seeds, :513-515
    return get_state(g)


def test_known_answer_head_and_tail():
    seeds, iseed = _default_state()
    u, pos = H.host_superkiss64_fill(seeds, iseed, N + 5)
    assert [float(t) for t in u[:10]] == [_to_real(i) for i in GOLD["superkiss64_head"]]
    # positions 20627 .. 20636 cross the second refill
    assert [float(t) for t in u[N - 5:N + 5]] == [_to_real(i) for i in GOLD["superkiss64_tail"]]
    assert pos == 5


@pytest.mark.parametrize("mype", [0, 1, 2, 3])
def test_stream_and_state_equal_the_oracle_after_init(mype):
    g = O.MultiRand()
    g.init_const(3, mype, 5)   # seed_type 1, warm-up 5: multirand_init as particle_load calls it
    seeds, iseed = get_state(g)
    assert iseed != 0 and iseed != N   # the warm-up leaves the table part-used
    for n in (7, 2 * N + 3, 100_003):
        got, iseed = H.host_superkiss64_fill(seeds, iseed, n)
        assert np.array_equal(got, g.real_array(n)), n
        want_seeds, want_iseed = get_state(g)
        assert iseed == want_iseed and np.array_equal(seeds, want_seeds), n


def _sequential_refill(seeds):
    """The oracle's refill: a draw at table position 20632 refills first (LCG / xorshift words are not compared)."""
    g = O.MultiRand()
    g.seed_default(3)
    set_state(g, seeds, N)
    g.int64()
    return get_state(g)[0]


def _h(q):
    return (q >> 23) + (q >> 25)


def _identity_chain(rng):
    """A table in which every carry map is the identity (b_i = b_{i-1}): the bit out of element 0 runs through the
    whole table, so every chunk of the scan depends on every chunk before it.  Element i needs H(Q[i-1]) odd and
    ((Q[i] << 41) >> 1) + ((Q[i] << 39) >> 1) + (H(Q[i-1]) >> 1) = 2^63 - 1; the high bits of Q[i] set H(Q[i]) = -1
    (mod 2^39) for the next element, the low 25 bits solve the equation."""
    words, hp = [], None
    while len(words) < N:
        t = (1 << 39) - 1 + (int(rng.integers(0, 3)) << 39)
        x = next((x for x in range(4 * t // 5 - 8, 4 * t // 5 + 9) if x + (x >> 2) == t), None)
        if x is None or x >= 1 << 41:
            continue
        if hp is None:
            low = int(rng.integers(0, 1 << 23))
        else:
            r = (((1 << 63) - 1 - (hp >> 1)) >> 38) - (x & 3) * (1 << 23)   # 5 (Q mod 2^23) + (bits 23, 24) 2^23
            if r % 5 or not 0 <= r // 5 < 1 << 23:
                continue
            low = r // 5
        q = ((x << 23) | low) & M64
        words.append(q)
        hp = _h(q)
    return np.array(words, dtype=np.uint64)


def _states():
    rng = np.random.default_rng(2024)
    out = []
    for _ in range(3):   # random tables and carries
        s = rng.integers(0, 1 << 63, N + 3, dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, N + 3, dtype=np.uint64)
        s[N] = np.uint64(int(rng.integers(0, 1 << 42)))
        out.append(("random", s))
    s = np.full(N + 3, M64, dtype=np.uint64)             # carry = 2^64 - 1, all-ones words: z wraps at element 0
    out.append(("ones_max_carry", s))
    s = np.zeros(N + 3, dtype=np.uint64)
    s[1:N:2] = np.uint64(M64)                            # alternating 0 / all-ones
    s[N] = np.uint64(M64)
    out.append(("alternating", s))
    for c in (0, 1, 2, 3, M64):                          # the identity chain with both bits into element 0
        s = np.zeros(N + 3, dtype=np.uint64)
        s[:N] = _identity_chain(np.random.default_rng(7))
        s[N] = np.uint64(c)
        out.append((f"identity_chain_c{c:x}", s))
    return out


STATES = _states()


@pytest.mark.parametrize("name,state", STATES, ids=[n for n, _ in STATES])
@pytest.mark.parametrize("nchunks", [1024, 1, 2, 31, 32, 33, 983, 4096, N])   # 1024: the kernel's chunking
def test_chunked_map_scan_refill_equals_sequential_refill(name, state, nchunks):
    seq, chunked = state.copy(), state.copy()
    for k in range(3):   # consecutive refills
        seq = _sequential_refill(seq)
        H.host_superkiss64_refill(chunked, nchunks)
        assert np.array_equal(chunked[:N + 1], seq[:N + 1]), (name, nchunks, k)


def test_identity_chain_propagates_the_carry_bit():
    """The adversarial table really is one: two carries that differ in the bit into element 0 change every word."""
    a = np.zeros(N + 3, dtype=np.uint64)
    a[:N] = _identity_chain(np.random.default_rng(7))
    b = a.copy()
    q0 = int(a[0])
    base = ((((q0 << 41) & M64) >> 1) + (((q0 << 39) & M64) >> 1)) & M64
    a[N], b[N] = np.uint64(0), np.uint64(M64 - 1)       # carry >> 1 = 0 and 2^63 - 1: z_0 = base, base + 2^63 - 1
    assert (base >> 63) != (((base + (1 << 63) - 1) & M64) >> 63)
    ra, rb = _sequential_refill(a), _sequential_refill(b)
    assert np.all(ra[1:N] != rb[1:N])


def test_bad_arguments_are_rejected():
    seeds, _ = _default_state()
    for iseed in (-1, N + 1):
        with pytest.raises(H.Pic1dpError):
            H.host_superkiss64_fill(seeds, iseed, 4)
    with pytest.raises(H.Pic1dpError):
        H.host_superkiss64_refill(seeds, 0)
