"""Maxwellian markers (input_imarker = 1) with both of particle_load's streams generated on the device:
multirand_gaussian_array(pv) (Marsaglia's polar method, src/multirand.F90:838-872) and then multirand_real_array(px), for
KISS64 (multirand_al_int = 1) and SuperKISS64 (al_int = 3).  Checked against the KAT-pinned oracle: the x stream and the
returned generator state exactly, the Gaussian values to a few ulp (the device log is not glibc's), the one-slot
Gaussian buffer across calls and species, refusals, and the C++ host driver with and without the device streams."""
import ctypes as C

import numpy as np
import pytest

import pic1dp_b200 as P
from pic1dp_b200 import _capi
from helpers import make_params
from multirand_state import get_spare, get_state, run_host, ulps
from oracle import oracle as O

pytestmark = pytest.mark.gpu
N_TABLE = 20632

class Stream:
    """The device loader of one generator with its state threaded through, in the oracle's representation."""

    def __init__(self, al, oracle):
        self.al = al
        seeds, self.iseed = get_state(oracle)
        self.seeds = seeds.copy() if al == 3 else seeds[:4].copy()
        self.filled, self.buf = get_spare(oracle)

    def load(self, g, isp, np_, nlocal, ninit, **kw):
        if self.al == 3:
            self.iseed, self.filled, self.buf = g.load_markers_maxwellian_superkiss64(
                isp, np_, nlocal, self.seeds, self.iseed, self.filled, self.buf, ninit, **kw)
        else:
            self.filled, self.buf = g.load_markers_maxwellian_kiss64(isp, np_, nlocal, self.seeds, self.filled,
                                                                     self.buf, ninit, **kw)

    def assert_state_equals(self, oracle, what):
        seeds, iseed = get_state(oracle)
        filled, buf = get_spare(oracle)
        if self.al == 3:
            assert self.iseed == iseed and np.array_equal(self.seeds, seeds), what
        else:
            assert np.array_equal(self.seeds, seeds[:4]), what
        assert self.filled == filled, what
        if filled:
            assert ulps(self.buf, buf) <= 4, what


SIZES = (1, 2, 3, 16_001, 16_002, 16_003, 16_500, 10_000_001)


@pytest.mark.parametrize("al", [1, 3])
@pytest.mark.parametrize("mype", [0, 1, 2, 3])
@pytest.mark.parametrize("spare", [False, True])
def test_stream_and_state_equal_the_oracle(al, mype, spare):
    """v = the Gaussian stream (T = m = 1, v0 = 0) within 4 ulp of gaussian_array, x bitwise equal to x loaded from the
    real_array that follows it, and the state after both calls (generator words, table position, Gaussian buffer) equal to the
    oracle's -- from init_const, with or without a value buffered by an earlier gaussian_array(7)."""
    nmax = max(SIZES)
    _, gp = make_params(nx=64, capacity=nmax, iptcldist=0, imarker=1, temperature=[1.0], mass=[1.0], v0=[0.0])
    with P.Pic1dGpu(gp) as g:
        for n in SIZES:
            r = O.MultiRand()
            r.init_const(al, mype, 5)
            if spare:
                r.gaussian_array(7)
                assert get_spare(r)[0] == 1
            s = Stream(al, r)
            s.load(g, 0, n, n, n)
            got = g.get_markers(0)
            draws, rounds, regenerated = g.last_gaussian_load()
            # the same loader fed with the oracle's streams: x = u lx from the uniforms that follow the Gaussian call,
            # v = the Gaussian values themselves (T = m = 1, v0 = 0)
            gauss, uni = r.gaussian_array(n), r.real_array(n)
            g.load_markers_maxwellian(0, gauss, uni, n)
            want = g.get_markers(0)
            assert np.array_equal(want["v"], gauss)
            assert np.array_equal(got["x"], want["x"]), (n, "x")
            d = ulps(got["v"], gauss)
            assert d.max() <= 4, (n, int(d.max()))
            s.assert_state_equals(r, n)
            assert draws >= n - int(spare)
            if n == nmax:
                print(f"al_int={al} rank {mype} spare={spare}: {np.mean(d == 0):.6f} of v bitwise equal, max {d.max()} "
                      f"ulp, {draws} draws in {rounds} rounds, {regenerated} regenerated")
                assert rounds >= 3 and (rounds - 1) * _capi.GAUSS_ROUND_DRAWS < draws <= rounds * _capi.GAUSS_ROUND_DRAWS
                assert 0 <= regenerated < _capi.GAUSS_ROUND_DRAWS if al == 3 else regenerated == 0


@pytest.mark.parametrize("al", [1, 3])
def test_two_species_with_tails_equal_the_host_stream_load(al):
    """Two species in sequence, np < nlocal, odd nlocal (the buffered value crosses from one species to the next):
    x, p, w bitwise equal to load_markers_maxwellian fed with the oracle's host streams, v within 1e-15 of max |v|, the
    final state equal to the oracle's, no marker-sized upload, and the moments of a drifting Maxwellian."""
    nlocal, nps = 200_003, (150_001, 200_003)
    kw = dict(nx=256, capacity=nlocal, nspecies=2, charge=[-1.0, -1.0], mass=[1.1, 1.0], temperature=[1.3, 1.0],
              temperature2=[1.0, 1.0], density=[0.85, 0.9], v0=[2.5, -1.0], iptcldist=0, imarker=1)
    modes = dict(init_mode=(1, 3), init_cos=(2e-6, 0.0), init_sin=(1e-5, 3e-6))
    _, gp = make_params(**kw)
    r = O.MultiRand()
    r.init_const(al, 2, 5)
    s = Stream(al, r)
    with P.Pic1dGpu(gp) as g:
        for isp, np_ in enumerate(nps):
            gv, ux = r.gaussian_array(nlocal), r.real_array(nlocal)
            g.load_markers_maxwellian(isp, gv[:np_].copy(), ux[:np_].copy(), 2 * nlocal, **modes)
            want = g.get_markers(isp)
            h2d = g.counters().h2d_bytes
            s.load(g, isp, np_, nlocal, 2 * nlocal, **modes)
            assert g.counters().h2d_bytes - h2d < 1_000_000      # no marker-sized upload
            got = g.get_markers(isp)
            for k in ("x", "p", "w"):
                assert got[k].size == np_ and np.array_equal(got[k], want[k]), (isp, k)
            assert np.max(np.abs(got["v"] - want["v"])) <= 1e-15 * np.max(np.abs(want["v"])), isp
            s.assert_state_equals(r, isp)
            v0, T, m = kw["v0"][isp], kw["temperature"][isp], kw["mass"][isp]
            assert abs(np.mean(got["v"]) - v0) < 0.02 and abs(np.std(got["v"]) / np.sqrt(T / m) - 1.0) < 0.01


@pytest.mark.parametrize("al", [1, 3])
def test_refusals_leave_the_state_alone(al):
    """iptcldist != 0, nlocal < np, a table position out of range, NULL state and np > capacity are refused with
    EINVAL / ECAPACITY, and the caller's generator words, table position and Gaussian buffer are unchanged."""
    L = _capi.load()
    r = O.MultiRand()
    r.init_const(al, 0, 5)
    r.gaussian_array(7)
    seeds0, iseed0 = get_state(r)
    seeds = seeds0.copy() if al == 3 else seeds0[:4].copy()
    ref = seeds.copy()
    filled0, buf0 = get_spare(r)
    im, ic, isn = (C.c_int32 * 1)(1), (C.c_double * 1)(0.0), (C.c_double * 1)(1e-5)

    def call(g, np_, nlocal, iseed=iseed0, null_seeds=False):
        pos, filled, buf = C.c_int32(iseed), C.c_int32(filled0), C.c_double(buf0)
        sp = None if null_seeds else seeds.ctypes.data_as(C.POINTER(C.c_uint64))
        if al == 3:
            rc = L.pic1dp_gpu_load_markers_maxwellian_superkiss64(g._h, 0, np_, nlocal, 1000, sp, C.byref(pos),
                                                                  C.byref(filled), C.byref(buf), 1, im, ic, isn)
        else:
            rc = L.pic1dp_gpu_load_markers_maxwellian_kiss64(g._h, 0, np_, nlocal, 1000, sp, C.byref(filled),
                                                             C.byref(buf), 1, im, ic, isn)
        assert np.array_equal(seeds, ref) and pos.value == iseed and filled.value == filled0 and buf.value == buf0
        return rc

    _, gp3 = make_params(capacity=1000, iptcldist=3)
    with P.Pic1dGpu(gp3) as g:
        assert call(g, 100, 100) == _capi.EINVAL
    _, gp = make_params(capacity=1000, iptcldist=0, imarker=1)
    with P.Pic1dGpu(gp) as g:
        assert call(g, 100, 99) == _capi.EINVAL
        assert call(g, 100, 100, null_seeds=True) == _capi.EINVAL
        if al == 3:
            assert call(g, 100, 100, iseed=-1) == _capi.EINVAL
            assert call(g, 100, 100, iseed=N_TABLE + 1) == _capi.EINVAL
        assert call(g, 1001, 2000) == _capi.ECAPACITY


@pytest.mark.parametrize("al", [1, 3])
def test_cpp_host_driver_maxwellian_device_streams(tmp_path, al):
    """host/pic1dp_host, imarker=1, seed_type 1, an unloaded tail: the markers right after particle_load with the device
    streams (device_rng=1) against the host streams (device_rng=0) -- x, p, w bitwise, v within 1e-15 -- and after 4
    steps with a split event (whose Gaussian draws continue the stream and its buffer) within 1e-12, same marker count."""
    from pic1dp_b200 import build
    exe = build.build_host()
    base = ["nparticle_max=300001", "nparticle_init=200001", "nx=192", "seed_type=1", "imarker=1", "iptcldist=0",
            f"al_int={al}", "v0=0.5", "temperature=1.2"]
    load = {}
    for dev in (1, 0):
        _, n, load[dev] = run_host(exe, tmp_path, f"load{dev}", base + ["ntime_max=0", f"device_rng={dev}"])
        assert n == 200_001
    for k in ("x", "p", "w"):
        assert np.array_equal(load[1][k], load[0][k]), k
    assert np.max(np.abs(load[1]["v"] - load[0]["v"])) <= 1e-15 * np.max(np.abs(load[0]["v"]))
    run = {}
    for dev in (1, 0):
        out, n, run[dev] = run_host(exe, tmp_path, f"run{dev}", base + ["ntime_max=4", "nsplit=1", "opt_t0=0.0",
                                                                       "opt_dt=0.1", f"device_rng={dev}"])
        assert "marker optimisation" in out
        run[dev]["n"] = n
    assert run[1]["n"] == run[0]["n"] > 200_001
    for k in ("x", "v", "p", "w"):
        scale = max(np.max(np.abs(run[0][k])), 1e-300)
        assert np.max(np.abs(run[1][k] - run[0][k])) <= 1e-12 * scale, k


def test_cpp_host_driver_kiss64_uniform_device_stream(tmp_path):
    """imarker=2 with KISS64 (al_int=1): the device stream (pic1dp_gpu_load_markers_kiss64, then the host generator
    jumped past it) against the host stream, bit for bit, including after remove / split events that draw from the
    generator afterwards."""
    from pic1dp_b200 import build
    exe = build.build_host()
    outs = {}
    for dev in (1, 0):
        out, n, m = run_host(exe, tmp_path, f"k{dev}", ["nparticle_max=300000", "nparticle_init=200000", "nx=192",
                                                        "ntime_max=4", "seed_type=1", "al_int=1", "nremove=1",
                                                        "nsplit=1", "opt_t0=0.0", "opt_dt=0.1", f"device_rng={dev}"])
        assert "marker optimisation" in out
        outs[dev] = (n, m)
    assert outs[1][0] == outs[0][0] > 100_000
    for k in ("x", "v", "p", "w"):
        assert np.array_equal(outs[1][1][k], outs[0][1][k]), k
