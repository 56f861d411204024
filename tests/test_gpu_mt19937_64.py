"""MT19937-64 (multirand_al_int = 2) generated on the device: the stream against the reference's known-answer vectors
(/root/reference/src/multirand.F90:396-425) and the KAT-pinned oracle, the state the device hands back, the uniform and
Maxwellian loaders against the host-stream loaders, refusals, and the C++ host driver with and without the device
streams."""
import ctypes as C
import json
import os

import numpy as np
import pytest

import pic1dp_b200 as P
from pic1dp_b200 import _capi
from helpers import make_params
from multirand_state import get_spare, get_state, run_host, to_real, ulps
from oracle import oracle as O

pytestmark = pytest.mark.gpu
NN = 312


def _mt_state(r):
    seeds, iseed = get_state(r)
    return seeds[:NN].copy(), iseed


def _assert_state(r, seeds, iseed, what):
    want, want_iseed = _mt_state(r)
    assert iseed == want_iseed and np.array_equal(seeds, want), what


def test_device_mt19937_64_known_answer_head_and_tail():
    """From the self test's seeds (iseed = 312: the first draw twists the seed block): outputs 1-10 and 308-317, the
    latter crossing into the second block."""
    gold = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "multirand_kat.json")))
    g0 = O.MultiRand()
    g0.seed_default(2)
    seeds, iseed = _mt_state(g0)
    assert iseed == NN
    _, gp = make_params(capacity=16)
    with P.Pic1dGpu(gp) as g:
        u, pos = g.mt19937_64_uniforms(seeds, iseed, NN + 5)
    assert [float(t) for t in u[:10]] == [to_real(i) for i in gold["mt19937_64_head"]]
    assert [float(t) for t in u[NN - 5:NN + 5]] == [to_real(i) for i in gold["mt19937_64_tail"]]
    g0.skip(NN + 5)
    _assert_state(g0, seeds, pos, "after the KAT")


@pytest.mark.parametrize("mype,lengths", [(0, (7, NN, 100_000_003)), (1, (1, NN - 1, NN + 1, 1_000_003)),
                                          (2, (NN, NN, 5, 65_536 * 3 + 17)), (3, (313, 10, 777_777))])
def test_device_stream_and_state_equal_the_oracle(mype, lengths):
    """Consecutive calls from the post-warm-up state and from the positions earlier calls left: every stream
    bit-identical to multirand_real_array, the returned state equal to the oracle's word for word."""
    r = O.MultiRand()
    r.init_const(2, mype, 5)
    seeds, iseed = _mt_state(r)
    _, gp = make_params(capacity=16)
    with P.Pic1dGpu(gp) as g:
        for n in lengths:
            got, iseed = g.mt19937_64_uniforms(seeds, iseed, n)
            assert np.array_equal(got, r.real_array(n)), (mype, n)
            _assert_state(r, seeds, iseed, (mype, n))


@pytest.mark.parametrize("dist", [0, 3])
def test_device_load_equals_host_stream_load_two_species(dist):
    """load_markers_mt19937_64 for two species in sequence with the state threaded through, np < nlocal (the unloaded
    tail is drawn and discarded): x, v, p, w bitwise equal to load_markers fed with the host stream of the same state,
    and the final state equal to the host generator's."""
    nlocal, nps = 200_003, (150_001, 200_003)
    kw = dict(nx=256, capacity=nlocal, nspecies=2, charge=[-1.0, -1.0], mass=[1.0, 1.0], temperature=[1.0, 1.0],
              temperature2=[1.0, 1.0], density=[0.9, 0.9], v0=[5.0, 5.0], iptcldist=dist)
    _, gp = make_params(**kw)
    r = O.MultiRand()
    r.init_const(2, 2, 5)
    seeds, iseed = _mt_state(r)
    with P.Pic1dGpu(gp) as g:
        for isp, np_ in enumerate(nps):
            u_v, u_x = r.real_array(nlocal), r.real_array(nlocal)
            g.load_markers(isp, u_v[:np_].copy(), u_x[:np_].copy(), 2 * nlocal)
            want = g.get_markers(isp)
            h2d = g.counters().h2d_bytes
            iseed = g.load_markers_mt19937_64(isp, np_, nlocal, seeds, iseed, 2 * nlocal)
            got = g.get_markers(isp)
            assert g.counters().h2d_bytes - h2d < 1_000_000      # no marker-sized upload
            for k in ("x", "v", "p", "w"):
                assert got[k].size == np_ and np.array_equal(got[k], want[k]), (isp, k)
            _assert_state(r, seeds, iseed, isp)


SIZES = (1, 2, 3, 16_001, 16_002, 700_001, 10_000_001)


@pytest.mark.parametrize("mype", [0, 3])
@pytest.mark.parametrize("spare", [False, True])
def test_maxwellian_stream_and_state_equal_the_oracle(mype, spare):
    """v within 4 ulp of gaussian_array (T = m = 1, v0 = 0), x bitwise equal to x loaded from the real_array that
    follows it, the draws consumed and the state after both calls (block, position, Gaussian buffer) equal to the
    oracle's -- from init_const, with or without a value buffered by an earlier gaussian_array(7)."""
    nmax = max(SIZES)
    _, gp = make_params(nx=64, capacity=nmax, iptcldist=0, imarker=1, temperature=[1.0], mass=[1.0], v0=[0.0])
    with P.Pic1dGpu(gp) as g:
        for n in SIZES:
            r = O.MultiRand()
            r.init_const(2, mype, 5)
            if spare:
                r.gaussian_array(7)
                assert get_spare(r)[0] == 1
            seeds, iseed = _mt_state(r)
            filled, buf = get_spare(r)
            iseed, filled, buf = g.load_markers_maxwellian_mt19937_64(0, n, n, seeds, iseed, filled, buf, n)
            got = g.get_markers(0)
            draws, rounds, regenerated = g.last_gaussian_load()
            probe = O.MultiRand()
            probe.init_const(2, mype, 5)
            if spare:
                probe.gaussian_array(7)
            probe.gaussian_array(n)
            before = _mt_state(probe)
            gauss, uni = r.gaussian_array(n), r.real_array(n)
            g.load_markers_maxwellian(0, gauss, uni, n)
            want = g.get_markers(0)
            assert np.array_equal(got["x"], want["x"]), (n, "x")
            d = ulps(got["v"], gauss)
            assert d.max() <= 4, (n, int(d.max()))
            _assert_state(r, seeds, iseed, n)
            want_filled, want_buf = get_spare(r)
            assert filled == want_filled and (not filled or ulps(buf, want_buf) <= 4), n
            # the draws the Gaussian call consumed: the oracle's state right after it, reached by skipping `draws`
            skip = O.MultiRand()
            skip.init_const(2, mype, 5)
            if spare:
                skip.gaussian_array(7)
            skip.skip(draws)
            assert np.array_equal(_mt_state(skip)[0], before[0]) and _mt_state(skip)[1] == before[1], n
            assert regenerated == 0
            if n == nmax:
                print(f"rank {mype} spare={spare}: {np.mean(d == 0):.6f} of v bitwise equal, max {d.max()} ulp, "
                      f"{draws} draws in {rounds} rounds")
                assert rounds >= 3 and (rounds - 1) * _capi.GAUSS_ROUND_DRAWS < draws <= rounds * _capi.GAUSS_ROUND_DRAWS


def test_refusals_leave_the_state_alone():
    """iptcldist != 0 (Maxwellian), nlocal < np, a block position out of range, NULL state and np > capacity are
    refused with EINVAL / ECAPACITY, and the caller's block, position and Gaussian buffer are unchanged."""
    L = _capi.load()
    r = O.MultiRand()
    r.init_const(2, 0, 5)
    r.gaussian_array(7)
    seeds, iseed0 = _mt_state(r)
    ref = seeds.copy()
    filled0, buf0 = get_spare(r)
    im, ic, isn = (C.c_int32 * 1)(1), (C.c_double * 1)(0.0), (C.c_double * 1)(1e-5)

    def call(g, np_, nlocal, iseed=iseed0, null_seeds=False, maxwellian=True):
        pos, filled, buf = C.c_int32(iseed), C.c_int32(filled0), C.c_double(buf0)
        sp = None if null_seeds else seeds.ctypes.data_as(C.POINTER(C.c_uint64))
        if maxwellian:
            rc = L.pic1dp_gpu_load_markers_maxwellian_mt19937_64(g._h, 0, np_, nlocal, 1000, sp, C.byref(pos),
                                                                 C.byref(filled), C.byref(buf), 1, im, ic, isn)
        else:
            rc = L.pic1dp_gpu_load_markers_mt19937_64(g._h, 0, np_, nlocal, 1000, sp, C.byref(pos), 8.0, 1, im, ic, isn)
        assert np.array_equal(seeds, ref) and pos.value == iseed and filled.value == filled0 and buf.value == buf0
        return rc

    _, gp3 = make_params(capacity=1000, iptcldist=3)
    with P.Pic1dGpu(gp3) as g:
        assert call(g, 100, 100) == _capi.EINVAL
    _, gp = make_params(capacity=1000, iptcldist=0, imarker=1)
    with P.Pic1dGpu(gp) as g:
        for mx in (True, False):
            assert call(g, 100, 99, maxwellian=mx) == _capi.EINVAL
            assert call(g, 100, 100, null_seeds=True, maxwellian=mx) == _capi.EINVAL
            assert call(g, 100, 100, iseed=-1, maxwellian=mx) == _capi.EINVAL
            assert call(g, 100, 100, iseed=NN + 1, maxwellian=mx) == _capi.EINVAL
            assert call(g, 1001, 2000, maxwellian=mx) == _capi.ECAPACITY
        pos = C.c_int32(NN + 1)
        out = np.empty(4)
        assert L.pic1dp_gpu_mt19937_64_uniforms(g._h, seeds.ctypes.data_as(C.POINTER(C.c_uint64)), C.byref(pos), 4,
                                                out.ctypes.data_as(C.POINTER(C.c_double))) == _capi.EINVAL
        assert np.array_equal(seeds, ref) and pos.value == NN + 1


def test_cpp_host_driver_uniform_device_stream(tmp_path):
    """host/pic1dp_host, al_int=2, imarker=2: the device stream (device_rng=1) against the host stream (device_rng=0),
    bit for bit, right after the load and after remove / split events that draw from the generator afterwards."""
    from pic1dp_b200 import build
    exe = build.build_host()
    base = ["nparticle_max=300000", "nparticle_init=200000", "nx=192", "seed_type=1", "al_int=2"]
    for extra in (["ntime_max=0"], ["ntime_max=4", "nremove=1", "nsplit=1", "opt_t0=0.0", "opt_dt=0.1"]):
        outs = {}
        for dev in (1, 0):
            _, n, m = run_host(exe, tmp_path, f"u{dev}", base + extra + [f"device_rng={dev}"])
            outs[dev] = (n, m)
        assert outs[1][0] == outs[0][0] > 100_000
        for k in ("x", "v", "p", "w"):
            assert np.array_equal(outs[1][1][k], outs[0][1][k]), (extra, k)


def test_cpp_host_driver_maxwellian_device_streams(tmp_path):
    """imarker=1, al_int=2, an unloaded tail: right after particle_load x, p, w bitwise and v within 1e-15, and after 4
    steps with a split event (whose Gaussian draws continue the stream and its buffer) within 1e-12."""
    from pic1dp_b200 import build
    exe = build.build_host()
    base = ["nparticle_max=300001", "nparticle_init=200001", "nx=192", "seed_type=1", "imarker=1", "iptcldist=0",
            "al_int=2", "v0=0.5", "temperature=1.2"]
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
