"""SuperKISS64 (multirand_al_int = 3, the reference's default) generated on the device: the stream against the
reference's known-answer vectors (/root/reference/src/multirand.F90:414-425) and the KAT-pinned oracle, the state the
device hands back, the marker loader against the host-stream loader, and the C++ host driver with and without it."""
import json
import os
import subprocess

import numpy as np
import pytest

import pic1dp_b200 as P
from pic1dp_b200 import _capi
from helpers import make_params
from multirand_state import get_state
from oracle import oracle as O

pytestmark = pytest.mark.gpu
N = 20632


def _to_real(i):
    return float(np.int64(i)) / 18446744073709551615.0 + 0.5


def test_device_superkiss64_known_answer_head_and_tail():
    gold = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "multirand_kat.json")))
    g0 = O.MultiRand()
    g0.seed_default(3)
    seeds, iseed = get_state(g0)
    _, gp = make_params(capacity=16)
    with P.Pic1dGpu(gp) as g:
        u, pos = g.superkiss64_uniforms(seeds, iseed, N + 5)
    assert [float(t) for t in u[:10]] == [_to_real(i) for i in gold["superkiss64_head"]]
    assert [float(t) for t in u[N - 5:N + 5]] == [_to_real(i) for i in gold["superkiss64_tail"]]
    g0.skip(N + 5)
    want_seeds, want_iseed = get_state(g0)
    assert pos == want_iseed and np.array_equal(seeds, want_seeds)


@pytest.mark.parametrize("mype,lengths", [(0, (10, N - 1, N, N + 1, 30_000_017)), (1, (10, N - 1, N, N + 1)),
                                          (3, (N + 1, 10, 777_777))])
def test_device_stream_and_state_equal_the_oracle(mype, lengths):
    """Consecutive calls from the post-warm-up state (table position 15) and from the positions earlier calls left:
    every stream bit-identical to multirand_real_array, the returned state equal to the oracle's word for word."""
    r = O.MultiRand()
    r.init_const(3, mype, 5)
    seeds, iseed = get_state(r)
    _, gp = make_params(capacity=16)
    with P.Pic1dGpu(gp) as g:
        for n in lengths:
            got, iseed = g.superkiss64_uniforms(seeds, iseed, n)
            assert np.array_equal(got, r.real_array(n)), (mype, n)
            want_seeds, want_iseed = get_state(r)
            assert iseed == want_iseed and np.array_equal(seeds, want_seeds), (mype, n)


@pytest.mark.parametrize("dist", [0, 3])
def test_device_load_equals_host_stream_load_two_species(dist):
    """load_markers_superkiss64 for two species in sequence with the state threaded through, np < nlocal (the unloaded
    tail is drawn and discarded): x, v, p, w bitwise equal to load_markers fed with the host stream of the same state,
    and the final state equal to the host generator's."""
    nlocal, nps = 200_003, (150_001, 200_003)
    kw = dict(nx=256, capacity=nlocal, nspecies=2, charge=[-1.0, -1.0], mass=[1.0, 1.0], temperature=[1.0, 1.0],
              temperature2=[1.0, 1.0], density=[0.9, 0.9], v0=[5.0, 5.0], iptcldist=dist)
    _, gp = make_params(**kw)
    r = O.MultiRand()
    r.init_const(3, 2, 5)
    seeds, iseed = get_state(r)
    with P.Pic1dGpu(gp) as g:
        for isp, np_ in enumerate(nps):
            u_v, u_x = r.real_array(nlocal), r.real_array(nlocal)
            g.load_markers(isp, u_v[:np_].copy(), u_x[:np_].copy(), 2 * nlocal)
            want = g.get_markers(isp)
            h2d = g.counters().h2d_bytes
            iseed = g.load_markers_superkiss64(isp, np_, nlocal, seeds, iseed, 2 * nlocal)
            got = g.get_markers(isp)
            assert g.counters().h2d_bytes - h2d < 1_000_000      # no marker-sized upload
            for k in ("x", "v", "p", "w"):
                assert got[k].size == np_ and np.array_equal(got[k], want[k]), (isp, k)
            want_seeds, want_iseed = get_state(r)
            assert iseed == want_iseed and np.array_equal(seeds, want_seeds), isp


def test_device_load_rejects_bad_stream_arguments():
    _, gp = make_params(capacity=1000)
    r = O.MultiRand()
    r.init_const(3, 0, 5)
    seeds, iseed = get_state(r)
    with P.Pic1dGpu(gp) as g:
        for np_, nlocal, pos in ((100, 99, iseed), (100, 100, -1), (100, 100, N + 1)):
            with pytest.raises(P.Pic1dpError) as e:
                g.load_markers_superkiss64(0, np_, nlocal, seeds, pos, 100)
            assert e.value.code == _capi.EINVAL
        with pytest.raises(P.Pic1dpError) as e:
            g.load_markers_superkiss64(0, 1001, 2000, seeds, iseed, 1001)
        assert e.value.code == _capi.ECAPACITY
    assert np.array_equal(seeds, get_state(r)[0])   # a refused call leaves the state alone


def test_cpp_host_driver_device_rng_writes_the_same_markers(tmp_path):
    """host/pic1dp_host with the default SuperKISS64 input, seed_type 1, an unloaded tail and marker optimisation events
    (whose remove / split draws continue the stream after particle_load): the final markers with the device stream
    (device_rng=1, the default) and with the host stream (device_rng=0) are bit-identical."""
    from pic1dp_b200 import build
    exe = build.build_host()
    outs = {}
    for dev in (1, 0):
        mk = tmp_path / f"markers{dev}.bin"
        r = subprocess.run([exe, "nparticle_max=300000", "nparticle_init=200000", "nx=192", "ntime_max=4", "seed_type=1",
                            "nremove=1", "nsplit=1", "opt_t0=0.0", "opt_dt=0.1", f"device_rng={dev}",
                            f"out={tmp_path / f'energy{dev}.txt'}", f"markers_out={mk}"],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout + r.stderr
        assert "marker optimisation" in r.stdout
        outs[dev] = mk.read_bytes()
    assert len(outs[1]) > 8 * 4 * 100_000 and outs[1] == outs[0]
