"""particle_load with MT19937-64 (multirand_al_int = 2) at the bench size, uniform-v (input_imarker = 2) and Maxwellian
(input_imarker = 1) markers: both streams generated on the device (pic1dp_gpu_load_markers_mt19937_64 /
_maxwellian_mt19937_64) against sequential host generation + pic1dp_gpu_load_markers(_maxwellian), on one GPU.

Prints one JSON line: the GPU and its power limit, per marker kind the device time of the loader (CUDA events, median of
the timed calls), the kernel times from a separate torch.profiler run (jump levels, fill, gauss), and the wall times of
the host path.  Also compares the two paths: x, p, w (and uniform v) and the final generator state must be identical;
for Maxwellian v it records the bit-equal fraction and the largest distance in ulp.

The host generator is the oracle's sequential restatement of multirand (oracle/multirand_oracle.c, gcc -O3), the same
algorithm as host/pic1dp_host.cpp's; the state is multirand_init's with seed_type 1 on rank 0 (5 warm-up passes).

    python tools_py3/dev/mt_load.py [--n 1e8] [--reps 3] [--out FILE]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.join(HERE, "..", "..")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import pic1dp_b200 as P  # noqa: E402
from multirand_state import get_state  # noqa: E402
from oracle import oracle as O  # noqa: E402
from maxwellian_load import ulps  # noqa: E402
from superkiss_load import gpu_info  # noqa: E402

KERNELS = ("k_mt64_jump", "k_mt64_fill", "k_gauss_count", "k_gauss_scatter", "k_load_markers")
NN = 312


def load(g, maxwellian, n, seeds, iseed):
    """One device load from (seeds, iseed) with an empty Gaussian buffer; seeds advanced in place."""
    if maxwellian:
        return g.load_markers_maxwellian_mt19937_64(0, n, n, seeds, iseed, 0, 0.0, n)[0]
    return g.load_markers_mt19937_64(0, n, n, seeds, iseed, 2 * n)


def measure(g, maxwellian, n, reps):
    r = O.MultiRand()
    r.init_const(2, 0, 5)
    seeds, iseed0 = get_state(r)
    seeds0 = seeds[:NN].copy()
    res = {}
    load(g, maxwellian, n, seeds0.copy(), iseed0)   # warm-up (allocations, module load)
    ms, walls = [], []
    for _ in range(reps):
        s = seeds0.copy()
        t0 = time.perf_counter()
        g.timer_start()
        pos = load(g, maxwellian, n, s, iseed0)
        ms.append(g.timer_stop())
        walls.append(time.perf_counter() - t0)
    dev, s_dev = g.get_markers(0), s
    res.update(device_load_ms=sorted(ms)[len(ms) // 2], device_load_ms_all=ms,
               device_load_wall_s=sorted(walls)[len(walls) // 2])
    if maxwellian:
        draws, rounds, regen = g.last_gaussian_load()
        res.update(gaussian_draws=draws, rounds=rounds, regenerated_draws=regen, round_draws=P._capi.GAUSS_ROUND_DRAWS)
    try:   # kernel times (separate run: the profiler slows the host)
        import torch
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.init()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            load(g, maxwellian, n, seeds0.copy(), iseed0)
        kt, calls = {}, {}
        for e in prof.key_averages():
            for key in KERNELS:
                if key in e.key:
                    kt[key] = kt.get(key, 0.0) + e.device_time_total / 1e3   # us -> ms, summed over launches
                    calls[key] = calls.get(key, 0) + e.count
        res["kernel_ms"] = kt
        res["kernel_launches"] = calls
    except Exception as ex:   # the timing above stands without the breakdown
        res["kernel_ms_error"] = repr(ex)
    # host path: sequential generation, then load_markers(_maxwellian) (16 B / marker uploaded)
    t0 = time.perf_counter()
    if maxwellian:
        v = r.gaussian_array(n)
    else:
        v = r.real_array(n)
    ux = r.real_array(n)
    t1 = time.perf_counter()
    if maxwellian:
        g.load_markers_maxwellian(0, v, ux, n)
    else:
        g.load_markers(0, v, ux, 2 * n)
    t2 = time.perf_counter()
    res.update(host_generate_s=t1 - t0, host_load_markers_s=t2 - t1, host_total_s=t2 - t0)
    host = g.get_markers(0)
    res["x_p_w_bitwise_equal"] = bool(all(np.array_equal(dev[k], host[k]) for k in ("x", "p", "w")))
    d = ulps(dev["v"], host["v"])
    res["v_bit_equal_fraction"] = float(np.mean(d == 0))
    res["v_max_ulp"] = int(d.max())
    want, want_iseed = get_state(r)
    res["state_equal"] = bool(np.array_equal(s_dev, want[:NN]) and pos == want_iseed)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=float, default=1e8, help="markers (nlocal = np)")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON line here")
    a = ap.parse_args()
    n = int(a.n)
    res = dict(gpu=gpu_info(), markers=n)
    with P.Pic1dGpu(P.default_params(nx=1024, capacity=n, iptcldist=0)) as g:
        res["uniform"] = measure(g, False, n, a.reps)
        res["maxwellian"] = measure(g, True, n, a.reps)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
