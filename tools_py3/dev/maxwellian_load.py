"""particle_load of Maxwellian markers (input_imarker = 1) at the bench size, for KISS64 and SuperKISS64: both streams
generated on the device (pic1dp_gpu_load_markers_maxwellian_kiss64 / _superkiss64) against sequential host generation
(multirand_gaussian_array, then multirand_real_array) + pic1dp_gpu_load_markers_maxwellian, on one GPU.

Prints one JSON line: the GPU and its power limit, per generator the device time of the loader (CUDA events, median of
the timed calls), the draws, rounds and regenerated draws of the device's Gaussian call, the kernel times from a separate
torch.profiler run, and the wall times of the host path.  Also compares the two paths: x, p, w and the final generator
state must be identical; for v it records the bit-equal fraction and the largest distance in ulp.

The host generator is the oracle's sequential restatement of multirand (oracle/multirand_oracle.c, gcc -O3), the same
algorithm as host/pic1dp_host.cpp's; the state is multirand_init's with seed_type 1 on rank 0 (5 warm-up passes).

    python tools_py3/dev/maxwellian_load.py [--n 1e8] [--reps 3] [--out FILE]
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
from superkiss_load import gpu_info  # noqa: E402

KERNELS = ("k_kiss64_fill", "k_superkiss64_table", "k_superkiss64_finish", "k_gauss_count", "k_gauss_scatter",
           "k_load_markers")


def ulps(a, b):
    def key(x):
        i = np.asarray(x, dtype=np.float64).view(np.int64)
        return np.where(i < 0, np.int64(-0x8000000000000000) - i, i)
    return np.abs(key(a) - key(b))


def device_state(al, oracle):
    seeds, iseed = get_state(oracle)
    return (seeds.copy() if al == 3 else seeds[:4].copy()), iseed


def load(g, al, n, seeds, iseed):
    """One device load from (seeds, iseed) with an empty Gaussian buffer; seeds advanced in place."""
    if al == 3:
        return g.load_markers_maxwellian_superkiss64(0, n, n, seeds, iseed, 0, 0.0, n)
    return (iseed,) + tuple(g.load_markers_maxwellian_kiss64(0, n, n, seeds, 0, 0.0, n))


def measure(g, al, n, reps):
    r = O.MultiRand()
    r.init_const(al, 0, 5)
    seeds0, iseed0 = device_state(al, r)
    res = {}
    load(g, al, n, seeds0.copy(), iseed0)   # warm-up (allocations, module load)
    ms, walls = [], []
    for _ in range(reps):
        s = seeds0.copy()
        t0 = time.perf_counter()
        g.timer_start()
        after = load(g, al, n, s, iseed0)
        ms.append(g.timer_stop())
        walls.append(time.perf_counter() - t0)
    dev, s_dev = g.get_markers(0), s
    draws, rounds, regen = g.last_gaussian_load()
    res.update(device_load_ms=sorted(ms)[len(ms) // 2], device_load_ms_all=ms,
               device_load_wall_s=sorted(walls)[len(walls) // 2], gaussian_draws=draws, rounds=rounds,
               regenerated_draws=regen, round_draws=P._capi.GAUSS_ROUND_DRAWS)
    try:   # kernel times (separate run: the profiler slows the host)
        import torch
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.init()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            load(g, al, n, seeds0.copy(), iseed0)
        kt = {}
        for e in prof.key_averages():
            for key in KERNELS:
                if key in e.key:
                    kt[key] = kt.get(key, 0.0) + e.device_time_total / 1e3   # us -> ms, summed over launches
        res["kernel_ms"] = kt
    except Exception as ex:   # the timing above stands without the breakdown
        res["kernel_ms_error"] = repr(ex)
    # host path: sequential gaussian_array + real_array, then load_markers_maxwellian (16 B / marker uploaded)
    t0 = time.perf_counter()
    gv = r.gaussian_array(n)
    ux = r.real_array(n)
    t1 = time.perf_counter()
    g.load_markers_maxwellian(0, gv, ux, n)
    t2 = time.perf_counter()
    res.update(host_generate_s=t1 - t0, host_load_markers_s=t2 - t1, host_total_s=t2 - t0)
    host = g.get_markers(0)
    d = ulps(dev["v"], host["v"])
    res["x_p_w_bitwise_equal"] = bool(all(np.array_equal(dev[k], host[k]) for k in ("x", "p", "w")))
    res["v_bit_equal_fraction"] = float(np.mean(d == 0))
    res["v_max_ulp"] = int(d.max())
    want_seeds, want_iseed = device_state(al, r)
    res["state_equal"] = bool(np.array_equal(s_dev, want_seeds) and (al != 3 or after[0] == want_iseed))
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
        for al, name in ((1, "kiss64"), (3, "superkiss64")):
            res[name] = measure(g, al, n, a.reps)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
