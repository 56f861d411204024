"""particle_load with SuperKISS64 (multirand_al_int = 3, the reference's default) at the bench size: the device stream
(pic1dp_gpu_load_markers_superkiss64) against host generation + pic1dp_gpu_load_markers, on one GPU.

Prints one JSON line: the GPU and its power limit, the device time of the loader (CUDA events, median of the timed
calls), the kernel times of the sequential refill CTA, the finishing kernel and the loader arithmetic from a separate
torch.profiler run, the time per refill, and the wall times of the host path (sequential generator, then the upload +
loader).  Also checks that both paths load bit-identical markers.

    python tools_py3/dev/superkiss_load.py [--n 1e8] [--reps 3] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", ".."))
import pic1dp_b200 as P  # noqa: E402
from pic1dp_b200 import _capi, host as H  # noqa: E402

N_TABLE = 20632


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True)
    except FileNotFoundError:
        return "unknown"
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def warmed_up_state():
    """The self test's default SuperKISS64 seeds (src/multirand.F90:513-515) and multirand_init's warm-up of
    5 * 20635 draws (:379-381), run with the library's sequential generator."""
    m64 = (1 << 64) - 1
    s = np.zeros(_capi.SUPERKISS64_NSEED, dtype=np.uint64)
    lcg, xs = 12367890123456, 521288629546311
    for i in range(N_TABLE):
        lcg = (lcg * 6906969069 + 123) & m64
        xs ^= (xs << 13) & m64
        xs ^= xs >> 17
        xs ^= (xs << 43) & m64
        s[i] = (lcg + xs) & m64
    s[N_TABLE:] = [36243678541, lcg, xs]
    _, iseed = H.host_superkiss64_fill(s, N_TABLE, 5 * _capi.SUPERKISS64_NSEED)
    return s, iseed


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=float, default=1e8, help="markers (nlocal = np)")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON line here")
    a = ap.parse_args()
    n = int(a.n)
    seeds0, iseed0 = warmed_up_state()
    ndraw = 2 * n
    nrefill = -(-(ndraw - (N_TABLE - iseed0)) // N_TABLE)
    res = dict(gpu=gpu_info(), markers=n, draws=ndraw, refills=nrefill)
    with P.Pic1dGpu(P.default_params(nx=1024, capacity=n)) as g:
        # device path: warm-up, then timed calls from the same starting state
        g.load_markers_superkiss64(0, n, n, seeds0.copy(), iseed0, n)
        ms, walls = [], []
        for _ in range(a.reps):
            s = seeds0.copy()
            t0 = time.perf_counter()
            g.timer_start()
            pos = g.load_markers_superkiss64(0, n, n, s, iseed0, n)
            ms.append(g.timer_stop())
            walls.append(time.perf_counter() - t0)
        dev, s_dev = g.get_markers(0), s
        res["device_load_ms"] = sorted(ms)[len(ms) // 2]
        res["device_load_ms_all"] = ms
        res["device_load_wall_s"] = sorted(walls)[len(walls) // 2]
        # kernel times (separate run: the profiler slows the host)
        try:
            import torch
            from torch.profiler import ProfilerActivity, profile
            torch.cuda.init()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                g.load_markers_superkiss64(0, n, n, seeds0.copy(), iseed0, n)
            kt = {}
            for e in prof.key_averages():
                for key in ("k_superkiss64_table", "k_superkiss64_finish", "k_load_markers"):
                    if key in e.key:
                        kt[key] = kt.get(key, 0.0) + e.device_time_total / 1e3   # us -> ms, summed over launches
            res["kernel_ms"] = kt
            if "k_superkiss64_table" in kt:
                res["us_per_refill"] = kt["k_superkiss64_table"] * 1e3 / nrefill
        except Exception as ex:   # the timing above stands without the breakdown
            res["kernel_ms_error"] = repr(ex)
        # host path: the library's sequential generator, then load_markers (16 B / marker uploaded)
        s = seeds0.copy()
        u = np.zeros(ndraw)        # pre-faulted
        pos_h = C.c_int32(iseed0)
        t0 = time.perf_counter()
        rc = _capi.load().pic1dp_host_superkiss64_fill(H._state_ptr(s, *H._SK), C.byref(pos_h), ndraw, H._dp(u))
        t1 = time.perf_counter()
        assert rc == 0
        p2 = pos_h.value
        g.load_markers(0, u[:n], u[n:], n)
        t2 = time.perf_counter()
        res["host_generate_s"] = t1 - t0
        res["host_load_markers_s"] = t2 - t1
        res["host_total_s"] = t2 - t0
        host = g.get_markers(0)
        res["bitwise_equal"] = bool(all(np.array_equal(dev[k], host[k]) for k in ("x", "v", "p", "w")))
        res["state_equal"] = bool(pos == p2 and np.array_equal(s_dev, s))
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
