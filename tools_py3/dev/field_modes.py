"""Cost of the field solve against the number of kept modes (pic1dp_gpu_set_modes), on one GPU.

Prints JSON lines (and appends them to --out): the GPU with its power limit and SM clock; per (nx, nmode, path) the
solve time from CUDA events around 1000 back-to-back solve_field calls (device time of the whole burst, so launch gaps
are included) and the summed kernel time per solve from a separate torch.profiler run; the host time of set_modes;
and the step time with 1 kept mode against the unfiltered set at the reference default (6.4e6 markers, nx = 192) and
at 1e8 markers, nx = 1024 (CUDA events around graph-replayed step() bursts, alternated twice).

The path is the one set_modes selects (single CTA up to 64 modes, multi-CTA above); at nmode = 64 and 128 both are
also forced with PIC1DP_EXP_FIELD=single|multi, which set_modes reads.

    python tools_py3/dev/field_modes.py [--out FILE] [--solves 1000] [--quick]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", ".."))
import pic1dp_b200 as P  # noqa: E402


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True)
    except FileNotFoundError:
        return "unknown"
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def emit(rec, out):
    line = json.dumps(rec)
    print(line, flush=True)
    if out:
        with open(out, "a") as f:
            f.write(line + "\n")


def set_modes(g, modes, path):
    if path:
        os.environ["PIC1DP_EXP_FIELD"] = path
    else:
        os.environ.pop("PIC1DP_EXP_FIELD", None)
    t0 = time.perf_counter()
    g.set_modes(modes)
    return time.perf_counter() - t0


def kernel_us_per_solve(g, nsolve):
    """Device time per solve of each field kernel, from torch.profiler (CUPTI sees the library's kernels too)."""
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile
        torch.cuda.init()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(nsolve):
                g.solve_field()
            g.sync()
        tot = {}
        for e in prof.key_averages():
            if "k_field" in e.key:
                t = getattr(e, "device_time_total", None)
                tot[e.key.split("(")[0].replace("void ", "")] = (t if t is not None else e.cuda_time_total) / nsolve
        return tot
    except Exception as ex:  # noqa: BLE001 -- the event timing above stands on its own
        return {"error": repr(ex)}


def time_solves(nx, modes, path, nsolve):
    gp = P.default_params(nx=nx, capacity=16)
    rho = np.random.default_rng(nx).standard_normal(nx) * 1e-4
    with P.Pic1dGpu(gp) as g:
        t_set = set_modes(g, modes, path)
        g.set_field(chargeden=rho)
        for _ in range(50):
            g.solve_field()
        g.sync()
        g.timer_start()
        for _ in range(nsolve):
            g.solve_field()
        ms = g.timer_stop()
        kern = kernel_us_per_solve(g, 200)
    return dict(kind="solve", nx=nx, nmode=len(modes), path=path or "auto", solves=nsolve,
                us_per_solve=1e3 * ms / nsolve, kernel_us_per_solve=kern, set_modes_s=t_set)


def time_steps(n, nx, full, steps, warm):
    gp = P.default_params(nx=nx, capacity=n)
    res = {1: [], len(full): []}
    with P.Pic1dGpu(gp) as g:
        g.load_markers_counter(0, n, 1234, 0, n)
        g.collect_charge()
        g.solve_field()
        for _ in range(2):
            for modes in ([1], full):
                set_modes(g, modes, None)
                g.step(warm)
                g.timer_start()
                g.step(steps)
                res[len(modes)].append(g.timer_stop() / steps)
    return dict(kind="step", markers=n, nx=nx, steps=steps, ms_per_step={str(k): v for k, v in res.items()},
                ratio=[b / a for a, b in zip(res[1], res[len(full)])])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--solves", type=int, default=1000)
    ap.add_argument("--quick", action="store_true", help="small sizes only (checks the script, not a measurement)")
    a = ap.parse_args()
    emit(dict(kind="gpu", gpu=gpu_info()), a.out)
    nxs = [192, 1024] if a.quick else [192, 1024, 4096, 8192]
    for nx in nxs:
        for M in sorted({64, nx // 8, nx // 2}):
            modes = list(range(1, M + 1))
            emit(time_solves(nx, modes, None, a.solves), a.out)
            if M in (64, 128):
                for path in ("single", "multi"):
                    emit(time_solves(nx, modes, path, a.solves), a.out)
        if 128 not in {64, nx // 8, nx // 2}:
            for path in ("single", "multi"):
                emit(time_solves(nx, list(range(1, 129)), path, a.solves), a.out)
    os.environ.pop("PIC1DP_EXP_FIELD", None)
    if a.quick:
        emit(time_steps(1_000_000, 192, list(range(1, 97)), 50, 5), a.out)
    else:
        emit(time_steps(6_400_000, 192, list(range(1, 97)), 2000, 50), a.out)
        emit(time_steps(100_000_000, 1024, list(range(1, 513)), 100, 10), a.out)
    emit(dict(kind="gpu", gpu=gpu_info()), a.out)


if __name__ == "__main__":
    main()
