#!/usr/bin/env python
"""bench.py -- throughput of the PIC1D hot path in particle-steps/s (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path through the C ABI
  python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU algorithm (oracle port) on host cores
  python bench.py ... --dump-outputs DIR                   # also saves the last timed step's field and markers as .npy

A "step" is one full timestep input_dt of the reference time loop (src/pic1dp.F90:79-93): 2 RK substeps, each
= gather + push(x, w, v) + wrap + deposit, plus 2 field solves and 2 density all-reduces.  1 particle-step = 1 marker
advanced one step.  Workload: BASELINE.json configs[3] -- bump-on-tail delta-f, 1e8 markers per GPU, nx=1024,
weak scaling (default) -- or configs[4] with --scaling strong: 1e9 markers in total, nx=8192.  Markers are synthetic:
particle_load's distribution from the device-side KISS64 stream (multirand_al_int = 1) of a rank-dependent seed.

Keys of the JSON line: see the measurement contract in DESIGN.md.  `value` = device-timed (CUDA events on the
library's stream), markers resident in HBM; `sustained` = the same over >= 500 further steps (the clock settles under
the power cap); `e2e` = same metric through the C ABI as the reference driver uses it, host wall clock: particle_load
(seeds from the host, streams generated on the device), get_field to pinned host memory after every step, and the output
step at the reference's cadence (every 10 steps, src/pic1dp_input.F90:250 / src/pic1dp.F90:98-108) and at the end.
With --gpus N > 1 a parity pre-flight (N ranks vs the oracle's N emulated ranks) runs first: `parity_check`.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark leaves the tree as it found it (no __pycache__ from the imports below)

BYTES_IRK1 = 56   # read x,v,w,p; write x',v',w'            (SURVEY.md 8d / DESIGN.md)
BYTES_IRK2 = 80   # read mid x,v,w + start x,v,w + p; write x,v,w
BYTES_STEP = BYTES_IRK1 + BYTES_IRK2
OUTPUT_EVERY = 10  # input_output_interval / input_dt = 0.5 / 0.05
DUMP_MARKERS = 1 << 20  # --dump-outputs marker sample: x, v, p, w x 8 B x 2^20 = 32 MiB


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--markers", type=float, default=1e8, help="markers per GPU (weak scaling)")
    ap.add_argument("--nx", type=int, default=None, help="grid cells (default 1024; 8192 with --scaling strong)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: configs[3], --markers per GPU; strong: configs[4], --total-markers split over the GPUs")
    ap.add_argument("--total-markers", type=float, default=1e9, help="markers of the whole job (strong scaling)")
    ap.add_argument("--sustained-steps", type=int, default=500, help="steps of the additional sustained region (0 = off)")
    ap.add_argument("--e2e-extras", action="store_true", help="also time the host-stream and host-refresh e2e variants")
    ap.add_argument("--no-parity-check", action="store_true")
    ap.add_argument("--no-alt-arith", action="store_true",
                    help="skip the second timed region in the other arithmetic mode (reported as 'alt_arith')")
    ap.add_argument("--p2p-trace", action="store_true",
                    help="stamp %%globaltimer at publish / wait entry / wait exit of every peer-memory all-reduce of the "
                         "timed region and report arrival skew vs exchange latency (adds 'p2p_trace' to the JSON line)")
    ap.add_argument("--deposit", type=int, default=0, help="PIC1DP_DEPOSIT_* (0 = auto)")
    ap.add_argument("--allreduce", default="auto", choices=["auto", "nccl", "p2p"],
                    help="density all-reduce: NCCL or peer-memory exchange (auto = p2p when it can be set up)")
    ap.add_argument("--load-path", type=int, default=0, help="PIC1DP_LOAD_* (0 auto, 1 direct, 2 TMA ring)")
    ap.add_argument("--arith", default="strict", choices=["strict", "tolerance"],
                    help="PIC1DP_ARITH_*: strict = the reference's operation order everywhere; tolerance = w path with one "
                         "exponential (x, v, cell index still bit-exact)")
    ap.add_argument("--no-launch-timing", action="store_true",
                    help="no per-launch CUDA events inside the timed region (the region then replays the step graph; the "
                         "per-kernel times come from separately profiled steps) -- for small problems, where launch gaps matter")
    ap.add_argument("--no-graph", action="store_true", help="launch the step's kernels one by one (no CUDA graph replay)")
    ap.add_argument("--cpu-markers", type=float, default=2e7, help="markers of the bounded CPU sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what they computed on rank 0 to DIR/<name>.npy (float64): the "
                         "field arrays and a fixed sample of %d markers -- to compare two builds output for output"
                         % DUMP_MARKERS)
    args = ap.parse_args()
    if args.nx is None:
        args.nx = 8192 if args.scaling == "strong" else 1024
    return args


def fill_markers(x, v, p, w, lx, seed, chunk=1 << 24):
    """Bump-on-tail markers like particle_load's default branch (src/pic1dp_particle.F90:179-237), in place."""
    n = x.size
    rng = np.random.default_rng(seed)
    c = lx * 16.0 / n
    s2pi = np.sqrt(2.0 * np.pi)
    for lo in range(0, n, chunk):
        hi = min(n, lo + chunk)
        xs = rng.random(hi - lo) * lx
        vs = (rng.random(hi - lo) - 0.5) * 16.0
        f0 = 0.9 * np.exp(-vs * vs / 2.0) / s2pi + 0.1 * np.exp(-(vs - 5.0) ** 2 / 2.0) / s2pi
        pp = c * f0
        ww = 1e-5 * np.sin(2.0 * np.pi / lx * xs) * pp
        x[lo:hi], v[lo:hi], w[lo:hi], p[lo:hi] = xs, vs, ww, pp + ww


def fill_uniforms(u_v, u_x, seed, chunk=1 << 24):
    """The two uniform [0, 1) streams particle_load draws (v first, then x), in place (numpy PCG64)."""
    rng = np.random.default_rng(seed)
    for arr in (u_v, u_x):
        for lo in range(0, arr.size, chunk):
            hi = min(arr.size, lo + chunk)
            arr[lo:hi] = rng.random(hi - lo)


class ClockSampler:
    """SM clock and throttle reasons during the timed region, sampled every 10 ms through NVML (the same counters
    `nvidia-smi --query-gpu=clocks.sm,clocks_event_reasons.*` prints; a piped nvidia-smi block-buffers its output,
    which loses samples of a ~100 ms region)."""

    # nvmlClocksEventReason* bits (gpu_idle 0x1 is not a slowdown of a busy GPU and is left out of `reasons`)
    REASONS = {"applications_clocks_setting": 0x2, "sw_power_cap": 0x4, "hw_slowdown": 0x8, "sync_boost": 0x10,
               "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40, "hw_power_brake_slowdown": 0x80,
               "display_clock_setting": 0x100}

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.stop_flag = False
        self.thread = None
        self.err = None

    def _run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.index
            if visible:
                try:
                    idx = int(visible.split(",")[self.index])
                except Exception:
                    pass
            h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            smax = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            while not self.stop_flag:
                sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
                try:
                    rs = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    rs = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.rows.append((time.time(), sm, smax, rs))
                time.sleep(0.01)
        except Exception as e:  # pragma: no cover
            self.err = repr(e)

    def start(self):
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def stop(self, t0, t1):
        self.stop_flag = True
        if self.thread:
            self.thread.join(timeout=2)
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["NVML unavailable: %s" % self.err], "samples": 0}
        inside = [r for r in self.rows if t0 <= r[0] <= t1]
        note = None
        if not inside:
            mid = 0.5 * (t0 + t1)
            inside = sorted(self.rows, key=lambda r: abs(r[0] - mid))[:3]
            note = "no sample inside the %.0f ms timed region; nearest samples used" % (1e3 * (t1 - t0))
        reasons = sorted(k for k, bit in self.REASONS.items() if any(r[3] & bit for r in inside))
        mask = 0
        for r in inside:
            mask |= int(r[3])
        out = {"sm_mhz": float(np.median([r[1] for r in inside])), "sm_max_mhz": float(inside[0][2]),
               "reasons": reasons, "samples": len(inside), "reason_mask": hex(mask),
               "sm_mhz_min": float(min(r[1] for r in inside))}
        if note:
            out["note"] = note
        return out


def measured_peak():
    try:
        d = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def dump_outputs(g, out_dir):
    """What a caller of the timed path receives after its last step: the field (get_field) and the markers
    (get_markers).  Markers beyond DUMP_MARKERS are sampled at fixed seeded indices, the same ones for the same marker
    count, so that two builds run with the same arguments compare element for element."""
    os.makedirs(out_dir, exist_ok=True)
    for k, a in g.get_field().items():
        np.save(os.path.join(out_dir, k + ".npy"), a)
    n = g.get_markers_ptr(0)
    idx = slice(None) if n <= DUMP_MARKERS else np.sort(np.random.default_rng(0).choice(n, DUMP_MARKERS, replace=False))
    for k in ("x", "v", "p", "w"):   # one array at a time: the whole set is 32 B per marker of host memory
        np.save(os.path.join(out_dir, k + ".npy"), g.get_markers(0, want=(k,))[k][idx])


def cpu_reference_run(nx, n_markers, steps, warmup, nthreads, repeats=1):
    """The reference's algorithm for this path on host cores: oracle port with the reference's structure
    (separate push / deposit passes, backup copies, per-rank private grids summed in rank order), one emulated
    MPI rank per thread.  Returns (median particle-steps/s over `repeats` timed runs, its seconds, all values)."""
    from oracle import oracle as O
    op = O.default_params(nx=nx)
    orc = O.Oracle(op)
    n = int(n_markers)
    x, v, p, w = (np.empty(n) for _ in range(4))
    fill_markers(x, v, p, w, op.lx, seed=999)
    parts = []
    for r in range(nthreads):
        lo, hi = O.petsc_decide(n, nthreads, r)
        parts.append(dict(x=x[lo:hi].copy(), v=v[lo:hi].copy(), p=p[lo:hi].copy(), w=w[lo:hi].copy()))
    E0 = np.zeros(nx)
    if warmup > 0:
        r = orc.run([parts], warmup, E0, nthreads=nthreads)
        E0 = r["E"]
    runs = []
    for _ in range(repeats):
        r = orc.run([parts], steps, E0, nthreads=nthreads)
        E0 = r["E"]
        runs.append((n * steps / r["seconds"], r["seconds"]))
    runs.sort()
    val, secs = runs[len(runs) // 2]
    return val, secs, [v for v, _ in runs]


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    n = int(args.cpu_markers)
    value, secs, vals = cpu_reference_run(args.nx, n, args.steps, args.warmup, cores, repeats=3)
    sample = (f"{n} markers x {args.steps} steps, nx={args.nx}, {cores} emulated MPI ranks (one per host thread); "
              f"median of 3 timed runs {['%.3g' % v for v in vals]}")
    cfg = workload_config(args, args.gpus)
    # this arm runs a bounded sample of the workload: say what it ran, next to what the GPU arm runs
    cfg["gpu_arm_markers_per_gpu"], cfg["gpu_arm_markers_total"] = cfg["markers_per_gpu"], cfg["markers_total"]
    cfg["markers_per_gpu"] = cfg["markers_total"] = n
    cfg["l2"] = "CPU sample: %d markers, %.2f GB of marker state" % (n, n * 80 / 1e9)
    cfg["parallelism"] = f"{cores} emulated MPI ranks on host threads, per-rank private grids summed in rank order"
    line = {
        "impl": "reference", "metric": "particle_steps_per_sec", "value": value, "unit": "particle-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / args.steps,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": value, "unit": "particle-steps/s", "cores": cores, "kind": "port", "sample": sample,
                         "note": "CPU restatement of the reference loops (oracle/), not the PETSc binary: no "
                                 "Fortran/MPI/PETSc toolchain exists in this image"},
        "e2e": {"value": value, "unit": "particle-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def markers_per_gpu(args, world):
    if args.scaling == "strong":
        return int(args.total_markers) // world
    return int(args.markers)


def workload_config(args, n_gpus):
    n = markers_per_gpu(args, n_gpus)
    if args.scaling == "strong":
        name = ("configs[4]: bump-on-tail delta-f nonlinear, strong scaling %.3g markers in total, nx=%d, 1 mode, "
                "dt=0.05, iptclshape=4" % (args.total_markers, args.nx))
    else:
        name = ("configs[3]: bump-on-tail delta-f nonlinear, weak scaling %.3g markers per GPU, nx=%d, 1 mode, dt=0.05, "
                "iptclshape=4" % (n, args.nx))
    return {"workload": name, "markers_per_gpu": n, "markers_total": n * n_gpus, "nx": args.nx, "nmode": 1,
            "bytes_per_particle_step": BYTES_STEP, "arith_mode": args.arith,
            "l2": "inputs larger than L2: %.1f GB of marker state streamed per step per GPU" % (n * BYTES_STEP / 1e9),
            "parallelism": f"particle-decomposition x{n_gpus}, replicated grid, density all-reduce per substep "
                           "(peer-memory exchange over NVLink, NCCL fallback)"}


def rank_seeds(rank):
    """multirand_seeds(0:3) of this rank as multirand_init leaves them for seed_type = 3 (four random 64-bit words,
    src/multirand.F90:275-300; here from a fixed-seed host generator so that runs repeat) after the warm-up of
    5 x 4 outputs (:376-381)."""
    from pic1dp_b200 import host as H
    words = [int(w) for w in np.random.default_rng(1234 + rank).integers(1, 2**63, size=4, dtype=np.int64)]
    return H.host_kiss64_jump(words, 20)


def setup_comm(P, dist, g, args, rank, world):
    """NCCL communicator + (when possible) the peer-memory exchange buffers; returns 'p2p' or 'nccl'."""
    uid = [g.comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    g.comm_init(uid[0])
    if args.allreduce in ("auto", "p2p") and world <= 8:
        try:
            handles = [None] * world
            dist.all_gather_object(handles, g.p2p_export())
            g.p2p_import(handles)
            return "p2p"
        except Exception as e:  # keep NCCL
            if args.allreduce == "p2p":
                raise
            print(f"[rank {rank}] peer-memory all-reduce unavailable, using NCCL: {e}", file=sys.stderr)
    return "nccl"


def analyse_trace(rows, nepochs, cap):
    """rows[r] = (stamps[cap][3] = publish, wait entry, wait exit in rank r's own %globaltimer ns, last epoch).
    Per all-reduce and rank: d = wait_exit - publish.  The rank that arrived last waits only for the kernel boundary and
    the flag reads, so min over ranks of d is the exchange floor; what the other ranks wait beyond it is arrival skew
    (they finished their particle kernel earlier).  No cross-GPU clock synchronisation is needed: every difference is
    taken on one GPU's clock."""
    last = min(r[1] for r in rows)
    eps = [e for e in range(last - nepochs + 1, last + 1) if e > 0]
    d = np.array([[rows[r][0][e % cap][2] - rows[r][0][e % cap][0] for r in range(len(rows))] for e in eps], dtype=np.float64)
    gap = np.array([[rows[r][0][e % cap][1] - rows[r][0][e % cap][0] for r in range(len(rows))] for e in eps], dtype=np.float64)
    spin = np.array([[rows[r][0][e % cap][2] - rows[r][0][e % cap][1] for r in range(len(rows))] for e in eps], dtype=np.float64)
    floor = d.min(axis=1)
    skew = d - floor[:, None]
    q = lambda a, p: float(np.percentile(a, p)) / 1e3
    return {"allreduces": len(eps), "ranks": len(rows), "unit": "us",
            "publish_to_wait_exit": {"median": q(d, 50), "p95": q(d, 95), "max": q(d, 100)},
            "exchange_floor_min_over_ranks": {"median": q(floor, 50), "p95": q(floor, 95)},
            "kernel_boundary_publish_to_wait_entry": {"median": q(gap, 50), "p95": q(gap, 95)},
            "spin_wait_entry_to_exit": {"median": q(spin, 50), "mean": float(spin.mean()) / 1e3, "p95": q(spin, 95)},
            "arrival_skew_wait": {"mean": float(skew.mean()) / 1e3, "median": q(skew, 50), "p95": q(skew, 95),
                                  "mean_of_worst_rank": float(skew.max(axis=1).mean()) / 1e3},
            "per_rank_mean_skew_wait": [float(v) / 1e3 for v in skew.mean(axis=0)],
            "last_arrival_counts_per_rank": [int(v) for v in np.bincount(d.argmin(axis=1), minlength=len(rows))],
            "per_step_cost_us": {"exchange_floor": 2 * float(floor.mean()) / 1e3,
                                 "skew_mean_rank": 2 * float(skew.mean()) / 1e3,
                                 "skew_worst_rank": 2 * float(skew.max(axis=1).mean()) / 1e3},
            "note": "d = wait_exit - publish per rank and all-reduce; floor = min over ranks (the last arrival); skew = d - floor; "
                    "per_rank_mean_skew_wait small / last_arrival_counts large for a rank = that GPU is systematically the slowest"}


def parity_preflight(P, dist, torch, args, rank, world, local):
    """tests/mgpu_worker.py's comparison inside the bench run, so that every multi-GPU line carries its own parity
    evidence: 4e5 markers split by the PETSC_DECIDE rule over the N ranks, 5 steps through the same all-reduce path the
    timed region uses, against the oracle's N emulated ranks (rank 0 compares; the oracle is only the checker)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from helpers import OracleRun, make_params, rel_err, synth_markers
    n, nx, nsteps = 400003, 256, 5
    op, gp = make_params(nx=nx, capacity=n, device=local, rank=rank, nranks=world, deposit_mode=args.deposit,
                         arith_mode=1 if args.arith == "tolerance" else 0)
    st = synth_markers(op, n, seed=99)
    lo, hi = P.petsc_decide(n, world, rank)
    g = P.Pic1dGpu(gp)
    path = setup_comm(P, dist, g, args, rank, world)
    g.set_markers(0, *(np.ascontiguousarray(st[k][lo:hi]) for k in ("x", "v", "p", "w")))
    g.collect_charge()
    g.solve_field()
    g.step(nsteps)
    f = g.get_field()
    mk = g.get_markers(0)
    c = g.counters()
    E_all = [torch.zeros(nx, dtype=torch.float64) for _ in range(world)]
    dist.all_gather(E_all, torch.from_numpy(f["electric"].copy()))
    same = all(torch.equal(E_all[0], e) for e in E_all)
    parts = [None] * world
    dist.all_gather_object(parts, {k: mk[k] for k in ("x", "v", "w")})
    g.close()
    res = [None]
    if rank == 0:
        states = []
        for r in range(world):
            a, b = P.petsc_decide(n, world, r)
            states.append({k: st[k][a:b].copy() for k in st})
        ref = OracleRun(op, [states])
        ref.init_field()
        for _ in range(nsteps):
            ref.step()
        e_rho, e_E = rel_err(f["chargeden"], ref.rho), rel_err(f["electric"], ref.E)
        e_mk = max(rel_err(parts[r][k], ref.st[0][r][k]) for r in range(world) for k in ("x", "v", "w"))
        ok = bool(same and e_rho < 1e-12 and e_E < 1e-12 and e_mk < 1e-12 and c.p2p_timeouts == 0)
        res[0] = {"ranks": world, "markers": n, "steps": nsteps, "allreduce": path, "rho": e_rho, "E": e_E, "markers_xvw": e_mk,
                  "replicated_equal": bool(same), "tolerance": 1e-12, "pass": ok,
                  "against": "oracle with %d emulated MPI ranks (PETSC_DECIDE blocks, grids summed in rank order)" % world}
    dist.broadcast_object_list(res, src=0)
    return res[0]


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if args.gpus > 1 and world == 1:
        raise SystemExit("for --gpus N > 1 launch with: python -m torch.distributed.run --nproc-per-node N bench.py ...")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group(backend="cpu:gloo,cuda:nccl", device_id=torch.device("cuda", local))

    from pic1dp_b200 import build as _build
    if rank == 0:
        _build.build()
    if world > 1:
        dist.barrier()
    import pic1dp_b200 as P

    # ---- multi-GPU parity pre-flight: N ranks vs the oracle's N emulated ranks ----
    parity = None
    if world > 1 and not args.no_parity_check:
        parity = parity_preflight(P, dist, torch, args, rank, world, local)
        if not parity["pass"]:
            if rank == 0:
                print(json.dumps({"parity_check": parity}), flush=True)
            raise SystemExit("multi-GPU parity pre-flight failed: " + json.dumps(parity))

    n = markers_per_gpu(args, world)
    ntotal = n * world
    gp = P.default_params(nx=args.nx, capacity=n, device=local, rank=rank, nranks=world, deposit_mode=args.deposit, load_path=args.load_path,
                          arith_mode=1 if args.arith == "tolerance" else 0, no_step_graph=1 if args.no_graph else 0)
    g = P.Pic1dGpu(gp)
    if world > 1:
        setup_comm(P, dist, g, args, rank, world)

    # ---- synthetic inputs: particle_load with the device-side KISS64 stream of this rank's seeds (no marker-sized
    # host-to-device copy; the host supplies 32 bytes of generator state) ----
    seeds = rank_seeds(rank)

    def load_from_host():  # particle_load through the C ABI: pv is drawn first, then px (src/pic1dp_particle.F90:180, :222)
        g.load_markers_kiss64(0, n, seeds, 0, n, ntotal, v_max=8.0)
    nx = args.nx
    hf = {k: torch.empty(m, dtype=torch.float64, pin_memory=True) for k, m in (("E", nx), ("rho", nx), ("re", 1), ("im", 1))}

    def barrier():
        g.sync()
        if world > 1:
            dist.barrier()
        g.sync()

    def max_over_ranks(val):
        if world == 1:
            return val
        t = torch.tensor([val], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- peer-memory all-reduce sanity: one step, then every rank must report no timeout and a finite field ----
    if world > 1 and args.allreduce != "nccl":
        load_from_host()
        g.collect_charge()
        g.solve_field()
        g.step(1)
        try:
            bad = float(g.counters().p2p_timeouts > 0 or not np.isfinite(g.field_energy()))
        except P.Pic1dpError:
            bad = 1.0
        bad = max_over_ranks(bad)
        if bad > 0:
            if args.allreduce == "p2p":
                raise SystemExit("peer-memory all-reduce failed (timeouts or non-finite field)")
            if rank == 0:
                print("peer-memory all-reduce failed its sanity step; falling back to NCCL", file=sys.stderr)
            g.close()
            g = P.Pic1dGpu(gp)
            uid = [g.comm_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(uid, src=0)
            g.comm_init(uid[0])

    # ---- device-resident throughput ("value") ----
    sampler = ClockSampler(local)
    sampler.start()   # started well before the timed region: the sampler needs a few hundred ms to deliver samples
    load_from_host()
    g.collect_charge()
    g.solve_field()
    g.step(args.warmup)
    tracing = args.p2p_trace and world > 1 and g.counters().p2p_allreduces > 0
    if tracing:
        g.p2p_trace(4 * args.steps + 16)
        g.step(1)   # re-captures the step graph with the trace buffer
    barrier()
    c0 = g.counters()
    t0 = time.time()
    if not args.no_launch_timing:
        g.launch_timing_start()   # event pair around every fused particle-kernel launch of the timed region
    g.timer_start()
    g.step(args.steps)
    ms = g.timer_stop()
    lt = g.launch_timing_stop() if not args.no_launch_timing else [(0.0, 0), (0.0, 0)]
    barrier()
    t1 = time.time()
    clocks = sampler.stop(t0, t1)
    c1 = g.counters()
    ms = max_over_ranks(ms)
    value = ntotal * args.steps / (ms * 1e-3)
    energy = g.field_energy()
    p2p_trace = None
    if tracing:
        cap = 4 * args.steps + 16
        stamps, last = g.p2p_trace_read(cap)
        g.p2p_trace(0)
        rows = [None] * world
        dist.all_gather_object(rows, (stamps.astype(np.int64), int(last)))
        if rank == 0:
            p2p_trace = analyse_trace(rows, 2 * args.steps, cap)
    if args.dump_outputs and rank == 0:   # before the regions below reload and advance the markers
        dump_outputs(g, args.dump_outputs)

    # ---- sustained: the same loop for >= 500 further steps (graph replay, no per-launch events).  Runs AFTER the
    # driver-length e2e region below, so that `value` and `e2e` are both measured from the same (cool) state and
    # `sustained` / `e2e.sustained` both under the power cap ----
    def run_sustained():
        s2 = ClockSampler(local)
        s2.start()
        time.sleep(0.05)
        barrier()
        ts0 = time.time()
        g.timer_start()
        g.step(args.sustained_steps)
        ms_s = g.timer_stop()
        barrier()
        ts1 = time.time()
        ms_s = max_over_ranks(ms_s)
        return {"steps": args.sustained_steps, "value": ntotal * args.sustained_steps / (ms_s * 1e-3),
                "unit": "particle-steps/s", "ms_per_step": ms_s / args.sustained_steps,
                "step_roofline_frac": n * BYTES_STEP / (ms_s / args.sustained_steps * 1e-3) / 1e9 / measured_peak()[0],
                "clocks": s2.stop(ts0, ts1), "graph_replays": int(g.counters().graph_replays)}
    sustained = None
    g.output_all(64, 64, 8.0)            # one-time scratch allocations of the diagnostics happen here, untimed

    # ---- roofline of the dominant kernel, CUDA events around each launch ----
    prof = np.array([g.profile_step() for _ in range(5)])[1:].mean(axis=0)  # ms: push1, collect1, field1, push2, ...
    # the two particle kernels: average over every launch INSIDE the timed region (the grid kernels come from the
    # separately profiled steps above)
    if lt[0][1] > 0 and lt[1][1] > 0:
        prof[0], prof[3] = lt[0][0] / lt[0][1], lt[1][0] / lt[1][1]
    peak, peak_src = measured_peak()
    # dram__bytes_read + dram__bytes_write of this kernel from the committed `ncu --set full` capture at the bench size
    traffic, traffic_src = None, None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
        if int(c1.deposit_mode) == tj.get("deposit_mode", 1) and args.nx == tj.get("nx", 1024):
            traffic = tj["irk2"]["dram_bytes_per_marker"] * n
            traffic_src = tj["source"] + "; per-marker DRAM bytes x markers of this launch"
    except Exception:
        pass
    ach2 = n * BYTES_IRK2 / (prof[3] * 1e-3) / 1e9
    ach1 = n * BYTES_IRK1 / (prof[0] * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": "k_push<bump-on-tail, irk=2, fused push+wrap+deposit>",
                "achieved": ach2, "peak": peak, "unit": "GB/s", "frac": ach2 / peak, "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": peak_src, "ms_per_launch": float(prof[3]), "launches_timed": int(lt[1][1]),
                "timing": ("CUDA events around each launch of this kernel inside the timed region, on the library's stream"
                           if lt[1][1] > 0 else "CUDA events around this kernel in 4 separately profiled steps (graph-replay run)"),
                "algorithmic_bytes_per_launch": n * BYTES_IRK2}
    if roofline["frac"] > 1.0:
        roofline["note"] = ("frac > 1: the denominator is the MEASURED copy bandwidth of MEASURED_PEAKS.json (a 1:1 read/write "
                            "stream); this kernel reads 56 B and writes 24 B per marker and sustains more than that copy "
                            "kernel (B200 HBM3e nominal: 7.7-8.0 TB/s).  DRAM bytes from ncu (`traffic`) equal the algorithmic bytes.")
    roofline_detail = {
        "irk1": {"achieved": ach1, "frac": ach1 / peak, "ms_per_launch": float(prof[0]), "bytes": n * BYTES_IRK1},
        "step": {"achieved": n * BYTES_STEP / (ms / args.steps * 1e-3) / 1e9,
                 "frac": n * BYTES_STEP / (ms / args.steps * 1e-3) / 1e9 / peak,
                 "note": "136 B x markers / whole-step time incl. reduce, all-reduce, field solve"},
        "grid_kernels_ms": {"reduce+allreduce+finalize": float(prof[1] + prof[4]), "field_solve": float(prof[2] + prof[5])},
    }

    # ---- end to end through the C ABI with host buffers ----
    e2e = None
    if not args.no_e2e:
        def e2e_run(k, load):
            """particle_load + k steps as the reference driver runs them (src/pic1dp.F90:63-109): every step the fields
            come back to pinned host memory; every OUTPUT_EVERY steps (and at the end) output_all runs on the device
            (one fused pass, a few KB of D2H)."""
            barrier()
            cc0 = g.counters()
            t_0 = time.perf_counter()
            load()
            g.collect_charge()
            g.solve_field()
            for it in range(1, k + 1):
                g.step(1)
                g.get_field_ptr(hf["E"].data_ptr(), hf["rho"].data_ptr(), hf["re"].data_ptr(), hf["im"].data_ptr())
                if it % OUTPUT_EVERY == 0 or it == k:                        # output_all cadence
                    g.output_all(64, 64, 8.0)
            g.sync()
            tw = max_over_ranks(time.perf_counter() - t_0)
            cc = g.counters()
            return {"value": ntotal * k / tw, "unit": "particle-steps/s", "steps": k, "ms_per_step": 1e3 * tw / k,
                    "h2d_bytes_per_step": (cc.h2d_bytes - cc0.h2d_bytes) / k,
                    "d2h_bytes_per_step": (cc.d2h_bytes - cc0.d2h_bytes) / k}

        e2e = e2e_run(args.steps, load_from_host)
        e2e["definition"] = ("reference driver loop through the C ABI, host wall clock, max over ranks: particle_load as "
                             "pic1dp_gpu_load_markers_kiss64 (the host passes multirand's 32-byte KISS64 state, the device "
                             "generates both uniform streams bit-exactly and applies the loader arithmetic) + K steps, "
                             "get_field (E, rho, modes) to pinned host memory after every step, output_all every "
                             f"{OUTPUT_EVERY} steps and at the end (reference cadence, src/pic1dp.F90:98-108) as "
                             "pic1dp_gpu_output_all (one fused device pass, results to the host)")
        if args.sustained_steps > 0:   # the same loop at the sustained length: start-up costs amortised as in a real run
            sustained = run_sustained()
            ks = min(args.sustained_steps, 200)
            e2e["sustained"] = e2e_run(ks, load_from_host)
        if args.e2e_extras and n <= 200_000_000:
            host = {k: torch.empty(n, dtype=torch.float64, pin_memory=True) for k in ("x", "v", "p", "w", "u_v", "u_x")}
            hv = {k: t.numpy() for k, t in host.items()}
            fill_uniforms(hv["u_v"], hv["u_x"], seed=1234 + rank)
            ptr = {k: t.data_ptr() for k, t in host.items()}
            e2e["host_stream_load"] = e2e_run(args.steps, lambda: g.load_markers(0, (ptr["u_v"], n), (ptr["u_x"], n), ntotal, v_max=8.0))
            e2e["host_stream_load"]["definition"] = ("same with the two uniform streams generated by the host (SuperKISS64 / "
                                                     "MT19937-64 have no device form): 16 B/marker of H2D in the load")
            g.get_markers_ptr(0, x=ptr["x"], v=ptr["v"], p=ptr["p"], w=ptr["w"])
            k2 = min(args.steps, 3)   # worst case: markers live on the host and make the round trip every step
            barrier()
            tw0 = time.perf_counter()
            for it in range(k2):
                g.set_markers_ptr(0, n, ptr["x"], ptr["v"], ptr["p"], ptr["w"])
                g.collect_charge()
                g.solve_field()
                g.step(1)
                g.get_field_ptr(hf["E"].data_ptr(), hf["rho"].data_ptr(), hf["re"].data_ptr(), hf["im"].data_ptr())
                g.get_markers_ptr(0, x=ptr["x"], v=ptr["v"], w=ptr["w"])
            tw2 = max_over_ranks(time.perf_counter() - tw0)
            e2e["roundtrip_every_step"] = {"value": ntotal * k2 / tw2, "steps": k2,
                                           "h2d_bytes_per_step": 4 * 8 * n, "d2h_bytes_per_step": 3 * 8 * n + (2 * nx + 2) * 8}
        # device time of one output step, and of the load
        g.timer_start()
        g.output_all(64, 64, 8.0)
        t_oa = g.timer_stop()
        g.timer_start()
        load_from_host()
        t_ld = g.timer_stop()
        e2e["output_step_ms"] = {"output_all": t_oa}
        e2e["particle_load_ms"] = t_ld

    if sustained is None and args.sustained_steps > 0:   # --no-e2e
        sustained = run_sustained()

    # ---- the other arithmetic mode, same workload, same box, same run (device-timed like `value`) ----
    alt = None
    if not args.no_alt_arith and args.scaling == "weak":
        other = "tolerance" if args.arith == "strict" else "strict"
        g.close()
        gp2 = P.default_params(nx=args.nx, capacity=n, device=local, rank=rank, nranks=world, deposit_mode=args.deposit,
                               load_path=args.load_path, arith_mode=1 if other == "tolerance" else 0,
                               no_step_graph=1 if args.no_graph else 0)
        g = P.Pic1dGpu(gp2)
        if world > 1:
            setup_comm(P, dist, g, args, rank, world)
        load_from_host()
        g.collect_charge()
        g.solve_field()
        g.step(args.warmup)
        barrier()
        g.launch_timing_start()
        g.timer_start()
        g.step(args.steps)
        ms2 = max_over_ranks(g.timer_stop())
        lt2 = g.launch_timing_stop()
        barrier()
        t_i1, t_i2 = lt2[0][0] / max(lt2[0][1], 1), lt2[1][0] / max(lt2[1][1], 1)
        alt = {"arith_mode": other, "deposit_mode": int(g.counters().deposit_mode),
               "value": ntotal * args.steps / (ms2 * 1e-3), "unit": "particle-steps/s",
               "ms_per_step": ms2 / args.steps, "step_roofline_frac": n * BYTES_STEP / (ms2 / args.steps * 1e-3) / 1e9 / peak,
               "irk1": {"ms_per_launch": t_i1, "frac": n * BYTES_IRK1 / (t_i1 * 1e-3) / 1e9 / peak},
               "irk2": {"ms_per_launch": t_i2, "frac": n * BYTES_IRK2 / (t_i2 * 1e-3) / 1e9 / peak},
               "note": "STRICT = the reference's operation order everywhere (the parity target of the tests); TOLERANCE = "
                       "-d ln f0/dv with one exponential instead of two: x, v, cell index still bit-exact, w within "
                       "1e-14 of max|w| per substep (tests/test_gpu_round2.py)"}

    # ---- CPU baseline beside it (rank 0, bounded sample) ----
    cpu = None
    if rank == 0 and not args.no_cpu_baseline and world == 1:
        cores = os.cpu_count() or 1
        ncpu = int(args.cpu_markers)
        csteps = max(3, int(round(4.0 * 2e8 * cores / 16 / max(ncpu, 1))))  # ~4 s per run at ~1.2e7 particle-steps/s/core
        val, secs, vals = cpu_reference_run(args.nx, ncpu, csteps, 1, cores, repeats=3)
        cpu = {"value": val, "unit": "particle-steps/s", "cores": cores, "kind": "port",
               "sample": f"{ncpu} markers x {csteps} steps (+1 warm-up), nx={args.nx}, {cores} emulated MPI ranks; median of 3 "
                         f"runs {['%.3g' % v for v in vals]}, {secs:.1f} s each",
               "note": "CPU restatement of the reference loops (oracle/), not the PETSc binary"}

    if rank == 0:
        line = {
            "metric": "particle_steps_per_sec", "value": value, "unit": "particle-steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args, world),
            "clocks": clocks, "sustained": sustained, "e2e": e2e, "gpu_launches": int(c1.kernel_launches - c0.kernel_launches),
            "nccl_calls": int(c1.nccl_calls - c0.nccl_calls),
            "p2p_allreduces": int(c1.p2p_allreduces - c0.p2p_allreduces), "p2p_timeouts": int(c1.p2p_timeouts),
            "parity_check": parity, "p2p_trace": p2p_trace, "alt_arith": alt,
            "roofline": roofline, "roofline_detail": roofline_detail, "cpu_baseline": cpu,
            "deposit_mode": int(c1.deposit_mode), "grid_ctas": int(c1.grid_ctas), "cta_threads": int(c1.cta_threads),
            "smem_bytes": int(c1.smem_bytes), "oob_markers": int(c1.oob_markers), "field_energy": energy,
        }
        print(json.dumps(line), flush=True)
    g.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
