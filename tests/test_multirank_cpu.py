"""world_size-2 gloo tests (CPU) of the N > 1 host-side logic: marker sharding by the PETSC_DECIDE block rule, the
unique-id broadcast plumbing bench.py uses, and that summing per-rank partial charge grids with an all-reduce
reproduces the single-rank density (the role of MPI_Allreduce at src/pic1dp_interaction.F90:132-133)."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import pic1dp_b200 as P
        from helpers import OracleRun, copy_state, make_params, synth_markers
        op, _ = make_params(nx=192)
        n = 50001
        st = synth_markers(op, n, seed=77)          # every rank generates the same global arrays
        lo, hi = P.petsc_decide(n, world, rank)     # ... and keeps its own contiguous block
        mine = {k: a[lo:hi].copy() for k, a in st.items()}
        # unique-id style broadcast of an opaque 128-byte token from rank 0
        tok = [bytes(range(128)) if rank == 0 else None]
        dist.broadcast_object_list(tok, src=0)
        assert tok[0] == bytes(range(128))
        # local deposit (charge2 of this rank), then all-reduce, then scale: :81-141
        run = OracleRun(op, [[mine]])
        c1, _ = run.o.deposit_species(mine["x"], mine["w"])
        c2 = torch.from_numpy(c1 * op.charge[0])
        dist.all_reduce(c2, op=dist.ReduceOp.SUM)
        rho = c2.numpy() * op.nx / op.lx
        counts = [torch.zeros(1, dtype=torch.int64) for _ in range(world)]
        dist.all_gather(counts, torch.tensor([hi - lo]))
        if rank == 0:
            single = OracleRun(op, [[copy_state(st)]])
            single.collect_charge()
            err = float(np.max(np.abs(rho - single.rho)) / np.max(np.abs(single.rho)))
            q.put(("ok", err, int(sum(int(c) for c in counts))))
    except Exception as e:  # pragma: no cover
        q.put(("fail", repr(e), 0))
    finally:
        dist.destroy_process_group()


def test_two_rank_sharding_and_allreduce_gloo():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    status, err, total = q.get(timeout=180)
    for p in procs:
        p.join(timeout=60)
    assert status == "ok", err
    assert total == 50001
    assert err < 1e-12


def _opt_worker(rank, world, port, q):
    """Marker optimisation across ranks (src/pic1dp_particle.F90:356-522): per-rank |w| histogram, all-reduce, then the
    product's host half of particle_merge on this rank's block against the oracle's."""
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import ctypes as C
        import pic1dp_b200 as P
        from helpers import make_params, synth_markers
        from oracle import oracle as O
        from pic1dp_b200 import _capi
        op, _ = make_params(nx=64)
        n = 60001
        st = synth_markers(op, n, seed=5, spread=0.2)
        st["w"] = st["w"] * (1.0 + 50.0 * np.exp(-(st["v"] - 3.2) ** 2)) * np.sign(np.sin(7.0 * st["x"]) + 0.3)
        lo, hi = P.petsc_decide(n, world, rank)
        mine = {k: a[lo:hi].copy() for k, a in st.items()}
        orc = O.Oracle(op)
        local = torch.from_numpy(orc.dist_pertb_abs_v([mine["v"]], [mine["w"]], 128, 8.0))
        dist.all_reduce(local, op=dist.ReduceOp.SUM)                 # MPI_Allreduce :392-395
        dist_v = local.numpy().copy()
        ref = {k: a.copy() for k, a in mine.items()}
        n_ref = orc.particle_merge(ref, hi - lo, dist_v, 0.3, 8.0)
        dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
        n_got = _capi.load().pic1dp_host_particle_merge(hi - lo, dp(mine["x"]), dp(mine["v"]), dp(mine["p"]), dp(mine["w"]),
                                                        dp(dist_v), 128, 8.0, 0.3, op.nx, op.lx)
        same = n_got == n_ref and all(np.array_equal(mine[k][:n_ref], ref[k][:n_ref]) for k in ("x", "v", "p", "w"))
        res = [None] * world
        dist.all_gather_object(res, (bool(same), int(n_ref), hi - lo, dist_v))
        if rank == 0:
            blocks = [P.petsc_decide(n, world, r) for r in range(world)]
            whole = orc.dist_pertb_abs_v([st["v"][a:b].copy() for a, b in blocks], [st["w"][a:b].copy() for a, b in blocks],
                                         128, 8.0)
            err = float(np.max(np.abs(res[0][3] - whole)) / np.max(whole))
            q.put(("ok", err, [r[:3] for r in res], bool(np.array_equal(res[0][3], res[1][3]))))
    except Exception as e:  # pragma: no cover
        q.put(("fail", repr(e), [], False))
    finally:
        dist.destroy_process_group()


def test_two_rank_marker_optimisation_gloo():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 31500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_opt_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    status, err, per_rank, identical = q.get(timeout=180)
    for p in procs:
        p.join(timeout=60)
    assert status == "ok", err
    assert err < 1e-13 and identical            # the all-reduced histogram is the emulated-rank one, same on both ranks
    assert all(ok and n_after < n_before for ok, n_after, n_before in per_rank)


def test_bench_reference_arm_runs_on_cpu():
    """`bench.py --impl reference` is the CPU arm: must work without a GPU and print one JSON line."""
    import json
    import subprocess
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--cpu-markers", "200000"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["value"] > 0 and line["unit"] == "particle-steps/s"
    assert line["cpu_baseline"]["kind"] == "port" and line["e2e"]["h2d_bytes_per_step"] == 0


def test_bench_trace_analysis_separates_skew_from_exchange_floor():
    """bench.py --p2p-trace: per all-reduce and rank d = wait_exit - publish on that rank's own clock; the last
    arrival's d is the exchange floor, the rest is arrival skew.  Synthetic stamps with known skew and unsynchronised
    clocks must come back out."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    cap, nep, ranks = 64, 40, 4
    rng = np.random.default_rng(0)
    clock_offset = [0, 5_000_000, -3_000_000, 123]          # ns: the GPUs' %globaltimer are not synchronised
    rows = []
    arrive = np.cumsum(rng.integers(900_000, 1_100_000, size=nep + 1))   # true time the LAST rank publishes
    skews = rng.integers(0, 30_000, size=(nep + 1, ranks))
    skews[:, 2] = 0                                                      # rank 2 always arrives last
    for r in range(ranks):
        st = np.zeros((cap, 3), dtype=np.int64)
        for e in range(1, nep + 1):
            pub = arrive[e] - skews[e, r] + clock_offset[r]
            st[e % cap] = (pub, pub + 3_000, arrive[e] + 4_500 + clock_offset[r])    # boundary 3 us, floor 4.5 us
        rows.append((st, nep))
    t = bench.analyse_trace(rows, nep, cap)
    assert t["allreduces"] == nep and t["ranks"] == ranks
    assert abs(t["exchange_floor_min_over_ranks"]["median"] - 4.5) < 1e-9
    assert abs(t["kernel_boundary_publish_to_wait_entry"]["median"] - 3.0) < 1e-9
    assert abs(t["arrival_skew_wait"]["mean"] - skews[1:].mean() / 1e3) < 1e-9
    assert abs(t["per_step_cost_us"]["skew_worst_rank"] - 2 * skews[1:].max(axis=1).mean() / 1e3) < 1e-9


def test_bench_dump_outputs_writes_field_and_a_fixed_marker_sample(tmp_path):
    """bench.py --dump-outputs: the field arrays whole, the markers at the same seeded indices on every run, in float64,
    within 64 MB; a marker set no larger than the sample is written whole."""
    sys.path.insert(0, ROOT)
    import bench

    class FakeGpu:   # the Pic1dGpu calls dump_outputs makes
        def __init__(self, n):
            self.mk = {k: np.arange(n, dtype=np.float64) + i for i, k in enumerate("xvpw")}

        def get_field(self):
            return dict(electric=np.full(16, 1.0), chargeden=np.full(16, 2.0), mode_re=np.ones(1), mode_im=np.zeros(1))

        def get_markers_ptr(self, isp):
            return self.mk["x"].size

        def get_markers(self, isp, want):
            return {k: self.mk[k].copy() for k in want}

    n = 3 * bench.DUMP_MARKERS + 7
    bench.dump_outputs(FakeGpu(n), str(tmp_path / "a"))
    bench.dump_outputs(FakeGpu(n), str(tmp_path / "b"))
    names = ("electric", "chargeden", "mode_re", "mode_im", "x", "v", "p", "w")
    assert sorted(os.listdir(tmp_path / "a")) == sorted(k + ".npy" for k in names)
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 64 << 20
    a = {k: np.load(tmp_path / "a" / (k + ".npy")) for k in names}
    b = {k: np.load(tmp_path / "b" / (k + ".npy")) for k in names}
    assert all(a[k].dtype == np.float64 and np.array_equal(a[k], b[k]) for k in names)
    assert np.array_equal(a["electric"], np.full(16, 1.0))
    x = a["x"]
    assert x.size == bench.DUMP_MARKERS and np.all(np.diff(x) > 0) and x[-1] < n   # distinct indices, in order
    assert all(np.array_equal(a[k], x + i) for i, k in enumerate("xvpw"))            # one index set for all four
    bench.dump_outputs(FakeGpu(1000), str(tmp_path / "c"))
    assert np.array_equal(np.load(tmp_path / "c" / "w.npy"), np.arange(1000) + 3.0)


def test_bench_rank_seeds_are_valid_kiss64_states_and_rank_dependent():
    sys.path.insert(0, ROOT)
    import bench
    a, b, a2 = bench.rank_seeds(0), bench.rank_seeds(1), bench.rank_seeds(0)
    assert a == a2 and a != b and len(a) == 4
    assert a[1] != 0 and a[3] < (1 << 58) + 1      # xorshift word non-zero, carry in range after the warm-up
