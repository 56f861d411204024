"""The push kernels' redo path against the oracle, on markers that raise every source of the fast body's `rare` flag.

Markers come from tests/push_edges.py: cold species whose -d ln f0 / dv needs libdevice exp beyond |a| = 700 or the
IEEE division out of range, placed by the launch geometry (both lanes of a pair, one lane with a calm partner, a whole
warp, a warp with one redoing lane, the last CTA, CTA 0's second persistent iteration, the partial tail, the last
marker).  w is held to a per-marker bound, so a tail marker is held to its own size, and the deposit is checked with
zero-weight ordinary markers, so that a redone pair deposited twice or never is an O(1) error.

The staged load paths (TMA ring, cp.async) map the TOLERANCE instantiations (cfg 33, 57) to the strict cfg 1 kernel,
so a TOLERANCE handle runs strict arithmetic in every substep whose ring fits, and is held to the STRICT bound there.
"""
import os

import numpy as np
import pytest

import pic1dp_b200 as P
import push_edges as PE
from helpers import ChunkedOracleRun, OracleRun, copy_state, make_params, rel_err, synth_markers

pytestmark = pytest.mark.gpu

SETS = list(PE.CONSTANT_SETS)
CASES = [(d, n) for d in (3, 2) for n in SETS]
DEPOSITS = [P.DEPOSIT_FIXED, P.DEPOSIT_SMEM_ATOMIC, P.DEPOSIT_GLOBAL_RED, P.DEPOSIT_WARP_PRIVATE]
ARITH = [P.ARITH_STRICT, P.ARITH_TOLERANCE]
CAPACITY = 700_000
E_AMP = 0.05


def _field(nx, phase=0.3):
    return E_AMP * np.sin(2 * np.pi * np.arange(nx) / nx + phase)


def _params(dist, name, arith, _op=None, **gpu):
    """Matching (oracle, GPU) parameters; _op: copy the model of these oracle parameters instead of a named set."""
    if _op is not None:
        kw = {k: (list(getattr(_op, k))[:_op.nspecies] if k in ("charge", "mass", "temperature", "temperature2",
                                                                "density", "v0") else getattr(_op, k))
              for k in ("iptcldist", "linear", "iptclshape", "charge", "mass", "temperature", "temperature2",
                        "density", "v0")}
    else:
        kw = PE.params_kw(dist, name)
    kw.update(nx=256, capacity=CAPACITY, arith_mode=arith)
    kw.update(gpu)
    return make_params(**kw)


def _handle(gp):
    """Pic1dGpu, or a skip where the configuration has no such kernel (EUNSUPPORTED)."""
    try:
        return P.Pic1dGpu(gp)
    except P.Pic1dpError as e:
        assert e.code == 8, e    # PIC1DP_EUNSUPPORTED
        pytest.skip("no kernel of this load path for this deposit mode / configuration")


def _markers(g, op, dist, tol, seed=0, zero_ordinary=False, load_path=None, weight=1.0):
    """Markers laid out by this handle's launch geometry, catalogue markers in the hostile slots.  weight scales the
    hostile markers' p and w: runs that solve for the field keep it small, so that the field they make moves no
    marker's exponential argument by more than the catalogue's margin (into the 0/0 of both exponentials zero)."""
    c = g.counters()
    tile = 1024 if load_path == P._capi.LOAD_TMA else 2 * c.cta_threads
    n, hostile, calm = PE.layout(c.grid_ctas, tile)
    assert n <= CAPACITY
    base = synth_markers(op, n, seed=seed)
    src = synth_markers(op, 20_000, seed=seed + 1)
    ok = PE.calm_mask(op, dist, src["v"])
    calm_src = {k: a[ok] for k, a in src.items()}
    cat = PE.catalogue(op, dist, tol, seed=seed)
    cat["p"] = weight * cat["p"]
    cat["w"] = weight * cat["w"]
    st = PE.place(base, cat, hostile, calm_src, calm)
    if zero_ordinary:
        mask = np.ones(n, bool)
        mask[hostile] = False
        st["p"][mask] = 0.0
        st["w"][mask] = 0.0
    return st, hostile


def _tol_kernel(op, gp, fuse, load_path=None):
    """Whether the push runs dlnf0_tol_n: TOLERANCE mode, fused, a specialised (cfg > 0) direct kernel."""
    return (gp.arith_mode == P.ARITH_TOLERANCE and fuse and op.linear == 0 and op.iptclshape >= 3 and
            load_path in (None, P._capi.LOAD_DIRECT, P._capi.LOAD_AUTO))


def _check_w(op, dist, pre, w_gpu, w_o, dt, E, tol):
    tmp1 = PE.tmp1_of(op, pre["p"], pre["w"], PE.gather(op, E, pre["x"]))
    bound = PE.w_bound(op, dist, pre["v"], w_o, tmp1, dt, tol)
    err = np.abs(w_gpu - w_o)
    bad = np.flatnonzero(~(err <= bound))
    assert bad.size == 0, (bad[:8], w_gpu[bad[:8]], w_o[bad[:8]], bound[bad[:8]], pre["v"][bad[:8]])


def _substeps(gp, op, dist, fuse, load_path=None, seed=0):
    E = _field(op.nx)
    tol = _tol_kernel(op, gp, fuse, load_path)
    # A staged load path runs the strict cfg 1 kernel for a TOLERANCE handle, but a substep whose ring does not fit
    # beside the deposit grids runs the direct TOLERANCE kernel instead.  A STRICT twin handle tells them apart: a
    # substep that matches the twin bit for bit ran the strict kernel and is held to the STRICT bound; any other is
    # held to the TOLERANCE bound, the bound of the direct kernel.
    twin = None
    if load_path is not None and gp.arith_mode == P.ARITH_TOLERANCE:
        _, tgp = _params(op.iptcldist, None, P.ARITH_STRICT, _op=op, deposit_mode=gp.deposit_mode, fuse=1,
                         load_path=load_path)
        twin = _handle(tgp)
    try:
        with _handle(gp) as g:
            st, hostile = _markers(g, op, dist, gp.arith_mode == P.ARITH_TOLERANCE, seed=seed, load_path=load_path)
            ref = OracleRun(op, [[copy_state(st)]])
            ref.E = E.copy()
            g.set_markers(0, st["x"], st["v"], st["p"], st["w"])
            g.set_field(electric=E)
            if twin is not None:
                twin.set_markers(0, st["x"], st["v"], st["p"], st["w"])
                twin.set_field(electric=E)
            for irk in (1, 2):
                r = ref.st[0][0]
                pre = {k: r[k].copy() for k in ("x", "v", "p", "w")}
                ref.push(irk)
                g.push(irk)
                if twin is not None:
                    twin.push(irk)
                    twin.collect_charge()
                    wt = twin.get_markers(0, want=("w",))["w"]
                    twin.set_field(electric=E)
                if not fuse:
                    assert np.array_equal(g.get_markers(0, want=("x",))["x"], r["x"]), irk   # unwrapped, as the reference
                ref.collect_charge()     # the wrap (and the out-of-range count) of the following deposit
                g.collect_charge()
                out = g.get_markers(0)
                assert np.array_equal(out["x"], r["x"]), irk
                assert np.array_equal(out["v"], r["v"]), irk
                assert np.array_equal(out["p"], st["p"]), irk
                assert np.array_equal(g.get_shape_x(0)[0], ref.o.shape(r["x"].copy())[0]), irk
                assert g.counters().oob_markers == ref.noob, irk
                dt = 0.5 * op.dt if irk == 1 else op.dt
                if twin is not None:
                    tol = not np.array_equal(out["w"], wt)
                _check_w(op, dist, pre, out["w"], r["w"], dt, E, tol)
                moved = np.abs(r["w"][hostile] - pre["w"][hostile])
                assert np.median(moved) > 1e-6     # the hostile markers' w update is not trivially small
                r["w"][:] = out["w"]     # continue from identical state so irk = 2 isolates one substep
                g.set_field(electric=E)
                ref.E = E.copy()
    finally:
        if twin is not None:
            twin.close()


@pytest.mark.parametrize("dep", DEPOSITS)
@pytest.mark.parametrize("arith", ARITH)
@pytest.mark.parametrize("dist,name", CASES)
def test_substeps_against_oracle(dist, name, arith, dep):
    op, gp = _params(dist, name, arith, deposit_mode=dep, fuse=1)
    _substeps(gp, op, dist, True, seed=11)


@pytest.mark.parametrize("dist,name", CASES)
def test_unfused_substeps_against_oracle(dist, name):
    op, gp = _params(dist, name, P.ARITH_TOLERANCE, fuse=0)
    _substeps(gp, op, dist, False, seed=12)


@pytest.mark.parametrize("load_path", [P._capi.LOAD_TMA, P._capi.LOAD_CPASYNC])
@pytest.mark.parametrize("dep", [P.DEPOSIT_SMEM_ATOMIC, P.DEPOSIT_GLOBAL_RED, P.DEPOSIT_WARP_PRIVATE])
@pytest.mark.parametrize("arith", ARITH)
@pytest.mark.parametrize("dist,name", CASES)
def test_staged_load_paths_against_oracle(dist, name, arith, dep, load_path):
    op, gp = _params(dist, name, arith, deposit_mode=dep, fuse=1, load_path=load_path)
    _substeps(gp, op, dist, True, load_path=load_path, seed=13)


def _run(gp, sts, nsteps, use_step):
    with _handle(gp) as g:
        for s, st in enumerate(sts):
            g.set_markers(s, st["x"], st["v"], st["p"], st["w"])
        g.collect_charge()
        g.solve_field()
        if use_step:
            g.step(nsteps)
        else:
            for _ in range(nsteps):
                for irk in (1, 2):
                    g.push(irk)
                    g.collect_charge()
                    g.solve_field()
        return [g.get_markers(s) for s in range(len(sts))], g.get_field(), g.counters().oob_markers


def _same_bits(a, b):
    mka, fa, oa = a
    mkb, fb, ob = b
    assert oa == ob
    for ma, mb in zip(mka, mkb):
        for k in ("x", "v", "w"):
            assert np.array_equal(ma[k], mb[k]), k
    for k in ("chargeden", "electric"):
        assert np.array_equal(fa[k], fb[k]), k


@pytest.mark.parametrize("no_graph", [0, 1])
@pytest.mark.parametrize("dep", [P.DEPOSIT_FIXED, P.DEPOSIT_WARP_PRIVATE])
@pytest.mark.parametrize("arith", ARITH)
@pytest.mark.parametrize("dist,name", CASES)
def test_step_equals_substeps(dist, name, arith, dep, no_graph):
    """step() (the recomputed-midpoint kernels at iptclshape 4, graph-replayed or launched directly) against three
    rounds of push / collect_charge / solve_field: bitwise."""
    op, gp = _params(dist, name, arith, deposit_mode=dep, no_step_graph=no_graph)
    with _handle(gp) as g:
        st, _ = _markers(g, op, dist, arith == P.ARITH_TOLERANCE, seed=21, weight=1e-3)
    _same_bits(_run(gp, [st], 3, False), _run(gp, [st], 3, True))


@pytest.mark.parametrize("dep", [P.DEPOSIT_FIXED, P.DEPOSIT_WARP_PRIVATE])
@pytest.mark.parametrize("arith", ARITH)
def test_step_equals_substeps_two_species(arith, dep):
    """A cold bump-on-tail species carrying the hostile markers beside a default species."""
    kw = dict(nx=256, capacity=CAPACITY, arith_mode=arith, deposit_mode=dep, nspecies=2, iptcldist=3,
              charge=[-1.0, 1.0], mass=[0.9, 1.0], temperature=[0.3, 1.0], temperature2=[0.05, 1.0],
              density=[0.9, 0.9], v0=[5.0, 5.0])
    op, gp = make_params(**kw)
    with _handle(gp) as g:
        st, _ = _markers(g, op, 3, arith == P.ARITH_TOLERANCE, seed=22, weight=1e-3)
    sts = [st, synth_markers(op, 150_001, seed=23, isp=1)]
    _same_bits(_run(gp, sts, 3, False), _run(gp, sts, 3, True))


@pytest.mark.parametrize("dist,name", [(3, "nonpow2-cold"), (2, "pow2-cold")])
def test_three_steps_against_oracle(dist, name):
    """step(3) with hostile markers against the oracle's driver loop, at the suite's summation-order bars."""
    op, gp = _params(dist, name, P.ARITH_STRICT, deposit_mode=P.DEPOSIT_FIXED)
    with _handle(gp) as g:
        st, _ = _markers(g, op, dist, False, seed=24, weight=1e-3)
    ref = OracleRun(op, [[copy_state(st)]])
    ref.init_field()
    for _ in range(3):
        ref.step()
    mk, f, noob = _run(gp, [st], 3, True)
    assert rel_err(f["chargeden"], ref.rho) < 1e-12 and rel_err(f["electric"], ref.E) < 1e-12
    for k in ("x", "v", "w"):
        assert rel_err(mk[0][k], ref.st[0][0][k]) < 1e-12, k
    assert noob == ref.noob


def _check_deposit(g, op, dep):
    """rho of the last deposit against the fsum reference of the GPU's own (wrapped) x and w."""
    mk = g.get_markers(0, want=("x", "w"))
    rho = g.get_field()["chargeden"]
    rho_ref, bound, fixed_extra = PE.deposit_reference(op, [mk["x"]], [mk["w"]])
    if dep == P.DEPOSIT_FIXED:
        bound = bound + fixed_extra
    assert np.max(np.abs(rho_ref)) > 1e-6
    bad = np.flatnonzero(~(np.abs(rho - rho_ref) <= bound))
    assert bad.size == 0, (bad[:8], rho[bad[:8]], rho_ref[bad[:8]], bound[bad[:8]])


@pytest.mark.parametrize("fuse", [1, 0])
@pytest.mark.parametrize("dep", DEPOSITS)
@pytest.mark.parametrize("arith", ARITH)
@pytest.mark.parametrize("dist,name", [(3, "unit"), (3, "nonpow2-cold"), (2, "pow2-cold"), (3, "generic-shape2")])
def test_deposit_exactly_once(dist, name, arith, dep, fuse):
    """Ordinary markers carry p = w = 0, hostile markers O(1): rho per cell against the exactly rounded sum after
    push(1), push(2) and (fused) a step(), whose kernels are the recomputed-midpoint ones at iptclshape 4."""
    op, gp = _params(dist, name, arith, deposit_mode=dep, fuse=fuse)
    with _handle(gp) as g:
        st, _ = _markers(g, op, dist, arith == P.ARITH_TOLERANCE, seed=31, zero_ordinary=True, weight=1e-3)
        g.set_markers(0, st["x"], st["v"], st["p"], st["w"])
        g.set_field(electric=_field(op.nx))
        for irk in (1, 2):
            g.push(irk)
            g.collect_charge()
            _check_deposit(g, op, dep)
            g.solve_field()
        if fuse:
            g.step(1)
            _check_deposit(g, op, dep)


# ---- the bench state ---------------------------------------------------------------------------------------------
N_BENCH = 100_000_000
NCHUNK = max(4, min(32, os.cpu_count() or 4))


def _bench_markers(g, op):
    """Default bump-on-tail markers with ~1e4 hostile ones (default constants, |v| in 28 .. 38) on full tiles deep in
    the persistent loop and on the tail."""
    c = g.counters()
    G, tile = c.grid_ctas, 2 * c.cta_threads
    st = synth_markers(op, N_BENCH, seed=103)
    cat = PE.catalogue(op, 3, False, seed=5)
    sweeps = N_BENCH // (G * tile)
    idx = []
    for k in (sweeps // 3, 2 * sweeps // 3, sweeps - 1):
        for cta in (0, G // 4, G // 2, G - 1):
            B = (k * G + cta) * tile
            idx += [B + 2, B + 3, B + 6, B + 11] + list(range(B + 64, B + 128)) + [B + 146]
    for k in (sweeps // 2, sweeps - 2):     # whole tiles of hostile markers
        B = (k * G + 7) * tile
        idx += list(range(B, B + tile))
    idx += list(range(N_BENCH // tile * tile, N_BENCH))      # the partial tail tile
    idx = np.unique(np.array(idx, dtype=np.int64))
    j = np.arange(idx.size) % cat["v"].size
    # p and w at the size of the ordinary markers' p and w, so that max |w|, which sets the fixed-point deposit's
    # quantum, stays what it is without them
    pmax, wmax = float(np.max(st["p"])), float(np.max(np.abs(st["w"])))
    for key in ("x", "v"):
        st[key][idx] = cat[key][j]
    st["p"][idx] = pmax * cat["p"][j]
    st["w"][idx] = 2 * wmax * cat["w"][j]
    assert 5000 <= idx.size <= 20000
    return st, idx


def test_bench_state_step_equals_substeps():
    """(a) step(2) at the bench state (the recomputed-midpoint kernels, graph-replayed, fixed-point deposit) equals
    the per-substep sequence bit for bit."""
    op, gp = make_params(nx=1024, capacity=N_BENCH)
    outs = []
    for use_step in (True, False):
        with P.Pic1dGpu(gp) as g:
            if use_step:
                st, _ = _bench_markers(g, op)
            g.set_markers(0, st["x"], st["v"], st["p"], st["w"])
            g.collect_charge()
            g.solve_field()
            if use_step:
                g.step(2)
                assert g.counters().graph_replays == 2 and g.counters().deposit_mode == P.DEPOSIT_FIXED
            else:
                for _ in range(2):
                    for irk in (1, 2):
                        g.push(irk)
                        g.collect_charge()
                        g.solve_field()
            outs.append((g.get_markers(0, want=("x", "v", "w")), g.get_field()))
    for k in ("x", "v", "w"):
        assert np.array_equal(outs[0][0][k], outs[1][0][k]), k
    for k in ("chargeden", "electric"):
        assert np.array_equal(outs[0][1][k], outs[1][1][k]), k


def test_bench_state_against_oracle():
    """(b) one step() against the oracle: rho, E within 1e-12 of max, x, v, w within 1e-12; (c) both substeps with a
    prescribed E: x, v and the cell index bit-exact for every marker, w within the per-marker bound."""
    op, gp = make_params(nx=1024, capacity=N_BENCH)
    with P.Pic1dGpu(gp) as g:
        st, idx = _bench_markers(g, op)
        ref = ChunkedOracleRun(op, copy_state(st), NCHUNK)
        g.set_markers(0, st["x"], st["v"], st["p"], st["w"])
        ref.init_field()
        g.collect_charge()
        g.solve_field()
        ref.step()
        g.step(1)
        f = g.get_field()
        assert rel_err(f["chargeden"], ref.rho) < 1e-12 and rel_err(f["electric"], ref.E) < 1e-12
        out = g.get_markers(0, want=("x", "v", "w"))
        for k in ("x", "v", "w"):
            assert rel_err(out[k], ref.full[k]) < 1e-12, k
        del out, ref
        # (c): both substeps from the initial markers with a prescribed E
        E = 1e-3 * np.sin(2 * np.pi * np.arange(op.nx) / op.nx + 0.3)
        g.set_markers(0, st["x"], st["v"], st["p"], st["w"])
        ref = ChunkedOracleRun(op, st, NCHUNK)     # advances st in place
        for irk in (1, 2):
            g.set_field(electric=E)
            ref.E = E.copy()
            pre = {k: ref.full[k].copy() for k in ("x", "v", "p", "w")}
            ref.push(irk)
            ref.collect_charge()
            g.push(irk)
            g.collect_charge()
            out = g.get_markers(0, want=("x", "v", "w"))
            assert np.array_equal(out["x"], ref.full["x"]), irk
            assert np.array_equal(out["v"], ref.full["v"]), irk
            assert np.array_equal(g.get_shape_x(0)[0], ref.cell_index()), irk
            dt = 0.5 * op.dt if irk == 1 else op.dt
            ch = 10_000_000
            for lo in range(0, N_BENCH, ch):
                s = slice(lo, lo + ch)
                _check_w(op, 3, {k: a[s] for k, a in pre.items()}, out["w"][s], ref.full["w"][s], dt, E, False)
            moved = np.abs(ref.full["w"][idx] - pre["w"][idx])
            assert np.median(moved) > 0
            ref.full["w"][:] = out["w"]
            del out, pre
