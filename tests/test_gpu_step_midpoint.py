"""step() against the per-substep calls where step() runs the recomputed-midpoint kernel pair.

At iptclshape 4 with the direct kernels, step()'s first substep stores only w' and its second substep rebuilds the
midpoint x' = wrap(x0 + dt/2 v0) and v' = v0 + dt/2 E_n(x0) Z/m from the start-of-step state and a copy of the field
the first substep gathered.  The per-substep push(1) / push(2) keep storing the midpoint, so the two call sequences
must agree: bitwise with the deterministic deposits, to 1e-12 with the fp64-atomic ones.  nx = 8192 with the
fixed-point deposit has no room for the second field table and keeps the stored-midpoint kernels in step().
"""
import numpy as np
import pytest

import pic1dp_b200 as P
from helpers import make_params, rel_err, synth_markers

pytestmark = pytest.mark.gpu

NP = 60_001   # odd and not a multiple of any CTA tile: the scalar tail path runs in both substeps


def _case(case, **over):
    """Model variants of test_gpu_parity.py::test_model_variants_three_steps at the bench grid."""
    kw = dict(nx=1024, capacity=NP + 64, deposit_mode=P.DEPOSIT_FIXED)
    kw.update(over)
    nsp = 1
    if case == "maxwell":
        kw.update(iptcldist=0, density=[1.0], v0=[0.0])
    elif case == "fullf":
        kw.update(deltaf=0, iptcldist=0, density=[1.0], v0=[0.0])
    elif case == "linear":
        kw.update(linear=1)
    elif case == "two_species":
        nsp = 2
        kw.update(nspecies=2, charge=[-1.0, 1.0], mass=[1.0, 4.0], temperature=[1.0, 0.5], temperature2=[1.0, 0.5],
                  density=[0.9, 1.0], v0=[5.0, 0.0], iptcldist=3)
    elif case == "pow2_nonunit":
        kw.update(temperature=[2.0], mass=[0.5], temperature2=[0.5])
    elif case == "nonpow2":
        kw.update(temperature=[1.3], mass=[0.9], temperature2=[0.7])
    elif case == "tolerance":
        kw.update(arith_mode=P.ARITH_TOLERANCE)
    op, gp = make_params(**kw)
    sts = [synth_markers(op, NP - 7 * s, seed=40 + s, isp=s) for s in range(nsp)]
    return op, gp, sts


def _edge_markers(gp, st):
    """Overwrite markers with ones that reach every branch of the midpoint rebuild (x0 + dt/2 v0 on lx, just below 0,
    more than a box away; x0 on cell edges, at 0 and below 2^-800 where the division x0 / lx takes the IEEE redo),
    inside full tiles and in the tail.  The far-away markers need |v| ~ 1e3: only with the Maxwellian (no exponential
    in -d ln f0 / dv), and with p = w = 0 so that they deposit nothing."""
    lx, dth = gp.lx, 0.5 * gp.dt
    x, v, p, w = st["x"].copy(), st["v"].copy(), st["p"].copy(), st["w"].copy()
    xs, vs = [], []
    for v0 in (1.0, 1.5, 2.0, 2.5, 3.0, 0.75):   # x0 + dth v0 == lx exactly
        x0 = lx - dth * v0
        for x1 in (x0, np.nextafter(x0, 0.0), np.nextafter(x0, 2 * lx)):
            if x1 + dth * v0 == lx and 0.0 <= x1 < lx:
                xs.append(x1)
                vs.append(v0)
    for v0 in (-1.0, -2.0, -0.5):                 # x0 + dth v0 just below 0: the wrap adds lx, may round to lx
        x0 = -dth * v0
        xs += [x0, np.nextafter(x0, 0.0), np.nextafter(np.nextafter(x0, 0.0), 0.0)]
        vs += [v0] * 3
    nfar = 0
    if gp.iptcldist == 0:
        for k in (3.0, -2.5, 7.25):               # more than a box length away: fmod on the redo path
            xs.append(0.5 * lx)
            vs.append(k * lx / dth)
        nfar = 3
    for j in (0, 1, 511, 1023):                   # cell edges
        xs.append(j * lx / gp.nx)
        vs.append(0.3)
    xs += [0.0, 1e-300, 5e-324]                   # zero, below 2^-800 and denormal x0: the division's IEEE redo
    vs += [0.4, -0.2, 0.1]
    n = len(x)
    where = [5, 6, 2047, 2048, 40_000, 40_001] + list(range(n - 3, n))
    assert len(xs) == len(vs) > len(where)
    where += list(range(1000, 1000 + len(xs) - len(where)))
    for j, (i, xi, vi) in enumerate(zip(where, xs, vs)):
        x[i], v[i] = xi, vi
        if len(xs) - 7 - nfar <= j < len(xs) - 7:
            p[i] = w[i] = 0.0
    return dict(x=x, v=v, p=p, w=w)


def _run(gp, sts, nsteps, use_step, set_E=None):
    with P.Pic1dGpu(gp) as g:
        for s, st in enumerate(sts):
            g.set_markers(s, st["x"], st["v"], st["p"], st["w"])
        g.collect_charge()
        g.solve_field()
        for it in range(nsteps):
            if set_E is not None and it == 1:
                g.set_field(electric=set_E)
            if use_step:
                g.step(1)
            else:
                for irk in (1, 2):
                    g.push(irk)
                    g.collect_charge()
                    g.solve_field()
        mk = [g.get_markers(s) for s in range(len(sts))]
        return mk, g.get_field(), g.counters().oob_markers


def _compare(a, b, bitwise):
    mka, fa, oa = a
    mkb, fb, ob = b
    assert oa == ob
    for ma, mb in zip(mka, mkb):
        for k in ("x", "v", "w"):
            if bitwise:
                assert np.array_equal(ma[k], mb[k]), k
            else:
                assert rel_err(ma[k], mb[k]) < 1e-12, k
    for k in ("chargeden", "electric"):
        if bitwise:
            assert np.array_equal(fa[k], fb[k]), k
        else:
            assert rel_err(fa[k], fb[k]) < 1e-12, k


@pytest.mark.parametrize("case", ["unit", "tolerance", "pow2_nonunit", "nonpow2", "maxwell", "fullf", "linear",
                                  "two_species"])
def test_step_equals_substeps_at_bench_grid(case):
    op, gp, sts = _case(case)
    sts[0] = _edge_markers(gp, sts[0])
    _compare(_run(gp, sts, 3, False), _run(gp, sts, 3, True), bitwise=True)


@pytest.mark.parametrize("dep", [P.DEPOSIT_SMEM_ATOMIC, P.DEPOSIT_GLOBAL_RED, P.DEPOSIT_WARP_PRIVATE])
@pytest.mark.parametrize("case", ["unit", "nonpow2"])
def test_step_equals_substeps_other_deposits(dep, case):
    op, gp, sts = _case(case, deposit_mode=dep)
    sts[0] = _edge_markers(gp, sts[0])
    _compare(_run(gp, sts, 2, False), _run(gp, sts, 2, True), bitwise=(dep == P.DEPOSIT_WARP_PRIVATE))


def test_set_field_between_steps():
    """The second substep gathers the field the first one used, also when the caller replaced it in between."""
    op, gp, sts = _case("unit")
    rng = np.random.default_rng(5)
    E = 1e-3 * rng.standard_normal(gp.nx)
    _compare(_run(gp, sts, 3, False, set_E=E), _run(gp, sts, 3, True, set_E=E), bitwise=True)


def test_graph_replay_and_direct_launches_same_bits():
    outs = []
    for no_graph in (0, 1):
        op, gp, sts = _case("unit", no_step_graph=no_graph)
        sts[0] = _edge_markers(gp, sts[0])
        outs.append(_run(gp, sts, 3, True))
        if no_graph == 0:
            outs.append(_run(gp, sts, 3, False))
    _compare(outs[0], outs[1], bitwise=True)
    _compare(outs[0], outs[2], bitwise=True)


def test_large_grid_keeps_stored_midpoint():
    """nx = 8192 with the fixed-point pair grid: no room for a second field table, step() keeps the stored midpoint."""
    op, gp, sts = _case("unit", nx=8192)
    sts[0] = _edge_markers(gp, sts[0])
    _compare(_run(gp, sts, 2, False), _run(gp, sts, 2, True), bitwise=True)
