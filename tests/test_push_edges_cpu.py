"""The hostile-marker catalogue and the per-marker w bound of tests/push_edges.py, checked without a GPU.

- every catalogue marker raises the flags its construction aims at (and no x-side flag), and the division's range
  flag agrees with an independent high-precision evaluation;
- every catalogue marker has a finite reference w, and the TOLERANCE-only cases are finite only for cold species;
- the float64 restatement reproduces the oracle's w bit for bit;
- the w bound has 2x headroom against +-1 and +-2 ulp errors of each exponential, over the catalogue and 1e5
  ordinary markers;
- the fsum deposit reference holds the oracle's own sequential deposit within its per-cell bound.
"""
import math
from decimal import Decimal, localcontext

import numpy as np
import pytest

import push_edges as PE
from helpers import make_params, synth_markers
from oracle import oracle as O

CASES = [(d, n) for d in (3, 2) for n in PE.CONSTANT_SETS]
E_AMP = 0.05


def _field(op):
    return E_AMP * np.sin(2 * np.pi * np.arange(op.nx) / op.nx + 0.3)


def _op(dist, name):
    return make_params(**PE.params_kw(dist, name))[0]


def _oracle_substep(op, st, E, irk=1):
    """One oracle push (irk) from state st; returns the new w and the dt it used."""
    x, v, p, w = (np.array(st[k], float) for k in ("x", "v", "p", "w"))
    n = x.size
    xb, vb, wb = np.zeros(n), np.zeros(n), np.zeros(n)
    if irk == 2:
        xb, vb, wb = x.copy(), v.copy(), w.copy()
    O.Oracle(op).push_species(0, irk, x, v, p, w, xb, vb, wb, E)
    return w, (0.5 * op.dt if irk == 1 else op.dt)


def _dec_log2(q):
    with localcontext() as ctx:
        ctx.prec = 60
        return float(abs(q).ln() / Decimal(2).ln()) if q != 0 else -math.inf


def _exact_num_den(c, dist, v):
    """num and den of orc_dlnf0 from the (double) arguments with exact exponentials and exact sums (Decimal, 60
    digits): an evaluation independent of the float64 restatement."""
    a1, a2 = PE.strict_args(c, dist, np.array([v]))
    with localcontext() as ctx:
        ctx.prec = 60
        e1, e2 = (Decimal(-float(a)).exp() for a in (a1[0], a2[0]))
        V, D = Decimal(float(v)), Decimal
        if dist == 3:
            vm = V - D(c.v0)
            num = D(c.n) * V / D(c.Tm) * e1 / D(c.sqTm) + D(c.omn) * vm / D(c.T2m) * e2 / D(c.sqT2m)
            den = D(c.n) * e1 / D(c.sqTm) + D(c.omn) * e2 / D(c.sqT2m)
        else:
            num = (V + D(c.v0)) * e1 + (V - D(c.v0)) * e2
            den = e1 + e2
    return num, den


@pytest.mark.parametrize("dist,name", CASES)
@pytest.mark.parametrize("tol", [False, True])
def test_catalogue_raises_the_flags_its_labels_name(dist, name, tol):
    op = _op(dist, name)
    c = PE.SpeciesConst(op)
    cat = PE.catalogue(op, dist, tol)
    assert len(cat["v"]) >= 20
    a1, a2 = PE.strict_args(c, dist, cat["v"])
    nd = PE.tol_nd(c, dist, cat["v"])
    for i, (tag, lab) in enumerate(zip(cat["tags"], cat["labels"])):
        assert "xdiv" not in lab and "wrap" not in lab, tag
        v = cat["v"][i]
        if not tol:
            if "above700" in tag or "beyond" in tag:
                assert "exp" in lab, tag
            if "at-or-below700" in tag or tag.endswith("-below700") or tag.endswith("-at700"):
                k = int(tag.split("-e")[1][0]) if tag.startswith("strict-e") else 0
                own = (a1, a2)[k - 1][i] if k else None
                if k:
                    assert own <= PE.EXP_BOUND, tag
                    assert ("exp" in lab) == (max(a1[i], a2[i]) > PE.EXP_BOUND), tag
            if tag == "strict-div-alone":
                assert lab == frozenset({"div"}), (tag, v)
            # the division's range flag, independently
            num, den = _exact_num_den(c, dist, v)
            l2n, l2d = _dec_log2(num), _dec_log2(den)
            if min(abs(l2n + 500), abs(l2d + 500), abs(l2n - 500), abs(l2d - 500)) > 1e-6:
                out = not (-500 <= l2n < 500 and -500 <= l2d < 500)
                assert ("div" in lab) == out, (tag, v, l2n, l2d)
        else:
            if tag.startswith("tol-nd") and "beyond" in tag:
                assert "exp" in lab and abs(nd[i]) > PE.EXP_BOUND, tag
            if tag.startswith("tol-nd") and "above700" in tag:
                assert "exp" in lab and abs(nd[i]) > PE.EXP_BOUND, tag
            if tag.startswith("tol-nd") and ("below700" in tag or tag.endswith("at700")):
                assert "exp" not in lab and abs(nd[i]) <= PE.EXP_BOUND, tag
            if tag.startswith("tol-den"):
                lnr = float(tag.split("-")[-1])
                assert ("div" in lab) == (lnr > 500 * math.log(2.0)), tag
            if abs(nd[i]) <= PE.EXP_BOUND - 1:
                assert "exp" not in lab, tag
    # the edges sit on both sides of 700: the largest reachable argument <= 700 and the smallest above it
    if not tol:
        at = [i for i, t in enumerate(cat["tags"]) if t.startswith("strict-e1-at")]
        ab = [i for i, t in enumerate(cat["tags"]) if t.startswith("strict-e1-above700")]
        for i in at:
            assert 700.0 - 4 * np.spacing(700.0) <= a1[i] <= 700.0
        for i in ab:
            assert 700.0 < a1[i] <= 700.0 + 4 * np.spacing(700.0)


def test_catalogue_covers_every_source_and_result_range():
    """Across the constant sets: exp alone, exp with div, div alone (STRICT and TOLERANCE), and exp_slow results that
    are normal, subnormal and zero with a positive denominator."""
    seen = set()
    kinds = set()
    for dist, name in CASES:
        op = _op(dist, name)
        c = PE.SpeciesConst(op)
        for tol in (False, True):
            cat = PE.catalogue(op, dist, tol)
            seen |= {(tol, lab) for lab in cat["labels"]}
            if not tol:
                a1, a2 = PE.strict_args(c, dist, cat["v"])
                for x in np.concatenate([PE.cexp(-a1[a1 > 700]), PE.cexp(-a2[a2 > 700])]):
                    kinds.add("zero" if x == 0 else "subnormal" if x < 2.0 ** -1022 else "normal")
    for want in [(False, frozenset({"exp"})), (False, frozenset({"exp", "div"})), (False, frozenset({"div"})),
                 (True, frozenset({"exp"})), (True, frozenset({"div"}))]:
        assert want in seen, want
    assert kinds == {"zero", "subnormal", "normal"}


@pytest.mark.parametrize("dist", [3, 2])
def test_catalogue_has_positive_tolerance_arguments_past_the_overflow(dist):
    """TOLERANCE markers whose exponential argument -nd lies in (709.8, 745] with a finite reference: there exp
    overflows, and the fast polynomial's exponent add wraps into a tiny negative r that no division flag catches, so
    only the bound at 700 sends them to the redo."""
    op = _op(dist, "cold-beam")
    c = PE.SpeciesConst(op)
    cat = PE.catalogue(op, dist, True)
    nd = PE.tol_nd(c, dist, cat["v"])
    hit = (-nd > math.log(np.finfo(float).max)) & (-nd <= 745.0)
    assert np.count_nonzero(hit) >= 3
    w, _ = _oracle_substep(op, {k: cat[k][hit] for k in ("x", "v", "p", "w")}, _field(op), 1)
    assert np.all(np.isfinite(w))
    r = PE.fast_exp_neg(nd[hit])
    assert np.all((r < 0) & (r > -1e-290))       # the wrapped result: tiny and negative, not huge
    tmp2, den = PE.tol_tmp2(c, dist, cat["v"][hit], r)
    assert np.all(PE._in_range(den) & (den > 0))   # ... so the division raises no flag
    ref = np.array([O.Oracle(op).dlnf0(0, v) for v in cat["v"][hit]])
    assert np.all(np.isfinite(ref))
    assert np.all(np.abs(tmp2 - ref) > 1e-3 * (1 + np.abs(ref)))   # a fast body past 700 would be visibly wrong
    assert all("exp" in cat["labels"][i] for i in np.flatnonzero(hit))


def test_fast_exp_restatement_matches_exp_inside_the_bound():
    """fast_exp_neg is exp_fast_neg_n: within ~1 ulp of exp over [-700, 700]."""
    na = np.linspace(-700.0, 700.0, 20001)
    fe, ce = PE.fast_exp_neg(na), PE.cexp(-na)
    assert np.max(np.abs(fe - ce) / ce) < 3 * PE.EPS


@pytest.mark.parametrize("dist,name", CASES)
def test_catalogue_reference_w_is_finite(dist, name):
    op = _op(dist, name)
    cat = PE.catalogue(op, dist, False)
    for irk in (1, 2):
        w, _ = _oracle_substep(op, cat, _field(op), irk)
        assert np.all(np.isfinite(w)), irk
        assert np.any(w != cat["w"])   # w moves: p - w is O(1)


@pytest.mark.parametrize("dist", [3, 2])
def test_tolerance_only_cases_are_0_over_0_for_unit_constants(dist):
    """|v^2 h1 - (v - v0)^2 h2| beyond 700 (bump-on-tail) and r + 1 >= 2^500 (two-stream2) have a finite reference
    only for cold species: with T = T2 = m = 1 both exponentials of the reference underflow there."""
    for name, finite in (("unit", False), ("nonpow2-cold", True), ("pow2-cold", True)):
        op = _op(dist, name)
        c = PE.SpeciesConst(op)
        vs = []
        if dist == 3:
            for nd in (PE.EXP_BOUND, -PE.EXP_BOUND, 800.0):
                vs += PE._tol_roots(c, dist, nd)
        else:
            vs += [500 * math.log(2.0) / c.tolk2 * f for f in (1.0, 1.2, 1.9)]
        vs = np.array([v for v in vs if math.isfinite(v)])
        if dist == 3 and name != "unit":
            vs = vs[[abs(PE.tol_nd(c, dist, np.array([v]))[0]) >= 699 for v in vs]]
        assert vs.size
        a1, a2 = PE.strict_args(c, dist, vs)
        tmp2 = PE.strict_terms(c, dist, vs, PE.cexp(-a1), PE.cexp(-a2))[0]
        ref = np.array([O.Oracle(op).dlnf0(0, v) for v in vs])
        assert np.array_equal(np.isnan(tmp2), np.isnan(ref))
        if finite:
            assert np.any(np.isfinite(ref)), name
        else:
            assert np.all(np.isnan(ref)), name


def _ordinary(op, dist, n=100_000, seed=3):
    st = synth_markers(op, n, seed=seed)
    st["p"] = st["p"] + 0.5    # O(1) p - w
    return st


@pytest.mark.parametrize("dist,name", CASES)
def test_restatement_reproduces_the_oracle_w_bit_for_bit(dist, name):
    op = _op(dist, name)
    E = _field(op)
    cat = PE.catalogue(op, dist, False)
    for st in (cat, _ordinary(op, dist, 20_000)):
        for irk in (1, 2):
            w_o, dt = _oracle_substep(op, st, E, irk)
            tmp1 = PE.tmp1_of(op, st["p"], st["w"], PE.gather(op, E, st["x"]))
            w_r = PE.w_strict(op, dist, st["v"], tmp1, st["w"], dt)
            assert np.array_equal(w_r, w_o), irk


def _headroom(op, dist, st, tol, E):
    """max over markers and perturbations of |w_pert - w_o| / bound."""
    c = PE.SpeciesConst(op)
    w_o, dt = _oracle_substep(op, st, E, 1)
    tmp1 = PE.tmp1_of(op, st["p"], st["w"], PE.gather(op, E, st["x"]))
    bound = PE.w_bound(op, dist, st["v"], w_o, tmp1, dt, tol)
    v, wb = st["v"], st["w"]
    worst = 0.0
    a1, a2 = PE.strict_args(c, dist, v)
    e1, e2 = PE.cexp(-a1), PE.cexp(-a2)
    use_tol = np.zeros(v.size, bool)
    if tol:   # the fast TOLERANCE body; markers it flags are redone with the strict scalar code
        fexp, fdiv = PE.w_flags(c, dist, v, True)
        use_tol = ~(fexp | fdiv)
        nd = PE.tol_nd(c, dist, v)
        r = PE.cexp(-nd)
    for k1 in (-2, -1, 0, 1, 2):
        for k2 in (-2, -1, 0, 1, 2):
            if k1 == k2 == 0:
                continue
            wp = PE.w_strict(op, dist, v, tmp1, wb, dt, PE.perturb_exp(e1, k1), PE.perturb_exp(e2, k2))
            if tol and k2 == 0:
                t = use_tol
                wp[t] = PE.w_tol(op, dist, v[t], tmp1[t], wb[t], dt, PE.perturb_exp(r[t], k1))
            q = np.abs(wp - w_o) / bound
            assert np.all(np.isfinite(q))
            worst = max(worst, float(np.max(q)))
    return worst


@pytest.mark.parametrize("dist,name", CASES)
@pytest.mark.parametrize("tol", [False, True])
def test_w_bound_has_twice_the_headroom(dist, name, tol):
    if tol and name.startswith("generic"):
        pytest.skip("the generic instantiation has no TOLERANCE form")
    op = _op(dist, name)
    E = _field(op)
    cat = PE.catalogue(op, dist, tol)
    assert _headroom(op, dist, cat, tol, E) <= 0.5
    assert _headroom(op, dist, _ordinary(op, dist), tol, E) <= 0.5


def test_layout_places_every_slot_inside_the_markers():
    for grid, tile in ((148, 2048), (296, 1024), (148, 1024), (3, 256)):
        n, hostile, calm = PE.layout(grid, tile)
        assert n % 2 == 1 and n == (grid + 1) * tile + tile // 2 + 7
        assert hostile[-1] == n - 1 and not set(hostile) & set(calm)
        # a whole warp of pairs in CTA 0's first tile, CTA 0's second iteration and the last CTA's first tile
        for B in (0, (grid - 1) * tile, grid * tile):
            assert set(range(B + 64, B + 128)) <= set(hostile)
            # one hostile lane in warp 2, every other marker of that warp calm
            assert (B + 146) in set(hostile) and len(set(range(B + 128, B + 192)) & set(calm)) == 63
        assert np.any(hostile >= (grid + 1) * tile)    # the partial tail tile


@pytest.mark.parametrize("dist,name", [(3, "nonpow2-cold"), (2, "pow2-cold"), (3, "generic-shape2")])
def test_fsum_deposit_reference_holds_the_oracle_deposit(dist, name):
    op = _op(dist, name)
    op.nx = 64
    st = _ordinary(op, dist, 50_000)
    cat = PE.catalogue(op, dist, False)
    n, hostile, calm = PE.layout(3, 256)
    base = {k: np.resize(st[k], n) for k in ("x", "v", "p", "w")}
    base["w"][:] = 0.0
    s = PE.place(base, cat, hostile, base, calm)
    rho_ref, bound, _ = PE.deposit_reference(op, [s["x"]], [s["w"]])
    rho, _ = O.Oracle(op).collect_charge([[s["x"].copy()]], [[s["w"]]])
    assert np.max(np.abs(rho_ref)) > 0.1
    assert np.all(np.abs(rho - rho_ref) <= bound)
