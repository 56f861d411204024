"""Hostile markers for the push kernels' redo path, and per-marker error bounds against the oracle (CPU only).

The 2-wide body of the fused push kernels (push_pair_fast, pic1dp_b200/csrc/particle_kernels.cuh) has no rare path:
an operand that needs an IEEE fallback only raises the thread's `rare` flag, and push_pair_slow redoes both markers
of the pair with the scalar functions.  The flag has four sources:

  exp   an exponential argument with |a| > 700 (exp_fast_neg_n; the scalar path calls libdevice exp)
  div   a division operand outside [2^-500, 2^500), or a denominator <= 0 (div_pos_n / div_fast_n)
  xdiv  x / lx next to a rounding midpoint, or x < 2^-800 (div_const_n)
  wrap  a wrap of more than one box length (wrap_n)

This module restates the w-path predicates in float64 with the kernels' operation order, which is the oracle's
(oracle/pic1dp_oracle.c orc_dlnf0), so every argument below is bit-identical to the one the kernel tests.  Fused
multiply-adds of the TOLERANCE form (dlnf0_tol_n) are evaluated exactly with fractions.Fraction and rounded once.
div_suspect's midpoint test of the w-path divisions (probability ~2^-50 per division) is not restated.

Exponentials use math.exp, the C library's exp that the oracle calls; numpy's own exp is a different implementation
and differs from it in the last bit for a few per cent of arguments.
"""
from __future__ import annotations

import math
from fractions import Fraction

import numpy as np

EPS = 2.0 ** -52
# Per-marker w bound: |w_gpu - w_o| <= 2 ulp(w_o) + W_BOUND_K * eps * |g| * S (see w_bound).
W_BOUND_K = 32.0
EXP_BOUND = 700.0

FLAG_NAMES = ("exp", "div", "xdiv", "wrap")

# name -> (species overrides, model overrides).  The CFG column is the instantiation the direct kernels select for a
# delta-f nonlinear shape-4 run (STRICT / TOLERANCE); "generic-*" select CFG -1 in both arithmetic modes.
CONSTANT_SETS = {
    "unit": (dict(temperature=[1.0], temperature2=[1.0], mass=[1.0]), {}),                  # CFG 25 / 57
    "pow2-cold": (dict(temperature=[0.25], temperature2=[2.0 ** -6], mass=[1.0]), {}),      # CFG 9 / 33
    "nonpow2-cold": (dict(temperature=[0.3], temperature2=[0.05], mass=[0.9]), {}),         # CFG 1 / 33
    "generic-linear": (dict(temperature=[0.3], temperature2=[0.05], mass=[0.9]), dict(linear=1)),      # CFG -1
    "generic-shape2": (dict(temperature=[0.3], temperature2=[0.05], mass=[0.9]), dict(iptclshape=2)),  # CFG -1
    # T/m = 0.025 below T2/m = 1: a cold bulk under a warm bump, and two-stream2 beams with v0 / v_th ~ 19.  The
    # TOLERANCE exponent's argument -nd (v^2 h1 - (v - v0)^2 h2, or v k2) passes +700 at ordinary velocities (near the
    # beam centre) while the reference stays finite; the sets above reach it only where both exponentials underflow.
    "cold-beam": (dict(temperature=[0.025], temperature2=[1.0], mass=[1.0]), {}),          # CFG 1 / 33
}
V0 = {3: 5.0, 2: 3.0}   # bump-on-tail: the default v0; two-stream2: two cold beams at +-3


def params_kw(dist, name):
    """Keyword arguments of helpers.make_params for (iptcldist, constant set)."""
    sp, model = CONSTANT_SETS[name]
    kw = dict(iptcldist=dist, v0=[V0[dist]], **sp, **model)
    return kw


class SpeciesConst:
    """species_const (pic1dp_b200/csrc/pic1dp_gpu.cu) in IEEE double, evaluated like the host does."""

    def __init__(self, op, isp=0):
        T, T2, m = op.temperature[isp], op.temperature2[isp], op.mass[isp]
        self.Z, self.m, self.T = op.charge[isp], m, T
        self.n, self.omn, self.v0 = op.density[isp], 1.0 - op.density[isp], op.v0[isp]
        self.Tm, self.T2m = T / m, T2 / m
        self.twoTm, self.twoT2m = 2.0 * T / m, 2.0 * T2 / m
        self.sqTm, self.sqT2m = math.sqrt(T / m), math.sqrt(T2 / m)
        self.tolA = self.n / (self.Tm * self.sqTm)
        self.tolB = self.omn / (self.T2m * self.sqT2m)
        self.tolC = self.n / self.sqTm
        self.tolD = self.omn / self.sqT2m
        self.tolh1 = 1.0 / self.twoTm
        self.tolh2 = 1.0 / self.twoT2m
        self.tolk2 = 2.0 * self.v0 / self.Tm
        self.tolmT = self.m / self.T
        self.Zm = self.Z / self.m


# ---- exact arithmetic helpers -------------------------------------------------------------------------------
def _fma1(x, y, z):
    """RN(x * y + z): the exact value as a ratio of integers (what Fraction(x) * Fraction(y) + Fraction(z) holds, with
    power-of-two denominators), then one correctly rounded integer division."""
    if not (math.isfinite(x) and math.isfinite(y) and math.isfinite(z)):
        return x * y + z
    (nx, dx), (ny, dy), (nz, dz) = x.as_integer_ratio(), y.as_integer_ratio(), z.as_integer_ratio()
    d = dx * dy
    try:
        if dz > d:
            return (nx * ny * (dz // d) + nz) / dz
        return (nx * ny + nz * (d // dz)) / d
    except OverflowError:
        return math.inf if Fraction(nx * ny, d) + Fraction(nz, dz) > 0 else -math.inf


def fma(a, b, c):
    """RN(a * b + c) of doubles elementwise, exact product and sum, rounded once; non-finite operands as numpy does."""
    a, b, c = np.broadcast_arrays(np.asarray(a, float), np.asarray(b, float), np.asarray(c, float))
    out = [_fma1(x, y, z) for x, y, z in zip(a.ravel().tolist(), b.ravel().tolist(), c.ravel().tolist())]
    return np.array(out, float).reshape(a.shape)


def cexp(a):
    """The C library's exp elementwise (the oracle's exp; +inf past the overflow, as C returns)."""
    def e(x):
        try:
            return math.exp(x)
        except OverflowError:
            return math.inf
    with np.errstate(over="ignore"):
        return np.frompyfunc(e, 1, 1)(np.asarray(a, float)).astype(float)


def ulps(x, k):
    """x moved by k ulps (np.nextafter, towards +inf for k > 0)."""
    x = np.array(x, float)
    for _ in range(abs(k)):
        x = np.nextafter(x, np.inf if k > 0 else -np.inf)
    return x


# exp_fast_neg_n's constants (particle_kernels.cuh: c_exp_poly, c_exp_red)
_EXP_POLY = [float.fromhex(h) for h in (
    "0x1.af38a9b0ec855p-26", "0x1.289185613a3d6p-22", "0x1.71de0dae63bb3p-19", "0x1.a019b90d2ae7ap-16",
    "0x1.a01a01a7c41d5p-13", "0x1.6c16c1788bd90p-10", "0x1.11111111109b3p-7", "0x1.5555555553d63p-5",
    "0x1.5555555555556p-3", "0x1.0000000000001p-1")]
_LOG2E, _LN2HI, _LN2LO = (float.fromhex(h) for h in ("0x1.71547652b82fep+0", "0x1.62e42fefa39efp-1",
                                                      "0x1.abc9e3b39803fp-56"))


def fast_exp_neg(na):
    """exp_fast_neg_n's value of exp(-na) as the fast body computes it, whatever |na| (it only flags |na| > 700):
    Cody-Waite reduction, the polynomial, and 2^n put in by an integer add to the high word, which wraps through the
    exponent and sign bits once n leaves the normal range."""
    import struct
    magic = 6755399441055744.0
    out = []
    for a in np.asarray(na, float).ravel().tolist():
        t = _fma1(-a, _LOG2E, magic)
        n = struct.unpack("<q", struct.pack("<d", t))[0] & 0xffffffff
        n = n - (1 << 32) if n >= 1 << 31 else n
        f = t - magic
        r = _fma1(f, -_LN2HI, -a)
        r = _fma1(f, -_LN2LO, r)
        q = _EXP_POLY[0]
        for c in _EXP_POLY[1:]:
            q = _fma1(q, r, c)
        pr = _fma1(r * r, q, r) + 1.0
        bits = struct.unpack("<Q", struct.pack("<d", pr))[0]
        hi = ((bits >> 32) + (n << 20)) & 0xffffffff
        out.append(struct.unpack("<d", struct.pack("<Q", (hi << 32) | (bits & 0xffffffff)))[0])
    return np.array(out, float).reshape(np.shape(na))


def perturb_exp(e, k):
    """An exponential moved by k ulps, the error a <= 1 ulp exp may make on either side.  An exponential that is exactly
    0 stays 0: the C library and libdevice both return +0 once the argument is below about -745.13, where the exact
    value is under half the smallest subnormal, so neither the oracle nor the redo path can return anything else."""
    return np.where(np.asarray(e) == 0.0, 0.0, ulps(e, k))


def _in_range(q):
    """div_pos_n's range test on one operand: |q| in [2^-500, 2^500) (the sign is masked off)."""
    aq = np.abs(q)
    return (aq >= 2.0 ** -500) & (aq < 2.0 ** 500)


# ---- the reference -d ln f0 / dv (orc_dlnf0) and its pieces -------------------------------------------------------
def strict_args(c, dist, v):
    """The two exponential arguments (positive), rounded exactly as the kernels and the oracle round them."""
    v = np.asarray(v, float)
    if dist == 3:
        vm = v - c.v0
        return (v * v) / c.twoTm, (vm * vm) / c.twoT2m
    vp, vm = v + c.v0, v - c.v0
    return (vp * vp) / c.twoTm, (vm * vm) / c.twoTm


def strict_terms(c, dist, v, e1, e2):
    """(tmp2, num, den, S) of orc_dlnf0 with the given exponentials.  S = (|a| + |b|) / den for bump-on-tail (a, b the
    two terms of the numerator), (|v+v0| ep + |v-v0| em) / (ep + em) m / T for two-stream2: the size of tmp2's
    sensitivity to relative errors of the exponentials."""
    v = np.asarray(v, float)
    with np.errstate(all="ignore"):
        if dist == 3:
            vm = v - c.v0
            a = ((c.n * v) / c.Tm * e1) / c.sqTm
            b = ((c.omn * vm) / c.T2m * e2) / c.sqT2m
            num = a + b
            den = (c.n * e1) / c.sqTm + (c.omn * e2) / c.sqT2m
            tmp2 = num / den
            S = (np.abs(a) + np.abs(b)) / den
        else:
            vp, vm = v + c.v0, v - c.v0
            num = vp * e1 + vm * e2
            den = e1 + e2
            tmp2 = num / den * c.m / c.T
            S = (np.abs(vp) * e1 + np.abs(vm) * e2) / den * c.m / c.T
    return tmp2, num, den, S


def tol_nd(c, dist, v):
    """dlnf0_tol_n's exponent operand nd (the kernel evaluates exp(-nd)) and its ratio's coefficients."""
    v = np.asarray(v, float)
    if dist == 3:
        vm = v - c.v0
        return fma(vm * vm, c.tolh2, -((v * v) * c.tolh1))
    return -(v * c.tolk2)


def tol_tmp2(c, dist, v, r):
    """dlnf0_tol_n with r = exp(-nd) given; (tmp2, den).  The kernel's division is within ~1 ulp of RN(num / den);
    RN is used here."""
    v = np.asarray(v, float)
    with np.errstate(all="ignore"):
        if dist == 3:
            vm = v - c.v0
            num = fma(c.tolB * vm, r, c.tolA * v)
            den = fma(c.tolD, r, c.tolC)
            return num / den, den
        num = fma(v - c.v0, r, v + c.v0)
        den = r + 1.0
        return num / den * c.tolmT, den


# ---- flags ------------------------------------------------------------------------------------------------------
def w_flags(c, dist, v, tol):
    """(exp, div) flags of the w path for velocities v: STRICT (dlnf0_impl_n) or TOLERANCE (dlnf0_tol_n).  The div
    flag is evaluated with the C library's exponentials, i.e. with the values the scalar redo sees; when the exp flag
    is raised the fast body's own division result is discarded anyway."""
    v = np.asarray(v, float)
    with np.errstate(all="ignore"):
        if not tol:
            a1, a2 = strict_args(c, dist, v)
            fexp = ~((np.abs(a1) <= EXP_BOUND) & (np.abs(a2) <= EXP_BOUND))
            _, num, den, _ = strict_terms(c, dist, v, cexp(-a1), cexp(-a2))
            fdiv = ~(_in_range(num) & _in_range(den) & (den > 0))
        else:
            nd = tol_nd(c, dist, v)
            fexp = ~(np.abs(nd) <= EXP_BOUND)
            _, den = tol_tmp2(c, dist, v, cexp(-nd))
            fdiv = ~(_in_range(den) & (den > 0))
    return fexp, fdiv


def xdiv_flag(x, lx):
    """div_const's test on x / lx: x < 2^-800, or the quotient within 2^-100 (relative) of a rounding midpoint (the
    kernel's residual test fires inside 2^-104; any marker this flags is at least suspicious)."""
    out = np.zeros(np.shape(x), bool)
    L = Fraction(lx)
    for i, xi in enumerate(np.asarray(x, float).ravel()):
        xi = float(xi)
        if not xi >= 2.0 ** -800:
            out.flat[i] = True
            continue
        q = Fraction(xi) / L
        r = float(q)
        lo, hi = math.nextafter(r, -math.inf), math.nextafter(r, math.inf)
        d = min(abs(q - (Fraction(r) + Fraction(lo)) / 2), abs(q - (Fraction(r) + Fraction(hi)) / 2))
        out.flat[i] = d <= q * Fraction(1, 2 ** 100)
    return out


def wrap_flag(x, lx):
    x = np.asarray(x, float)
    return ~((x > -lx) & (x < lx + lx))


def all_flags(c, dist, x, v, dt_half, lx, tol):
    """Flags a first substep raises for markers (x, v): the w path at v, the shape at x and at x + dt/2 v (after the
    wrap), the wrap itself.  Returns a list of frozensets of FLAG_NAMES."""
    fexp, fdiv = w_flags(c, dist, v, tol)
    xo = x + dt_half * v
    xw = np.where(xo >= lx, xo - lx, xo)
    xw = np.where(xo < 0.0, xo + lx, xw)
    fx = xdiv_flag(x, lx) | xdiv_flag(xw, lx)
    fw = wrap_flag(xo, lx)
    out = []
    for i in range(len(v)):
        s = {n for n, f in zip(FLAG_NAMES, (fexp[i], fdiv[i], fx[i], fw[i])) if f}
        out.append(frozenset(s))
    return out


# ---- the catalogue ----------------------------------------------------------------------------------------------
def _scan(f, v_guess, target, mode, half=160):
    """Among the doubles within `half` ulps of v_guess, the one whose f(v) is target ('eq', None if none is), the
    smallest f(v) above target ('above'), or the largest f(v) at or below target ('below')."""
    vs = v_guess + np.arange(-half, half + 1) * np.spacing(abs(v_guess))
    fv = np.asarray(f(vs), float)
    if mode == "eq":
        hit = np.flatnonzero(fv == target)
        return float(vs[hit[0]]) if hit.size else None
    if mode == "above":
        ok = np.flatnonzero(fv > target)
        return float(vs[ok[np.argmin(fv[ok])]]) if ok.size else None
    ok = np.flatnonzero(fv <= target)
    return float(vs[ok[np.argmax(fv[ok])]]) if ok.size else None


def _edge_vs(f, roots, target):
    """(tag suffix, v) at f(v) == target exactly, the first value above it, and target - 1e-9."""
    out = []
    for r in roots:
        if not math.isfinite(r):
            continue
        v = _scan(f, r, target, "eq")
        if v is None:
            v = _scan(f, r, target, "below")
            out.append(("at-or-below", v))
        else:
            out.append(("at", v))
        out.append(("above", _scan(f, r, target, "above")))
        out.append(("below", _scan(f, r, target - 1e-9, "below", half=4000)))
    return [(t, v) for t, v in out if v is not None]


def _strict_roots(c, dist, k, arg):
    """Velocities where the k-th strict exponential argument (k = 1, 2) equals arg."""
    if dist == 3:
        if k == 1:
            s = math.sqrt(arg * c.twoTm)
            return [s, -s]
        s = math.sqrt(arg * c.twoT2m)
        return [c.v0 + s, c.v0 - s]
    s = math.sqrt(arg * c.twoTm)
    return [s - c.v0, -s - c.v0] if k == 1 else [s + c.v0, -s + c.v0]


def _tol_roots(c, dist, nd):
    """Velocities where the TOLERANCE exponent operand equals nd."""
    if dist == 2:
        return [-nd / c.tolk2]
    h1, h2, v0 = c.tolh1, c.tolh2, c.v0
    qa, qb, qc = h2 - h1, -2.0 * v0 * h2, v0 * v0 * h2 - nd
    if qa == 0.0:
        return [-qc / qb]
    disc = qb * qb - 4 * qa * qc
    if disc < 0:
        return []
    sq = math.sqrt(disc)
    return [(-qb + sq) / (2 * qa), (-qb - sq) / (2 * qa)]


def catalogue_velocities(op, dist):
    """(tag, v) of every hostile velocity for this species, before the finiteness filter."""
    c = SpeciesConst(op)
    out = []
    for k in (1, 2):
        f = (lambda u, k=k: strict_args(c, dist, u)[k - 1])
        for t, v in _edge_vs(f, _strict_roots(c, dist, k, EXP_BOUND), EXP_BOUND):
            out.append((f"strict-e{k}-{t}700", v))
        for arg in (704.0, 708.0, 712.0, 725.0, 740.0, 745.0, 746.0, 760.0, 900.0):   # exp_slow: normal, subnormal, 0
            for v in _strict_roots(c, dist, k, arg):
                out.append((f"strict-e{k}-beyond-{arg:g}", v))
    # the division's range flag alone: every argument <= 700, the denominator below 2^-500
    grid = np.linspace(-60.0, 60.0, 48001)
    a1, a2 = strict_args(c, dist, grid)
    with np.errstate(all="ignore"):
        _, num, den, _ = strict_terms(c, dist, grid, np.exp(-a1), np.exp(-a2))
        lden = np.log2(den)
    ok = np.flatnonzero((np.maximum(a1, a2) < 690.0) & (lden < -505.0) & (lden > -1000.0))
    for i in ok[np.linspace(0, ok.size - 1, min(ok.size, 6)).astype(int)] if ok.size else []:
        out.append(("strict-div-alone", float(grid[i])))
    # TOLERANCE: the exponent operand across 700 (both signs), two-stream2's denominator r + 1 at 2^500
    for nd in (EXP_BOUND, -EXP_BOUND):
        f = (lambda u: np.abs(tol_nd(c, dist, u)))
        for t, v in _edge_vs(f, _tol_roots(c, dist, nd), EXP_BOUND):
            out.append((f"tol-nd{'+' if nd > 0 else '-'}-{t}700", v))
    # ... and beyond it on both sides.  A negative nd is a positive argument of the exponential: past ~709.78 the
    # polynomial's exponent add wraps through the sign bit into a tiny negative r, which leaves the denominator in
    # range, so the bound at 700 is the only test that sends such a marker to the redo.
    for nd in (704.0, 712.0, 725.0, 740.0, 745.0):
        for sgn in (1.0, -1.0):
            for v in _tol_roots(c, dist, sgn * nd):
                out.append((f"tol-nd{'+' if sgn > 0 else '-'}-beyond-{nd:g}", v))
    if dist == 2:
        for lnr in (500 * math.log(2.0) - 1e-6, 500 * math.log(2.0) + 1e-6, 400.0, 600.0, 699.0):
            out.append((f"tol-den-{lnr:.6f}", lnr / c.tolk2))
    return out


_CATALOGUES = {}


def catalogue(op, dist, arith_tol, seed=0):
    """Copy of the (memoised) catalogue of _catalogue."""
    key = (dist, bool(arith_tol), seed, op.lx, op.dt, op.linear, op.iptclshape, op.charge[0], op.mass[0],
           op.temperature[0], op.temperature2[0], op.density[0], op.v0[0])
    if key not in _CATALOGUES:
        _CATALOGUES[key] = _catalogue(op, dist, arith_tol, seed)
    cat = _CATALOGUES[key]
    return {k: (a.copy() if isinstance(a, np.ndarray) else list(a)) for k, a in cat.items()}


def _catalogue(op, dist, arith_tol, seed):
    """Hostile markers of one (iptcldist, constant set, arithmetic): dict x, v, p, w (O(1) p - w, so that w moves),
    tags and labels (frozensets of FLAG_NAMES the first substep raises).  Markers whose reference w is not finite, or
    whose reference denominator is subnormal (its own rounding is then coarser than eps, so no per-marker bound in
    eps holds), are left out."""
    c = SpeciesConst(op)
    tv = catalogue_velocities(op, dist)
    v = np.array([t[1] for t in tv])
    a1, a2 = strict_args(c, dist, v)
    tmp2, num, den, _ = strict_terms(c, dist, v, cexp(-a1), cexp(-a2))
    keep = np.isfinite(tmp2) & (den >= 2.0 ** -1022)
    v = v[keep]
    tags = [t[0] for t, k in zip(tv, keep) if k]
    rng = np.random.default_rng(seed)
    lx = op.lx
    x = lx * (0.2 + 0.6 * rng.random(v.size))
    p = 0.5 + rng.random(v.size)
    w = 0.5 * (rng.random(v.size) - 0.5)
    labels = all_flags(c, dist, x, v, 0.5 * op.dt, lx, arith_tol)
    return dict(x=x, v=v, p=p, w=w, tags=tags, labels=labels)


def calm_mask(op, dist, v, margin=10.0):
    """Velocities whose w path raises no flag in either arithmetic, with a margin (float64, no exact fma needed)."""
    c = SpeciesConst(op)
    v = np.asarray(v, float)
    a1, a2 = strict_args(c, dist, v)
    with np.errstate(all="ignore"):
        _, num, den, _ = strict_terms(c, dist, v, np.exp(-a1), np.exp(-a2))
        if dist == 3:
            vm = v - c.v0
            nd = vm * vm * c.tolh2 - v * v * c.tolh1
            tden = c.tolD * np.exp(-nd) + c.tolC
        else:
            nd = -(v * c.tolk2)
            tden = np.exp(-nd) + 1.0
    lim = EXP_BOUND - margin
    rng_ok = lambda q: (np.abs(q) > 2.0 ** (-500 + margin)) & (np.abs(q) < 2.0 ** (500 - margin))
    return (a1 < lim) & (a2 < lim) & (np.abs(nd) < lim) & rng_ok(num) & rng_ok(den) & rng_ok(tden)


# ---- placement by launch geometry --------------------------------------------------------------------------------
def layout(grid, tile):
    """Marker count and hostile slots for a persistent grid of `grid` CTAs dealing tiles of `tile` markers
    round-robin.  np = one sweep + one more full tile (CTA 0's second persistent iteration) + half a tile + 7 (the
    partial tail tile, odd).  Slots (marker indices; thread t of a tile at base B owns B + 2t and B + 2t + 1):
    both lanes of a pair, lane 0 alone, lane 1 alone (partner calm), a whole warp of hostile pairs, a warp with a
    single hostile lane (the others calm), in CTA 0's first tile, the last CTA's first tile and CTA 0's second
    iteration; the partial tail tile; the last marker.  Returns (np, hostile indices, calm indices)."""
    n = (grid + 1) * tile + tile // 2 + 7
    hostile, calm = [], []

    def tile_slots(B):
        h = [B + 2, B + 3,            # both lanes of thread 1
             B + 6, B + 11,           # lane 0 of thread 3, lane 1 of thread 5
             B + tile - 2, B + tile - 1]
        c_ = [B + 7, B + 10]          # their partners
        w = 1 if tile >= 128 else 0   # warp 1: every marker hostile
        h += list(range(B + 64 * w, B + 64 * w + 64)) if tile >= 128 else []
        if tile >= 192:               # warp 2: one hostile lane (lane 9's first marker), the rest calm
            h.append(B + 128 + 18)
            c_ += [i for i in range(B + 128, B + 192) if i != B + 128 + 18]
        return h, c_

    for B in (0, (grid - 1) * tile, grid * tile):
        h, c_ = tile_slots(B)
        hostile += h
        calm += c_
    tail = (grid + 1) * tile
    hostile += [tail, tail + 1, tail + 4, tail + tile // 2 - 1, n - 2, n - 1]
    calm += [tail + 5]
    hs = sorted(set(hostile))
    cs = sorted(set(calm) - set(hs))
    assert hs[-1] == n - 1 and all(0 <= i < n for i in hs + cs)
    return n, np.array(hs, dtype=np.int64), np.array(cs, dtype=np.int64)


def place(base, cat, hostile, calm_src, calm):
    """Copy of marker dict `base` with catalogue markers cycled into `hostile` and calm markers (from calm_src) into
    `calm`."""
    st = {k: base[k].copy() for k in ("x", "v", "p", "w")}
    k = np.arange(hostile.size) % cat["v"].size
    for key in ("x", "v", "p", "w"):
        st[key][hostile] = cat[key][k]
    j = np.arange(calm.size) % calm_src["v"].size
    for key in ("x", "v", "p", "w"):
        st[key][calm] = calm_src[key][j]
    return st


# ---- per-marker w bound -----------------------------------------------------------------------------------------
def gather(op, E, x):
    """The oracle's gathered field at x (orc_push_species: E[ix] sl + E[ix + 1] sr)."""
    from oracle import oracle as O
    ix, sl, sr = O.Oracle(op).shape(np.array(x, float), right_frac=(op.iptclshape <= 2))
    ixr = np.where(ix + 1 > op.nx - 1, 0, ix + 1)
    return E[ix] * sl + E[ixr] * sr


def w_bound(op, dist, v, w_o, tmp1, dt, tol, isp=0, k=W_BOUND_K):
    """Largest admissible |w_gpu - w_o| after one substep with identical inputs.

    The GPU and the oracle share every rounded exponential argument and differ only through exp (<= 1.05 ulp on the
    device by tests/csrc/exp_model.c, <= 1 ulp for libdevice and glibc).  A relative error d of e1 or e2 moves
    tmp2 = num / den by at most 2 S d (numerator and denominator), and the roundings after it (S dt tmp1 Z / m, the add
    to wb) stay at a few eps: about 12 eps |g| S in all with g = dt tmp1 Z / m, so k = 32 leaves room.  TOLERANCE
    rounds the difference of the two arguments (and its coefficients), an absolute error of ~eps (arg1 + arg2) in the
    exponent, hence the factor (1 + arg1 + arg2).  tests/test_push_edges_cpu.py checks 2x headroom of this bound."""
    c = SpeciesConst(op, isp)
    v = np.asarray(v, float)
    a1, a2 = strict_args(c, dist, v)
    with np.errstate(all="ignore"):
        _, _, _, S = strict_terms(c, dist, v, np.exp(-a1), np.exp(-a2))
    g = np.abs(dt * tmp1 * c.Z / c.m)
    fac = k * EPS * g * S
    if tol:
        fac = fac * (1.0 + a1 + a2)
    return 2.0 * np.spacing(np.abs(w_o)) + fac


def tmp1_of(op, p, w, electric):
    return (p * electric) if op.linear else ((p - w) * electric)


# ---- w of one substep, restated ---------------------------------------------------------------------------------
def w_strict(op, dist, v, tmp1, wb, dt, e1=None, e2=None, isp=0):
    """orc_push_species's w update (:329-330) with orc_dlnf0; e1, e2 default to the C library's exponentials."""
    c = SpeciesConst(op, isp)
    a1, a2 = strict_args(c, dist, v)
    e1 = cexp(-a1) if e1 is None else e1
    e2 = cexp(-a2) if e2 is None else e2
    tmp2 = strict_terms(c, dist, v, e1, e2)[0]
    with np.errstate(all="ignore"):
        return wb + dt * tmp1 * tmp2 * c.Z / c.m


def w_tol(op, dist, v, tmp1, wb, dt, r=None, isp=0):
    """push_n's TOLERANCE w update: fma(RN(tmp1 * RN(dt Z/m)), tmp2, wb) with dlnf0_tol_n's tmp2."""
    c = SpeciesConst(op, isp)
    nd = tol_nd(c, dist, v)
    r = cexp(-nd) if r is None else r
    tmp2 = tol_tmp2(c, dist, v, r)[0]
    cz = dt * c.Zm
    return fma(tmp1 * cz, tmp2, wb)


# ---- deposit reference ------------------------------------------------------------------------------------------
def deposit_reference(op, xs, qs):
    """rho of interaction_collect_charge (orc_collect_charge, src/pic1dp_interaction.F90:96-151) with every cell sum
    of sl q and sr q exactly rounded (math.fsum), and a per-cell bound for a deposit that sums the same products in
    any order.  xs, qs: per species (x wrapped).  Returns (rho, bound_float, bound_fixed_extra).

    Float deposits: the products RN(sl q), RN(sr q) are the oracle's; a cell receives n_j of them in some order, and the
    per-warp and per-CTA grids are added over at most n_j non-zero partials at each level (adding a zero is exact), so
    at most 3 n_j roundings of partial sums, each below eps sum_j |c|, plus the scaling by Z nx / lx:
    (3 n_j + 3) eps sum_j |c| |Z| nx / lx + 4 eps |rho_j|.
    Fixed-point deposit: every product is rounded to a quantum q_f (at most 2^-39 max |q| at 1e8 markers per GPU, less
    below) and then summed exactly; bound_fixed_extra = (n_j + 1) quanta on top of the float bound (which covers the
    conversion of each CTA's integer cell sum and the reduce over CTAs)."""
    from oracle import oracle as O
    nx, lx = op.nx, op.lx
    right_frac = op.iptclshape <= 2
    o = O.Oracle(op)
    rho_terms = [[] for _ in range(nx)]
    abs_sum = np.zeros(nx)
    nj = np.zeros(nx, dtype=np.int64)
    qmax = 0.0
    for s, (x, q) in enumerate(zip(xs, qs)):
        ix, sl, sr = o.shape(np.array(x, float), right_frac=right_frac)
        ixr = np.where(ix + 1 > nx - 1, 0, ix + 1)
        Z = op.charge[s]
        nz = np.flatnonzero(q != 0.0)
        cl, cr = sl[nz] * q[nz], sr[nz] * q[nz]
        qmax = max(qmax, float(np.max(np.abs(q), initial=0.0)))
        for j, cc in zip(np.concatenate([ix[nz], ixr[nz]]), np.concatenate([cl, cr])):
            rho_terms[j].append(float(cc) * Z)   # exact: |Z| is a power of two in every test here
            abs_sum[j] += abs(float(cc) * Z)
            nj[j] += 1
    scale = nx / lx
    rho = np.array([math.fsum(t) for t in rho_terms]) * scale
    if op.deltaf == 0:
        for s in range(op.nspecies):
            rho = rho - op.charge[s] * op.density[s]
    bound = (3 * nj + 3) * EPS * abs_sum * scale + 4 * EPS * np.abs(rho)
    fixed_extra = (nj + 1) * 2.0 ** -39 * qmax * scale * max(abs(op.charge[s]) for s in range(op.nspecies))
    return rho, bound, fixed_extra
