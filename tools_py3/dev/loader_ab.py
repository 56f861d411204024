"""Old-versus-new equivalence of particle_load's loader entry points: runs every loader and the three parity calls with
two builds of the library, each in its own process (the in-tree library, and the one PIC1DP_B200_LIB names, e.g. the
parent commit's build), and compares what they return.

Cases: every generator (KISS64, SuperKISS64, MT19937-64) with uniform-v and Maxwellian markers, plus the counter and the
host-stream loaders; (np, nlocal) in {(0, 0), (1, 1), (150 001, 200 003), (10 000 001, 10 000 001)}; two species
chained through the returned state; the Gaussian buffer empty and filled; table / block positions at the end (20632 /
312, multirand_init's) and in the middle (after the warm-up); parity lengths across a table / block boundary; refusals.
Compared: x, v, p, w (SHA-1 of the bytes), the returned state and Gaussian buffer, last_gaussian_load, return codes and
the per-call deltas of kernel_launches, h2d_bytes and d2h_bytes.

    python tools_py3/dev/loader_ab.py --base scratch/libBASE.so [--out profiles/r06_loader_ab.md]
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.join(HERE, "..", "..")
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SIZES = ((0, 0), (1, 1), (150_001, 200_003), (10_000_001, 10_000_001))
NAMES = {1: "kiss64", 2: "mt19937_64", 3: "superkiss64"}
NSEED = {1: 4, 2: 312, 3: 20635}
SK_STATE_BYTES = 20633 * 8   # the SuperKISS64 table and carry


def _u64(a):
    return a.ctypes.data_as(C.POINTER(C.c_uint64))


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _digest(a):
    return hashlib.sha1(np.ascontiguousarray(a).view(np.uint8)).hexdigest()


class Runner:
    def __init__(self, g):
        from pic1dp_b200 import host as H
        self.g, self.L = g, g.L
        self.modes = H._modes((1, 3), (2e-6, 0.0), (1e-5, 3e-6))

    def call(self, fn, *args):
        """rc and counter deltas of one entry point called on the handle."""
        c0 = self.g.counters()
        rc = getattr(self.L, fn)(self.g._h, *args)
        c1 = self.g.counters()
        return dict(rc=int(rc), launches=c1.kernel_launches - c0.kernel_launches, h2d=c1.h2d_bytes - c0.h2d_bytes,
                    d2h=c1.d2h_bytes - c0.d2h_bytes)

    def markers(self, isp):
        m = self.g.get_markers(isp)
        return {k: _digest(m[k]) for k in ("x", "v", "p", "w")} | {"n": int(m["x"].size)}

    def gauss_stats(self):
        return list(self.g.last_gaussian_load())


def oracle_state(al, start, spare=False):
    """(seeds, iseed, gauss_filled, gauss_buf) of the oracle generator: multirand_init's (start = "end": table / block
    position 20632 / 312) or after rank 1's warm-up and 100 draws ("mid"), then gaussian_array(7) when spare (one value
    buffered)."""
    from multirand_state import get_spare, get_state
    from oracle import oracle as O
    r = O.MultiRand()
    if start == "end":
        r.seed_default(al)
    else:
        r.init_const(al, 1, 5)
        r.real_array(100)
    if spare:
        r.gaussian_array(7)
    seeds, iseed = get_state(r)
    return (seeds[:NSEED[al]].copy(), iseed) + get_spare(r)


def state_record(seeds, iseed, filled=None, buf=None):
    d = dict(seeds=_digest(seeds), iseed=int(iseed))
    if filled is not None:
        d.update(filled=int(filled), buf=float(buf).hex())
    return d


def run_loads(R, out):
    im, ic, isn = R.modes
    nm = len(im)
    for al in (1, 2, 3):
        name = NAMES[al]
        for start in (("mid",) if al == 1 else ("mid", "end")):
            for np_, nlocal in SIZES:
                for kind in ("uniform", "maxwellian"):
                    for spare in ((False,) if kind == "uniform" else (False, True)):
                        seeds, iseed, filled, buf = oracle_state(al, start, spare)
                        off = 0
                        recs = []
                        for isp in (0, 1):   # two species chained through the returned state
                            pos, fl, bf = C.c_int32(iseed), C.c_int32(filled), C.c_double(buf)
                            if kind == "uniform" and al == 1:
                                rec = R.call("pic1dp_gpu_load_markers_kiss64", isp, np_, 2 * max(nlocal, 1),
                                             (C.c_uint64 * 4)(*[int(w) for w in seeds]), off, off + nlocal, C.c_double(8.0),
                                             nm, im, ic, isn)
                                off += 2 * nlocal
                            elif kind == "uniform":
                                rec = R.call(f"pic1dp_gpu_load_markers_{name}", isp, np_, nlocal, 2 * max(nlocal, 1),
                                             _u64(seeds), C.byref(pos), C.c_double(8.0), nm, im, ic, isn)
                            elif al == 1:
                                rec = R.call("pic1dp_gpu_load_markers_maxwellian_kiss64", isp, np_, nlocal,
                                             2 * max(nlocal, 1), _u64(seeds), C.byref(fl), C.byref(bf), nm, im, ic, isn)
                            else:
                                rec = R.call(f"pic1dp_gpu_load_markers_maxwellian_{name}", isp, np_, nlocal,
                                             2 * max(nlocal, 1), _u64(seeds), C.byref(pos), C.byref(fl), C.byref(bf),
                                             nm, im, ic, isn)
                            iseed, filled, buf = pos.value, fl.value, bf.value
                            rec["state"] = state_record(seeds, iseed, filled, buf)
                            if kind == "maxwellian":
                                rec["gauss"] = R.gauss_stats()
                            if rec["rc"] == 0:
                                rec["markers"] = R.markers(isp)
                            recs.append(rec)
                        out[f"{name}/{kind}/start={start}/np={np_}/nlocal={nlocal}/spare={int(spare)}"] = recs
    # the loaders this change keeps as they are: counter and host streams
    rng = np.random.default_rng(7)
    for np_, nlocal in SIZES:
        recs = []
        for isp in (0, 1):
            recs.append(R.call("pic1dp_gpu_load_markers_counter", isp, np_, 2 * max(np_, 1), C.c_uint64(1234),
                               isp * np_, C.c_double(8.0), nm, im, ic, isn))
            recs[-1]["markers"] = R.markers(isp)
        out[f"counter/np={np_}"] = recs
        u, x, gv = rng.random(np_), rng.random(np_), rng.standard_normal(np_)
        recs = [R.call("pic1dp_gpu_load_markers", 0, np_, 2 * max(np_, 1), _dp(u), _dp(x), C.c_double(8.0), nm, im, ic,
                       isn)]
        recs[-1]["markers"] = R.markers(0)
        recs.append(R.call("pic1dp_gpu_load_markers_maxwellian", 1, np_, 2 * max(np_, 1), _dp(gv), _dp(x), nm, im, ic,
                           isn))
        recs[-1]["markers"] = R.markers(1)
        out[f"host_stream/np={np_}"] = recs


def run_parity(R, out):
    seeds4 = oracle_state(1, "mid")[0]
    for off, n in ((0, 1), (7, 5), (1_000_003, 100_003)):
        o = np.empty(n)
        rec = R.call("pic1dp_gpu_kiss64_uniforms", (C.c_uint64 * 4)(*[int(w) for w in seeds4]), off, n, _dp(o))
        rec["out"] = _digest(o)
        out[f"kiss64/uniforms/offset={off}/n={n}"] = [rec]
    for al, N in ((2, 312), (3, 20632)):
        for start in ("mid", "end"):
            seeds, iseed, _, _ = oracle_state(al, start)
            recs = []
            for n in (1, 5, N + 7, 2 * N - 3, 100_003):   # chained: the lengths cross the table / block boundary
                o = np.empty(n)
                pos = C.c_int32(iseed)
                rec = R.call(f"pic1dp_gpu_{NAMES[al]}_uniforms", _u64(seeds), C.byref(pos), n, _dp(o))
                iseed = pos.value
                rec.update(out=_digest(o), state=state_record(seeds, iseed))
                recs.append(rec)
            out[f"{NAMES[al]}/uniforms/start={start}"] = recs


def run_refusals(R, Rdist, out):
    """Refused calls: the return code, no counter movement, the state and last_gaussian_load untouched."""
    im, ic, isn = R.modes
    nm = len(im)
    for al in (1, 2, 3):
        name = NAMES[al]
        seeds0, iseed0, _, _ = oracle_state(al, "mid")
        N = {1: 0, 2: 312, 3: 20632}[al]
        cases = [("nlocal<np", dict(np_=100, nlocal=99)), ("null_seeds", dict(null=True)),
                 ("capacity", dict(np_=10_000_002 + 5, nlocal=10_000_002 + 5)), ("null_gauss", dict(null_gauss=True))]
        if al != 1:
            cases += [("iseed=-1", dict(iseed=-1)), (f"iseed={N + 1}", dict(iseed=N + 1))]
        for kind in ("uniform", "maxwellian"):
            for tag, kw in cases + ([("iptcldist=3", dict(dist=True))] if kind == "maxwellian" else []):
                if (kind == "uniform" and (al == 1 or tag == "null_gauss")):
                    continue
                seeds = seeds0.copy()
                pos, fl, bf = C.c_int32(kw.get("iseed", iseed0)), C.c_int32(1), C.c_double(0.25)
                sp = None if kw.get("null") else _u64(seeds)
                np_, nlocal = kw.get("np_", 100), kw.get("nlocal", 100)
                RR = Rdist if kw.get("dist") else R
                gauss0 = RR.gauss_stats()
                flp = None if kw.get("null_gauss") else C.byref(fl)
                if kind == "uniform":
                    rec = RR.call(f"pic1dp_gpu_load_markers_{name}", 0, np_, nlocal, 1000, sp, C.byref(pos),
                                  C.c_double(8.0), nm, im, ic, isn)
                elif al == 1:
                    rec = RR.call("pic1dp_gpu_load_markers_maxwellian_kiss64", 0, np_, nlocal, 1000, sp, flp,
                                  C.byref(bf), nm, im, ic, isn)
                else:
                    rec = RR.call(f"pic1dp_gpu_load_markers_maxwellian_{name}", 0, np_, nlocal, 1000, sp, C.byref(pos),
                                  flp, C.byref(bf), nm, im, ic, isn)
                rec.update(state=state_record(seeds, pos.value, fl.value, bf.value),
                           gauss_untouched=RR.gauss_stats() == gauss0)
                out[f"refusal/{name}/{kind}/{tag}"] = [rec]
        if al != 1:
            seeds = seeds0.copy()
            pos = C.c_int32(N + 1)
            o = np.empty(4)
            rec = R.call(f"pic1dp_gpu_{name}_uniforms", _u64(seeds), C.byref(pos), 4, _dp(o))
            rec["state"] = state_record(seeds, pos.value)
            out[f"refusal/{name}/uniforms/iseed={N + 1}"] = [rec]
    o = np.empty(4)
    out["refusal/kiss64/uniforms/offset=-1"] = [R.call("pic1dp_gpu_kiss64_uniforms", (C.c_uint64 * 4)(1, 2, 3, 4), -1,
                                                       4, _dp(o))]


def child(path):
    import pic1dp_b200 as P
    cap = 10_000_002
    out = {}
    with P.Pic1dGpu(P.default_params(nx=256, capacity=cap, nspecies=2, iptcldist=0)) as g:
        R = Runner(g)
        run_loads(R, out)
        run_parity(R, out)
        with P.Pic1dGpu(P.default_params(nx=256, capacity=1000, iptcldist=3)) as g3:
            run_refusals(R, Runner(g3), out)
    with open(path, "w") as f:
        json.dump(dict(lib=P._capi._LIB_PATH, cases=out), f)


def expected_difference(key, a, b):
    """The one difference the refactor makes on a path these cases reach: a SuperKISS64 Maxwellian call with
    nlocal = 0 returns early and no longer moves its 165 KB state up and down."""
    if not key.startswith("superkiss64/maxwellian/") or "/nlocal=0/" not in key:
        return False
    for ra, rb in zip(a, b):
        da = {k: v for k, v in ra.items() if k not in ("h2d", "d2h")}
        db = {k: v for k, v in rb.items() if k not in ("h2d", "d2h")}
        if da != db or ra["h2d"] - rb["h2d"] != SK_STATE_BYTES or ra["d2h"] - rb["d2h"] != SK_STATE_BYTES:
            return False
    return True


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base", help="the library to compare against (PIC1DP_B200_LIB)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_loader_ab.md"))
    ap.add_argument("--child", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.child:
        child(a.child)
        return
    import tempfile
    from superkiss_load import gpu_info
    res = {}
    with tempfile.TemporaryDirectory() as tmp:
        for tag, lib in (("base", os.path.abspath(a.base)), ("new", "")):
            env = dict(os.environ, PIC1DP_B200_LIB=lib)
            path = os.path.join(tmp, tag + ".json")
            subprocess.run([sys.executable, os.path.abspath(__file__), "--child", path], env=env, check=True)
            res[tag] = json.load(open(path))
    base, new = res["base"]["cases"], res["new"]["cases"]
    assert base.keys() == new.keys()
    same, expected, unexpected = [], [], []
    for k in base:
        if base[k] == new[k]:
            same.append(k)
        elif expected_difference(k, base[k], new[k]):
            expected.append(k)
        else:
            unexpected.append(k)
    calls = sum(len(v) for v in base.values())
    lines = ["# Loader refactor: old-versus-new equivalence (`tools_py3/dev/loader_ab.py`)", "",
             f"GPU: {json.dumps(gpu_info())}", "",
             f"Base library: `{os.path.relpath(res['base']['lib'], ROOT)}`; new: the in-tree build.", "",
             f"{len(base)} cases, {calls} calls: {len(same)} cases identical, {len(expected)} with the expected "
             f"difference, {len(unexpected)} unexpected.", "",
             "Expected: a SuperKISS64 Maxwellian call with nlocal = 0 moves 165 064 B less each way "
             "(h2d_bytes and d2h_bytes); everything else about it is identical.", ""]
    for k in expected:
        lines.append(f"- {k}: h2d {[r['h2d'] for r in base[k]]} -> {[r['h2d'] for r in new[k]]}, "
                     f"d2h {[r['d2h'] for r in base[k]]} -> {[r['d2h'] for r in new[k]]}")
    if unexpected:
        lines += ["", "Unexpected differences:"]
        for k in unexpected:
            lines.append(f"- {k}: base {json.dumps(base[k])} new {json.dumps(new[k])}")
    lines += ["", "Identical cases:", ""] + [f"- {k}" for k in same]
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write("\n".join(lines) + "\n")
    print("\n".join(lines[:9 + len(expected) + (2 + len(unexpected) if unexpected else 0)]))
    sys.exit(1 if unexpected else 0)


if __name__ == "__main__":
    main()
