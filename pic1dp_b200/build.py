"""Builds libpic1dp_b200.so (hand-written sm_100a CUDA + C ABI) in-tree with nvcc.

The .so is git-ignored but travels to the GPU box with the gpurun snapshot.  nvcc cross-compiles without a GPU.
"""
from __future__ import annotations

import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libpic1dp_b200.so")
# translation units: (object name, source, extra defines).  The fused particle kernels are instantiated once per
# iptcldist in push_dist.cu, so the four equilibria (and the C ABI unit) compile in parallel.
UNITS = [("pic1dp_gpu", "pic1dp_gpu.cu", [])] + \
        [("push_dist%d" % d, "push_dist.cu", ["-DPIC1DP_DIST=%d" % d]) for d in range(4)]
HEADERS = ["particle_kernels.cuh", "field_kernels.cuh", "diag_kernels.cuh", "optimize_kernels.cuh", "optimize_host.hpp",
           "push_tables.hpp", "fp_strict.cuh", "grid_device.cuh", "loader_kernels.cuh", "rng_kernels.cuh", "kiss_jump_tables.h"]
OBJDIR = os.path.join(HERE, "build")
# generated, not committed: the MT19937-64 jump polynomials, written into the object directory before compiling
MT_GEN = os.path.join(HERE, "..", "tools_py3", "gen_mt_jump.py")
MT_TABLES = "mt_jump_tables.h"
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC",
    "-Xcompiler", "-ffp-contract=off",   # host-side arithmetic (marker optimisation) must not be contracted to FMA
]


def _extra_flags():
    """Experiment hook: PIC1DP_NVCC_EXTRA='-DPIC1DP_PF_MASK=5 ...' builds a variant (used with PIC1DP_B200_LIB)."""
    return os.environ.get("PIC1DP_NVCC_EXTRA", "").split()


def _headers():
    return [os.path.join(CSRC, f) for f in HEADERS if os.path.exists(os.path.join(CSRC, f))] + \
        [os.path.join(HERE, "..", "include", "pic1dp_gpu.h")]


def _unit_hash(src, defines) -> str:
    import hashlib
    h = hashlib.sha256()
    for d in [os.path.join(CSRC, src), MT_GEN] + _headers():
        h.update(open(d, "rb").read())
    h.update(" ".join(NVCC_FLAGS + defines + _extra_flags()).encode())
    return h.hexdigest()


def _source_hash() -> str:
    """Content hash of everything the library is built from (mtimes do not survive the copy to a GPU box)."""
    import hashlib
    h = hashlib.sha256()
    for name, src, defines in UNITS:
        h.update(_unit_hash(src, defines).encode())
    return h.hexdigest()


def needs_build(lib: str = LIB) -> bool:
    if not os.path.exists(lib) or not os.path.exists(lib + ".hash"):
        return True
    return open(lib + ".hash").read().strip() != _source_hash()


def _compile_unit(args):
    name, src, defines, objdir, verbose, force = args
    obj = os.path.join(objdir, name + ".o")
    hh = _unit_hash(src, defines)
    if not force and os.path.exists(obj) and os.path.exists(obj + ".hash") and open(obj + ".hash").read().strip() == hh:
        return obj, ""
    nvcc = os.environ.get("NVCC", "nvcc")
    cmd = [nvcc] + NVCC_FLAGS + defines + _extra_flags() + (["-Xptxas", "-v"] if verbose else []) + \
        ["-I", objdir, "-c", "-o", obj, os.path.join(CSRC, src)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
    with open(obj + ".hash", "w") as f:
        f.write(hh)
    return obj, r.stderr


def write_mt_tables(path: str) -> None:
    """Run tools_py3/gen_mt_jump.py's generator into path (rewritten only when its text changes)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("gen_mt_jump", MT_GEN)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    mod.write(path)


def build(force: bool = False, verbose: bool = False, lib: str = LIB, objdir: str = OBJDIR) -> str:
    """nvcc -c every unit (in parallel, content-hashed objects), then link the shared library in-tree."""
    if not (force or needs_build(lib)):
        return lib
    from concurrent.futures import ThreadPoolExecutor
    os.makedirs(objdir, exist_ok=True)
    write_mt_tables(os.path.join(objdir, MT_TABLES))
    with ThreadPoolExecutor(max_workers=len(UNITS)) as ex:
        res = list(ex.map(_compile_unit, [(n, s, d, objdir, verbose, force) for n, s, d in UNITS]))
    if verbose:
        for _, log in res:
            print(log)
    nvcc = os.environ.get("NVCC", "nvcc")
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", lib] + [o for o, _ in res] + ["-ldl"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
    with open(lib + ".hash", "w") as f:
        f.write(_source_hash())
    return lib


HOST_SRC = os.path.join(HERE, "..", "host", "pic1dp_host.cpp")
HOST_EXE = os.path.join(HERE, "..", "host", "pic1dp_host")


def build_host(force: bool = False) -> str:
    """C++ host driver above the C ABI (host/pic1dp_host.cpp): the reference's `program pic1dp` sequence."""
    build()
    import hashlib
    hh = hashlib.sha256(open(HOST_SRC, "rb").read() + open(os.path.join(HERE, "..", "include", "pic1dp_gpu.h"), "rb").read()).hexdigest()
    if not force and os.path.exists(HOST_EXE) and os.path.exists(HOST_EXE + ".hash") and \
            open(HOST_EXE + ".hash").read().strip() == hh:
        return HOST_EXE
    cmd = ["g++", "-O2", "-std=c++17", "-pthread", "-I", os.path.join(HERE, "..", "include"), HOST_SRC,
           "-L", HERE, "-lpic1dp_b200", "-Wl,-rpath,$ORIGIN/../pic1dp_b200", "-o", HOST_EXE]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("g++ failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
    with open(HOST_EXE + ".hash", "w") as f:
        f.write(hh)
    return HOST_EXE


if __name__ == "__main__":
    import sys
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
    print(build_host(force="--force" in sys.argv))
