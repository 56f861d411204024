"""Host-side mirror of the reference's module interface for the hot path, over the C ABI.

The reference exposes the path as argument-less Fortran module procedures over module-global state
(/root/reference/src/pic1dp_interaction.F90:33,161; src/pic1dp_particle.F90:66,275,819;
src/pic1dp_field.F90:55,218,315) driven by `program pic1dp` (src/pic1dp.F90:63-109).  `Pic1dpModules` keeps
the same procedure names, the same implicit inputs (`global_irk`, the `input_*` parameters) and the same
error behaviour (every call leaves its status in `global_ierr`; non-zero raises, like CHKERRQ aborts), so a
test can replay the reference driver line by line.  The Fortran ISO_C_BINDING shim with the identical
structure is fortran/pic1dp_gpu_shim.F90.

Everything here is plumbing: the work happens in libpic1dp_b200.so.  There is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import numpy as np

from . import _capi
from ._capi import Counters, Params


class Pic1dpError(RuntimeError):
    def __init__(self, code: int, where: str, detail: str):
        self.code = code
        super().__init__(f"{where}: error {code} ({_capi.load().pic1dp_gpu_strerror(code).decode()}): {detail}")


def default_params(**over) -> Params:
    """Defaults of src/pic1dp_input.F90.  Keyword overrides: scalars, or sequences for per-species/per-mode fields."""
    p = Params()
    _capi.load().pic1dp_gpu_params_default(C.byref(p))
    for k, v in over.items():
        cur = getattr(p, k)
        if hasattr(cur, "__len__"):
            for i, vi in enumerate(v):
                cur[i] = vi
        else:
            setattr(p, k, v)
    return p


def _dp(a: Optional[np.ndarray]):
    if a is None:
        return None
    assert a.dtype == np.float64 and a.flags["C_CONTIGUOUS"], "fp64 C-contiguous arrays only"
    return a.ctypes.data_as(C.POINTER(C.c_double))


_KISS, _SK, _MT = (4, "KISS64"), (_capi.SUPERKISS64_NSEED, "SuperKISS64"), (_capi.MT19937_64_NSEED, "MT19937-64")


def _state_ptr(seeds: np.ndarray, nwords: int, name: str):
    """A generator state multirand_seeds(0:nwords-1), passed for in-place update (_state_ptr(seeds, *_SK))."""
    assert seeds.dtype == np.uint64 and seeds.size == nwords and seeds.flags["C_CONTIGUOUS"], \
        f"{name} state: C-contiguous uint64 array of {nwords} words"
    return seeds.ctypes.data_as(C.POINTER(C.c_uint64))


def _modes(init_mode, init_cos, init_sin):
    """The initial perturbation's mode numbers and cos / sin amplitudes as ctypes arrays of init_nmode elements."""
    nm = len(init_mode)
    return (C.c_int32 * nm)(*init_mode), (C.c_double * nm)(*init_cos), (C.c_double * nm)(*init_sin)


def _ptr(addr: int):
    return C.cast(C.c_void_p(addr), C.POINTER(C.c_double))


class Pic1dGpu:
    """RAII wrapper of one pic1dp_gpu_t handle (one GPU, one stream)."""

    def __init__(self, params: Params):
        self.L = _capi.load()
        self.params = params
        self._h = C.c_void_p()
        rc = self.L.pic1dp_gpu_create(C.byref(params), C.byref(self._h))
        if rc:
            self._h = C.c_void_p()
            raise Pic1dpError(rc, "pic1dp_gpu_create", self.L.pic1dp_gpu_last_error(None).decode())
        self.modes = [params.modes[m] for m in range(params.nmode)]   # the handle's kept-mode set

    def _ck(self, rc: int, where: str):
        if rc:
            raise Pic1dpError(rc, where, self.L.pic1dp_gpu_last_error(self._h).decode())

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.L.pic1dp_gpu_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ---- communicator ----
    def comm_unique_id(self) -> bytes:
        buf = (C.c_uint8 * _capi.UNIQUE_ID_BYTES)()
        rc = self.L.pic1dp_gpu_comm_unique_id(buf)
        if rc:
            raise Pic1dpError(rc, "pic1dp_gpu_comm_unique_id", self.L.pic1dp_gpu_last_error(None).decode())
        return bytes(buf)

    def comm_init(self, uid: bytes):
        buf = (C.c_uint8 * _capi.UNIQUE_ID_BYTES).from_buffer_copy(uid)
        self._ck(self.L.pic1dp_gpu_comm_init(self._h, buf), "pic1dp_gpu_comm_init")

    def p2p_export(self) -> bytes:
        buf = (C.c_uint8 * _capi.IPC_HANDLE_BYTES)()
        self._ck(self.L.pic1dp_gpu_p2p_export(self._h, buf), "pic1dp_gpu_p2p_export")
        return bytes(buf)

    def p2p_import(self, handles):
        """handles: list of nranks 64-byte IPC handles in rank order (all-gathered by the host)."""
        blob = b"".join(handles)
        buf = (C.c_uint8 * len(blob)).from_buffer_copy(blob)
        self._ck(self.L.pic1dp_gpu_p2p_import(self._h, buf), "pic1dp_gpu_p2p_import")

    # ---- markers ----
    def set_markers(self, isp: int, x, v, p, w):
        n = x.size
        assert v.size == n and p.size == n and w.size == n
        self._ck(self.L.pic1dp_gpu_set_markers(self._h, isp, n, _dp(x), _dp(v), _dp(p), _dp(w)), "set_markers")

    def set_markers_ptr(self, isp: int, n: int, x: int, v: int, p: int, w: int):
        """Raw host addresses (e.g. pinned torch tensors' data_ptr())."""
        self._ck(self.L.pic1dp_gpu_set_markers(self._h, isp, n, _ptr(x), _ptr(v), _ptr(p), _ptr(w)), "set_markers")

    def load_markers(self, isp: int, rand_v, rand_x, nparticle_init: int, v_max: float = 8.0, init_mode=(1,),
                     init_cos=(0.0,), init_sin=(1e-5,)):
        """Device-side particle_load from the two uniform streams (arrays or raw host addresses)."""
        im, ic, isn = _modes(init_mode, init_cos, init_sin)
        if isinstance(rand_v, np.ndarray):
            n, pv, px = rand_v.size, _dp(rand_v), _dp(rand_x)
        else:
            n, pv, px = rand_v[1], _ptr(rand_v[0]), _ptr(rand_x[0])
        self._ck(self.L.pic1dp_gpu_load_markers(self._h, isp, n, int(nparticle_init), pv, px, float(v_max), len(im), im,
                                                ic, isn), "load_markers")

    def load_markers_kiss64(self, isp: int, n: int, seeds, offset_v: int, offset_x: int, nparticle_init: int,
                            v_max: float = 8.0, init_mode=(1,), init_cos=(0.0,), init_sin=(1e-5,)):
        """Device-side particle_load with the device KISS64 stream (multirand_al_int = 1), bit-exact to multirand.
        seeds: multirand_seeds(0:3) after multirand_init; offsets: outputs consumed before pv / px of this rank."""
        im, ic, isn = _modes(init_mode, init_cos, init_sin)
        sd = (C.c_uint64 * 4)(*[int(v) & 0xFFFFFFFFFFFFFFFF for v in seeds])
        self._ck(self.L.pic1dp_gpu_load_markers_kiss64(self._h, isp, int(n), int(nparticle_init), sd, int(offset_v),
                                                       int(offset_x), float(v_max), len(im), im, ic, isn),
                 "load_markers_kiss64")

    def load_markers_superkiss64(self, isp: int, n: int, nlocal: int, seeds, iseed: int, nparticle_init: int,
                                 v_max: float = 8.0, init_mode=(1,), init_cos=(0.0,), init_sin=(1e-5,)) -> int:
        """Device-side particle_load with the device SuperKISS64 stream (multirand_al_int = 3), bit-exact to multirand.
        seeds: multirand_seeds(0:20634) as a uint64 array, advanced IN PLACE past the 2 * nlocal draws; iseed: the
        table position before them.  Returns the table position after them."""
        im, ic, isn = _modes(init_mode, init_cos, init_sin)
        pos = C.c_int32(int(iseed))
        self._ck(self.L.pic1dp_gpu_load_markers_superkiss64(
            self._h, isp, int(n), int(nlocal), int(nparticle_init), _state_ptr(seeds, *_SK), C.byref(pos),
            float(v_max), len(im), im, ic, isn), "load_markers_superkiss64")
        return pos.value

    def load_markers_maxwellian_kiss64(self, isp: int, n: int, nlocal: int, seeds, gauss_filled: int, gauss_buf: float,
                                       nparticle_init: int, init_mode=(1,), init_cos=(0.0,), init_sin=(1e-5,)):
        """Device-side particle_load for input_imarker = 1 with both streams (gaussian_array(pv, nlocal), then
        real_array(px, nlocal)) generated on the device by KISS64.  seeds: multirand_seeds(0:3) as a C-contiguous uint64
        array, advanced IN PLACE past every draw; (gauss_filled, gauss_buf): the Gaussian one-slot buffer before the
        call.  Returns the buffer after it."""
        im, ic, isn = _modes(init_mode, init_cos, init_sin)
        filled, buf = C.c_int32(int(gauss_filled)), C.c_double(float(gauss_buf))
        self._ck(self.L.pic1dp_gpu_load_markers_maxwellian_kiss64(
            self._h, isp, int(n), int(nlocal), int(nparticle_init), _state_ptr(seeds, *_KISS),
            C.byref(filled), C.byref(buf), len(im), im, ic, isn), "load_markers_maxwellian_kiss64")
        return filled.value, buf.value

    def load_markers_maxwellian_superkiss64(self, isp: int, n: int, nlocal: int, seeds, iseed: int, gauss_filled: int,
                                            gauss_buf: float, nparticle_init: int, init_mode=(1,), init_cos=(0.0,),
                                            init_sin=(1e-5,)):
        """The same with SuperKISS64: seeds = multirand_seeds(0:20634) (advanced in place), iseed = the table position.
        Returns (iseed, gauss_filled, gauss_buf) after the call."""
        im, ic, isn = _modes(init_mode, init_cos, init_sin)
        pos, filled, buf = C.c_int32(int(iseed)), C.c_int32(int(gauss_filled)), C.c_double(float(gauss_buf))
        self._ck(self.L.pic1dp_gpu_load_markers_maxwellian_superkiss64(
            self._h, isp, int(n), int(nlocal), int(nparticle_init), _state_ptr(seeds, *_SK), C.byref(pos),
            C.byref(filled), C.byref(buf), len(im), im, ic, isn), "load_markers_maxwellian_superkiss64")
        return pos.value, filled.value, buf.value

    def load_markers_mt19937_64(self, isp: int, n: int, nlocal: int, seeds, iseed: int, nparticle_init: int,
                                v_max: float = 8.0, init_mode=(1,), init_cos=(0.0,), init_sin=(1e-5,)) -> int:
        """Device-side particle_load with the device MT19937-64 stream (multirand_al_int = 2), bit-exact to multirand.
        seeds: multirand_seeds(0:311) as a C-contiguous uint64 array, advanced IN PLACE past the 2 * nlocal draws;
        iseed: the block position before them.  Returns the block position after them."""
        im, ic, isn = _modes(init_mode, init_cos, init_sin)
        pos = C.c_int32(int(iseed))
        self._ck(self.L.pic1dp_gpu_load_markers_mt19937_64(
            self._h, isp, int(n), int(nlocal), int(nparticle_init), _state_ptr(seeds, *_MT), C.byref(pos),
            float(v_max), len(im), im, ic, isn), "load_markers_mt19937_64")
        return pos.value

    def load_markers_maxwellian_mt19937_64(self, isp: int, n: int, nlocal: int, seeds, iseed: int, gauss_filled: int,
                                           gauss_buf: float, nparticle_init: int, init_mode=(1,), init_cos=(0.0,),
                                           init_sin=(1e-5,)):
        """The Maxwellian loader with MT19937-64: seeds = multirand_seeds(0:311) (advanced in place), iseed = the block
        position.  Returns (iseed, gauss_filled, gauss_buf) after the call."""
        im, ic, isn = _modes(init_mode, init_cos, init_sin)
        pos, filled, buf = C.c_int32(int(iseed)), C.c_int32(int(gauss_filled)), C.c_double(float(gauss_buf))
        self._ck(self.L.pic1dp_gpu_load_markers_maxwellian_mt19937_64(
            self._h, isp, int(n), int(nlocal), int(nparticle_init), _state_ptr(seeds, *_MT), C.byref(pos),
            C.byref(filled), C.byref(buf), len(im), im, ic, isn), "load_markers_maxwellian_mt19937_64")
        return pos.value, filled.value, buf.value

    def mt19937_64_uniforms(self, seeds, iseed: int, n: int):
        """(n uniforms of the device MT19937-64 stream, block position after them); seeds advanced in place."""
        out = np.empty(n)
        pos = C.c_int32(int(iseed))
        self._ck(self.L.pic1dp_gpu_mt19937_64_uniforms(self._h, _state_ptr(seeds, *_MT), C.byref(pos), int(n), _dp(out)),
                 "mt19937_64_uniforms")
        return out, pos.value

    def last_gaussian_load(self):
        """(draws the Gaussian call consumed, rounds, SuperKISS64 draws regenerated) of the last Maxwellian load."""
        d, r, g = C.c_int64(), C.c_int64(), C.c_int64()
        self._ck(self.L.pic1dp_gpu_last_gaussian_load(self._h, C.byref(d), C.byref(r), C.byref(g)), "last_gaussian_load")
        return d.value, r.value, g.value

    def superkiss64_uniforms(self, seeds, iseed: int, n: int):
        """(n uniforms of the device SuperKISS64 stream, table position after them); seeds advanced in place."""
        out = np.empty(n)
        pos = C.c_int32(int(iseed))
        self._ck(self.L.pic1dp_gpu_superkiss64_uniforms(self._h, _state_ptr(seeds, *_SK), C.byref(pos), int(n),
                                                        _dp(out)), "superkiss64_uniforms")
        return out, pos.value

    def load_markers_counter(self, isp: int, n: int, seed: int, first_index: int, nparticle_init: int,
                             v_max: float = 8.0, init_mode=(1,), init_cos=(0.0,), init_sin=(1e-5,)):
        """Device-side particle_load with the counter-based generator (synthetic markers, no reference stream)."""
        im, ic, isn = _modes(init_mode, init_cos, init_sin)
        self._ck(self.L.pic1dp_gpu_load_markers_counter(self._h, isp, int(n), int(nparticle_init), int(seed),
                                                        int(first_index), float(v_max), len(im), im, ic, isn),
                 "load_markers_counter")

    def kiss64_uniforms(self, seeds, offset: int, n: int) -> np.ndarray:
        sd = (C.c_uint64 * 4)(*[int(v) & 0xFFFFFFFFFFFFFFFF for v in seeds])
        out = np.empty(n)
        self._ck(self.L.pic1dp_gpu_kiss64_uniforms(self._h, sd, int(offset), int(n), _dp(out)), "kiss64_uniforms")
        return out

    def p2p_trace(self, capacity: int):
        self._ck(self.L.pic1dp_gpu_p2p_trace(self._h, int(capacity)), "p2p_trace")

    def p2p_trace_read(self, capacity: int):
        buf = np.zeros(capacity * 3, dtype=np.uint64)
        ep = C.c_int64()
        self._ck(self.L.pic1dp_gpu_p2p_trace_read(self._h, buf.ctypes.data_as(C.POINTER(C.c_uint64)), C.byref(ep)),
                 "p2p_trace_read")
        return buf.reshape(capacity, 3), ep.value

    def load_markers_maxwellian(self, isp: int, gauss_v, rand_x, nparticle_init: int, init_mode=(1,), init_cos=(0.0,),
                                init_sin=(1e-5,)):
        """Device-side particle_load for input_imarker = 1 (Gaussian v stream, iptcldist = 0)."""
        im, ic, isn = _modes(init_mode, init_cos, init_sin)
        self._ck(self.L.pic1dp_gpu_load_markers_maxwellian(self._h, isp, gauss_v.size, int(nparticle_init), _dp(gauss_v),
                                                           _dp(rand_x), len(im), im, ic, isn),
                 "load_markers_maxwellian")

    def get_markers(self, isp: int, want=("x", "v", "p", "w")):
        n = C.c_int64()
        self._ck(self.L.pic1dp_gpu_get_markers(self._h, isp, None, None, None, None, C.byref(n)), "get_markers")
        out = {k: np.empty(n.value) for k in want}
        self._ck(self.L.pic1dp_gpu_get_markers(self._h, isp, _dp(out.get("x")), _dp(out.get("v")), _dp(out.get("p")),
                                               _dp(out.get("w")), C.byref(n)), "get_markers")
        return out

    def get_markers_ptr(self, isp: int, x: int = 0, v: int = 0, p: int = 0, w: int = 0) -> int:
        n = C.c_int64()
        f = lambda a: _ptr(a) if a else None
        self._ck(self.L.pic1dp_gpu_get_markers(self._h, isp, f(x), f(v), f(p), f(w), C.byref(n)), "get_markers")
        return n.value

    def get_shape_x(self, isp: int):
        """(indexes, values_left, values_right) of the current x -- particle_shape_x_indexes / _values."""
        n = C.c_int64()
        self._ck(self.L.pic1dp_gpu_get_markers(self._h, isp, None, None, None, None, C.byref(n)), "get_markers")
        ix = np.empty(n.value, dtype=np.int32)
        sl, sr = np.empty(n.value), np.empty(n.value)
        self._ck(self.L.pic1dp_gpu_get_shape_x(self._h, isp, ix.ctypes.data_as(C.POINTER(C.c_int32)), _dp(sl), _dp(sr)),
                 "get_shape_x")
        return ix, sl, sr

    # ---- the hot path ----
    def compute_shape_x(self):
        self._ck(self.L.pic1dp_gpu_compute_shape_x(self._h), "compute_shape_x")

    def collect_charge(self):
        self._ck(self.L.pic1dp_gpu_collect_charge(self._h), "collect_charge")

    def solve_field(self):
        self._ck(self.L.pic1dp_gpu_solve_field(self._h), "solve_field")

    def push(self, irk: int):
        self._ck(self.L.pic1dp_gpu_push(self._h, irk), "push")

    def step(self, nsteps: int = 1):
        self._ck(self.L.pic1dp_gpu_step(self._h, nsteps), "step")

    # ---- fields ----
    def set_modes(self, modes):
        """Replace the kept-mode set (input_modes(1:input_nmode), any count, e.g. range(1, nx // 2 + 1) for the
        unfiltered solve): rebuilds the field operators; takes effect from the next solve."""
        ms = [int(m) for m in modes]
        arr = (C.c_int32 * len(ms))(*ms) if ms else None
        self._ck(self.L.pic1dp_gpu_set_modes(self._h, len(ms), arr), "set_modes")
        self.modes = ms

    def get_field(self):
        nx, M = self.params.nx, len(self.modes)
        E, rho, mre, mim = np.empty(nx), np.empty(nx), np.empty(M), np.empty(M)
        self._ck(self.L.pic1dp_gpu_get_field(self._h, _dp(E), _dp(rho), _dp(mre), _dp(mim)), "get_field")
        return dict(electric=E, chargeden=rho, mode_re=mre, mode_im=mim)

    def get_field_ptr(self, E: int = 0, rho: int = 0, mre: int = 0, mim: int = 0):
        f = lambda a: _ptr(a) if a else None
        self._ck(self.L.pic1dp_gpu_get_field(self._h, f(E), f(rho), f(mre), f(mim)), "get_field")

    def set_field(self, electric=None, chargeden=None):
        e = None if electric is None else np.ascontiguousarray(electric, dtype=np.float64)
        r = None if chargeden is None else np.ascontiguousarray(chargeden, dtype=np.float64)
        self._ck(self.L.pic1dp_gpu_set_field(self._h, _dp(e), _dp(r)), "set_field")

    def get_operators(self):
        nx, M = self.params.nx, len(self.modes)
        Fre, Fim, g = np.empty(nx * M), np.empty(nx * M), np.empty(M)
        self._ck(self.L.pic1dp_gpu_get_operators(self._h, _dp(Fre), _dp(Fim), _dp(g)), "get_operators")
        return Fre.reshape(nx, M), Fim.reshape(nx, M), g

    def field_energy(self) -> float:
        e = C.c_double()
        self._ck(self.L.pic1dp_gpu_field_energy(self._h, C.byref(e)), "field_energy")
        return e.value

    # ---- on-device diagnostics of pic1dp_output ----
    def output_field(self) -> np.ndarray:
        """[|E|^2 lx/nx, then per species sum v^2, sum v^2 p, sum v^2 w | perturbed energy] (output_field)."""
        out = np.empty(1 + 3 * self.params.nspecies)
        self._ck(self.L.pic1dp_gpu_output_field(self._h, _dp(out)), "output_field")
        return out

    def output_ptcldist(self, isp: int, nx_opd: int = 64, nv_opd: int = 64, v_max: float = 8.0):
        nc = nx_opd * nv_opd
        outs = [np.empty(nc), np.empty(nc), np.empty(nc), np.empty(nv_opd), np.empty(nv_opd), np.empty(nv_opd)]
        self._ck(self.L.pic1dp_gpu_output_ptcldist(self._h, isp, nx_opd, nv_opd, float(v_max), *[_dp(o) for o in outs]),
                 "output_ptcldist")
        return dict(zip(("markr_xv", "total_xv", "pertb_xv", "markr_v", "total_v", "pertb_v"), outs))

    def output_all(self, nx_opd: int = 64, nv_opd: int = 64, v_max: float = 8.0):
        """(output_field scalars, [output_ptcldist dict per species]) from one pass over the markers."""
        nsp, nc = self.params.nspecies, nx_opd * nv_opd
        sc = np.empty(1 + 3 * nsp)
        per = 3 * nc + 3 * nv_opd
        buf = np.empty(per * nsp)
        self._ck(self.L.pic1dp_gpu_output_all(self._h, nx_opd, nv_opd, float(v_max), _dp(sc), _dp(buf)), "output_all")
        names = ("markr_xv", "total_xv", "pertb_xv", "markr_v", "total_v", "pertb_v")
        dists = []
        for s in range(nsp):
            o = buf[per * s: per * (s + 1)]
            parts = [o[0:nc], o[nc:2 * nc], o[2 * nc:3 * nc], o[3 * nc:3 * nc + nv_opd],
                     o[3 * nc + nv_opd:3 * nc + 2 * nv_opd], o[3 * nc + 2 * nv_opd:]]
            dists.append({k: a.copy() for k, a in zip(names, parts)})
        return sc, dists

    # ---- marker optimisation (src/pic1dp_particle.F90:356-746) ----
    def compute_dist_pertb_abs_v(self, nv: int = 128, v_max: float = 8.0) -> np.ndarray:
        """particle_dist_pertb_abs_v as [nspecies, nv], reduced on the device and over ranks."""
        out = np.empty((self.params.nspecies, nv))
        self._ck(self.L.pic1dp_gpu_compute_dist_pertb_abs_v(self._h, nv, float(v_max), _dp(out)),
                 "compute_dist_pertb_abs_v")
        return out

    def _np_out(self):
        return (C.c_int64 * self.params.nspecies)()

    def particle_merge(self, thsh: float):
        n = self._np_out()
        self._ck(self.L.pic1dp_gpu_particle_merge(self._h, float(thsh), n), "particle_merge")
        return list(n)

    def particle_remove(self, thsh: float, typeremove: int, remove_frac: float, real64):
        """real64: callable returning the next multirand_real64() of this rank's generator."""
        n = self._np_out()
        # ctypes swallows an exception raised inside a call-back (the C loop would go on with garbage): keep it,
        # feed harmless values for the rest of the call and re-raise once the C call has returned
        err = []

        def dice(_ctx):
            if err:
                return 1.0
            try:
                return float(real64())
            except BaseException as e:  # noqa: BLE001
                err.append(e)
                return 1.0
        cb = _capi.REAL64_FN(dice)
        rc = self.L.pic1dp_gpu_particle_remove(self._h, float(thsh), typeremove, float(remove_frac), cb, None, n)
        if err:
            raise RuntimeError("particle_remove: the real64 call-back raised; the markers on the device are invalid") from err[0]
        self._ck(rc, "particle_remove")
        return list(n)

    def particle_split(self, thsh: float, ngroup: int, dv_sig_frac: float, gaussian_array):
        """gaussian_array: callable n -> array of n draws, like multirand_gaussian_array."""
        n = self._np_out()

        err = []

        def fill(_ctx, a, k):
            try:
                if err:
                    raise err[0]
                g = gaussian_array(k)
                for i in range(k):
                    a[i] = g[i]
            except BaseException as e:  # noqa: BLE001 -- see particle_remove
                if not err:
                    err.append(e)
                for i in range(k):
                    a[i] = 0.0
        cb = _capi.GAUSSIAN_ARRAY_FN(fill)
        rc = self.L.pic1dp_gpu_particle_split(self._h, float(thsh), ngroup, float(dv_sig_frac), cb, None, n)
        if err:
            raise RuntimeError("particle_split: the gaussian_array call-back raised; the markers on the device are invalid") from err[0]
        self._ck(rc, "particle_split")
        return list(n)

    # ---- instrumentation ----
    def sync(self):
        self._ck(self.L.pic1dp_gpu_sync(self._h), "sync")

    def timer_start(self):
        self._ck(self.L.pic1dp_gpu_timer_start(self._h), "timer_start")

    def timer_stop(self) -> float:
        ms = C.c_float()
        self._ck(self.L.pic1dp_gpu_timer_stop(self._h, C.byref(ms)), "timer_stop")
        return ms.value

    def counters(self) -> Counters:
        c = Counters()
        self._ck(self.L.pic1dp_gpu_get_counters(self._h, C.byref(c)), "get_counters")
        return c

    def launch_timing_start(self):
        self._ck(self.L.pic1dp_gpu_launch_timing_start(self._h), "launch_timing_start")

    def launch_timing_stop(self):
        """[(ms_sum, launches) for irk = 1, 2] of the fused particle kernels since launch_timing_start."""
        ms = (C.c_double * 2)()
        n = (C.c_int64 * 2)()
        self._ck(self.L.pic1dp_gpu_launch_timing_stop(self._h, ms, n), "launch_timing_stop")
        return [(ms[0], n[0]), (ms[1], n[1])]

    def profile_step(self):
        ms = (C.c_float * 6)()
        self._ck(self.L.pic1dp_gpu_profile_step(self._h, ms), "profile_step")
        return list(ms)


def petsc_decide(n: int, npe: int, rank: int):
    """Contiguous block split PETSc makes for VecSetSizes(PETSC_DECIDE, n) (requested at
    src/pic1dp_particle.F90:91): rank r owns n/npe + (r < n mod npe) entries.  Returns [low, high)."""
    base, rem = divmod(n, npe)
    low = base * rank + min(rank, rem)
    return low, low + base + (1 if rank < rem else 0)


class Pic1dpModules:
    """The three reference modules as one object: same procedure names and implicit state.

    Usage replays src/pic1dp.F90:57-90::

        m = Pic1dpModules(params); m.particle_init(); m.field_init()
        m.particle_set(0, x, v, p, w)             # host-generated markers; or m.particle_load(0, rand_v, rand_x, n)
        if m.input.iptclshape < 4: m.particle_compute_shape_x()
        m.interaction_collect_charge(); m.field_solve_electric()
        for m.global_irk in (1, 2):
            m.interaction_push_particle()
            if m.input.iptclshape < 4: m.particle_compute_shape_x()
            m.interaction_collect_charge(); m.field_solve_electric()
    """

    def __init__(self, params: Params):
        self.input = params          # input_* parameters (src/pic1dp_input.F90)
        self.global_irk = 1          # src/pic1dp_global.F90:64
        self.global_ierr = 0         # src/pic1dp_global.F90:59
        self.global_mype = params.rank
        self.global_npe = params.nranks
        self.gpu: Optional[Pic1dGpu] = None
        self.particle_np = [0] * params.nspecies  # src/pic1dp_particle.F90:54

    def _call(self, fn, *a):
        try:
            r = fn(*a)
            self.global_ierr = 0
            return r
        except Pic1dpError as e:  # CHKERRQ(global_ierr)
            self.global_ierr = e.code
            raise

    # pic1dp_particle
    def particle_init(self):
        if self.gpu is None:
            self.gpu = self._call(Pic1dGpu, self.input)

    def particle_set(self, isp: int, x, v, p, w):
        self.particle_np[isp] = x.size
        self._call(self.gpu.set_markers, isp, x, v, p, w)

    def particle_load(self, isp: int, rand_v, rand_x, nparticle_init: int, v_max: float = 8.0, init_mode=(1,),
                      init_cos=(0.0,), init_sin=(1e-5,)):
        """particle_load (src/pic1dp_particle.F90:145-269) for uniform-v markers: the host draws the two uniform streams
        in the reference's order (multirand_real_array(pv) :180, then (px) :222); the loader arithmetic runs on the
        device.  particle_np = number of streamed values (the unloaded tail, :240-248, is simply not passed)."""
        self.particle_np[isp] = rand_v.size
        self._call(self.gpu.load_markers, isp, rand_v, rand_x, nparticle_init, v_max, init_mode, init_cos, init_sin)

    def particle_get(self, isp: int):
        return self._call(self.gpu.get_markers, isp)

    def particle_compute_shape_x(self):
        self._call(self.gpu.compute_shape_x)

    # marker optimisation: the schedule of particle_optimize (src/pic1dp_particle.F90:752-813) with run-time copies of
    # input_nmerge/_tmerge/_thshmerge, ... (src/pic1dp_input.F90:146-206); `rng` supplies multirand draws
    def particle_optimize_setup(self, tmerge=(), thshmerge=(), tremove=(), thshremove=(), typeremove=2, remove_frac=0.9,
                                tsplit=(), thshsplit=(), split_ngroup=5, split_dv_sig_frac=0.1, nv=128, v_max=8.0,
                                rng=None):
        self.input_tmerge, self.input_thshmerge = list(tmerge), list(thshmerge)
        self.input_tremove, self.input_thshremove = list(tremove), list(thshremove)
        self.input_tsplit, self.input_thshsplit = list(tsplit), list(thshsplit)
        self.input_typeremove, self.input_remove_frac = typeremove, remove_frac
        self.input_split_ngroup, self.input_split_dv_sig_frac = split_ngroup, split_dv_sig_frac
        self.input_nv, self.input_v_max = nv, v_max
        self.particle_imerge = 1 if self.input_tmerge else 0    # :73-87
        self.particle_iremove = 1 if self.input_tremove else 0
        self.particle_isplit = 1 if self.input_tsplit else 0
        self.multirand = rng

    def particle_compute_dist_pertb_abs_v(self):
        self.particle_dist_pertb_abs_v = self._call(self.gpu.compute_dist_pertb_abs_v, self.input_nv, self.input_v_max)

    def particle_merge(self, thsh):
        self.particle_np = self._call(self.gpu.particle_merge, thsh)

    def particle_remove(self, thsh):
        self.particle_np = self._call(self.gpu.particle_remove, thsh, self.input_typeremove, self.input_remove_frac,
                                      self.multirand.real64)

    def particle_split(self, thsh):
        self.particle_np = self._call(self.gpu.particle_split, thsh, self.input_split_ngroup,
                                      self.input_split_dv_sig_frac, self.multirand.gaussian_array)

    def particle_optimize(self, global_time: float) -> bool:
        """flag_optimized of particle_optimize; global_time is the time at the START of the current step."""
        flag = False
        if self.input.deltaf == 0:          # :762
            return flag
        dt = self.input.dt
        if 0 < self.particle_imerge <= len(self.input_tmerge):
            if global_time + dt >= self.input_tmerge[self.particle_imerge - 1] and self.global_irk == 2:
                self.particle_compute_dist_pertb_abs_v()
                self.particle_merge(self.input_thshmerge[self.particle_imerge - 1])
                self.particle_imerge += 1
                flag = True
        if 0 < self.particle_iremove <= len(self.input_tremove):
            if global_time + dt >= self.input_tremove[self.particle_iremove - 1] and self.global_irk == 2:
                self.particle_compute_dist_pertb_abs_v()
                self.particle_remove(self.input_thshremove[self.particle_iremove - 1])
                self.particle_iremove += 1
                flag = True
        if 0 < self.particle_isplit <= len(self.input_tsplit):
            if global_time + dt >= self.input_tsplit[self.particle_isplit - 1] and self.global_irk == 2:
                self.particle_compute_dist_pertb_abs_v()
                self.particle_split(self.input_thshsplit[self.particle_isplit - 1])
                self.particle_isplit += 1
                flag = True
        return flag

    def particle_final(self):
        if self.gpu is not None:
            self.gpu.close()
            self.gpu = None

    # pic1dp_field
    def field_init(self):
        self.particle_init()  # one handle owns both modules' state

    def field_solve_electric(self):
        self._call(self.gpu.solve_field)

    def field_test(self):
        """field_test (src/pic1dp_field.F90:276-309): chargeden = cos(2 pi ix / nx), solve, return field_electric
        (the reference prints it with VecView)."""
        nx = self.input.nx
        ix = np.arange(nx, dtype=np.float64)
        values = np.cos(2.0 * 3.14159265358979323846264338327950288419716939937510582 * ix / float(nx))  # :290
        self._call(self.gpu.set_field, None, values)
        self.field_solve_electric()
        return self.field_electric

    def field_final(self):
        self.particle_final()

    @property
    def field_electric(self):
        return self._call(self.gpu.get_field)["electric"]

    @property
    def field_chargeden(self):
        return self._call(self.gpu.get_field)["chargeden"]

    @property
    def field_mode_re(self):
        return self._call(self.gpu.get_field)["mode_re"]

    @property
    def field_mode_im(self):
        return self._call(self.gpu.get_field)["mode_im"]

    # pic1dp_interaction
    def interaction_collect_charge(self):
        self._call(self.gpu.collect_charge)

    def interaction_push_particle(self):
        self._call(self.gpu.push, self.global_irk)


# ---- host-side generator helpers (no GPU): the same code the device runs ----
def host_kiss64_jump(seeds, n: int):
    """multirand_seeds(0:3) advanced by n outputs (O(log n) table steps)."""
    sd = (C.c_uint64 * 4)(*[int(v) & 0xFFFFFFFFFFFFFFFF for v in seeds])
    rc = _capi.load().pic1dp_host_kiss64_jump(sd, int(n))
    if rc:
        raise Pic1dpError(rc, "pic1dp_host_kiss64_jump", "bad argument")
    return [int(v) for v in sd]


def host_kiss64_fill(seeds, n: int):
    """(n uniforms of multirand_real_array, state afterwards)."""
    sd = (C.c_uint64 * 4)(*[int(v) & 0xFFFFFFFFFFFFFFFF for v in seeds])
    out = np.empty(n)
    rc = _capi.load().pic1dp_host_kiss64_fill(sd, int(n), _dp(out))
    if rc:
        raise Pic1dpError(rc, "pic1dp_host_kiss64_fill", "bad argument")
    return out, [int(v) for v in sd]


def host_counter_uniforms(seed: int, stream: int, first_index: int, n: int):
    u_v, u_x = np.empty(n), np.empty(n)
    _capi.load().pic1dp_host_counter_uniforms(int(seed), int(stream), int(first_index), int(n), _dp(u_v), _dp(u_x))
    return u_v, u_x


def host_superkiss64_fill(seeds, iseed: int, n: int):
    """(n uniforms of multirand_real_array with SuperKISS64, table position after them); seeds (uint64 array of
    20635 words) advanced in place."""
    out = np.empty(n)
    pos = C.c_int32(int(iseed))
    rc = _capi.load().pic1dp_host_superkiss64_fill(_state_ptr(seeds, *_SK), C.byref(pos), int(n), _dp(out))
    if rc:
        raise Pic1dpError(rc, "pic1dp_host_superkiss64_fill", "bad argument")
    return out, pos.value


def host_superkiss64_refill(seeds, nchunks: int):
    """One table refill of seeds (in place) by the device's chunked carry-map scan, run on the host."""
    rc = _capi.load().pic1dp_host_superkiss64_refill(_state_ptr(seeds, *_SK), int(nchunks))
    if rc:
        raise Pic1dpError(rc, "pic1dp_host_superkiss64_refill", "bad argument")



def host_mt19937_64_jump(seeds, iseed: int, n: int) -> int:
    """multirand_seeds(0:311) (uint64 array, in place) and the block position advanced by n draws with the device's
    window-XOR jump run on the host.  Returns the block position after them."""
    pos = C.c_int32(int(iseed))
    rc = _capi.load().pic1dp_host_mt19937_64_jump(_state_ptr(seeds, *_MT), C.byref(pos), int(n))
    if rc:
        raise Pic1dpError(rc, "pic1dp_host_mt19937_64_jump", "bad argument")
    return pos.value
