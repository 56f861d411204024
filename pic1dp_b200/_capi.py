"""ctypes binding of the C ABI declared in include/pic1dp_gpu.h (libpic1dp_b200.so).

This is the only way Python reaches the product: no torch types cross the boundary, and there is no CPU
fallback -- if the CUDA library is missing or no GPU is present the calls fail loudly.
"""
from __future__ import annotations

import ctypes as C
import os

MAX_SPECIES = 4
MAX_MODES = 64                     # kept modes Params.modes holds; pic1dp_gpu_set_modes takes any count
MAX_FIELD_TABLE_BYTES = 1 << 32    # PIC1DP_MAX_FIELD_TABLE_BYTES: 32 * nx * nmode bytes of field tables at most
UNIQUE_ID_BYTES = 128
IPC_HANDLE_BYTES = 64
SUPERKISS64_NSEED = 20635
MT19937_64_NSEED = 312
GAUSS_ROUND_DRAWS = 4194304   # PIC1DP_GAUSS_ROUND_DRAWS: draws per round of the device Gaussian stream

OK, EINVAL, ECUDA, ENCCL, ENOMEM, ESTATE, ECAPACITY, ENODEVICE, EUNSUPPORTED = range(9)
DEPOSIT_AUTO, DEPOSIT_SMEM_ATOMIC, DEPOSIT_GLOBAL_RED, DEPOSIT_WARP_PRIVATE, DEPOSIT_FIXED = range(5)
ARITH_STRICT, ARITH_TOLERANCE = range(2)
FIELD_TREE, FIELD_SEQUENTIAL = range(2)
LOAD_AUTO, LOAD_DIRECT, LOAD_TMA, LOAD_CPASYNC = range(4)

# PIC1DP_B200_LIB overrides the library path (kernel A/B experiments under scratch/); the product default is in-tree
_LIB_PATH = os.environ.get("PIC1DP_B200_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)),
                                                               "libpic1dp_b200.so")


class Params(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32),
        ("struct_bytes", C.c_int32),
        ("nx", C.c_int32),
        ("nmode", C.c_int32),
        ("modes", C.c_int32 * MAX_MODES),
        ("lx", C.c_double),
        ("dt", C.c_double),
        ("nspecies", C.c_int32),
        ("charge", C.c_double * MAX_SPECIES),
        ("mass", C.c_double * MAX_SPECIES),
        ("temperature", C.c_double * MAX_SPECIES),
        ("temperature2", C.c_double * MAX_SPECIES),
        ("density", C.c_double * MAX_SPECIES),
        ("v0", C.c_double * MAX_SPECIES),
        ("iptcldist", C.c_int32),
        ("deltaf", C.c_int32),
        ("linear", C.c_int32),
        ("iptclshape", C.c_int32),
        ("capacity", C.c_int64),
        ("device", C.c_int32),
        ("rank", C.c_int32),
        ("nranks", C.c_int32),
        ("deposit_mode", C.c_int32),
        ("field_mode", C.c_int32),
        ("fuse", C.c_int32),
        ("load_path", C.c_int32),
        ("arith_mode", C.c_int32),
        ("no_step_graph", C.c_int32),
        ("reserved", C.c_int32 * 5),
    ]


class Counters(C.Structure):
    _fields_ = [
        ("kernel_launches", C.c_int64),
        ("nccl_calls", C.c_int64),
        ("p2p_allreduces", C.c_int64),
        ("p2p_timeouts", C.c_int64),
        ("oob_markers", C.c_int64),
        ("h2d_bytes", C.c_int64),
        ("d2h_bytes", C.c_int64),
        ("deposit_mode", C.c_int32),
        ("grid_ctas", C.c_int32),
        ("cta_threads", C.c_int32),
        ("smem_bytes", C.c_int32),
        ("graph_replays", C.c_int64),
    ]


# every symbol include/pic1dp_gpu.h declares; tests check the .so exports each of them
EXPORTS = [
    "pic1dp_gpu_params_default", "pic1dp_gpu_abi_version", "pic1dp_gpu_strerror", "pic1dp_gpu_last_error",
    "pic1dp_gpu_create", "pic1dp_gpu_destroy", "pic1dp_gpu_comm_unique_id", "pic1dp_gpu_comm_init",
    "pic1dp_gpu_p2p_export", "pic1dp_gpu_p2p_import",
    "pic1dp_gpu_set_markers", "pic1dp_gpu_load_markers", "pic1dp_gpu_load_markers_maxwellian", "pic1dp_gpu_get_markers", "pic1dp_gpu_compute_shape_x", "pic1dp_gpu_get_shape_x",
    "pic1dp_gpu_collect_charge", "pic1dp_gpu_solve_field", "pic1dp_gpu_push", "pic1dp_gpu_step",
    "pic1dp_gpu_get_field", "pic1dp_gpu_set_field", "pic1dp_gpu_get_operators", "pic1dp_gpu_field_energy",
    "pic1dp_gpu_output_field", "pic1dp_gpu_output_ptcldist",
    "pic1dp_gpu_sync", "pic1dp_gpu_timer_start", "pic1dp_gpu_timer_stop", "pic1dp_gpu_get_counters",
    "pic1dp_gpu_profile_step",
    "pic1dp_gpu_compute_dist_pertb_abs_v", "pic1dp_gpu_particle_merge", "pic1dp_gpu_particle_remove",
    "pic1dp_gpu_particle_split",
    "pic1dp_host_particle_merge", "pic1dp_host_particle_remove", "pic1dp_host_particle_split",
    "pic1dp_gpu_launch_timing_start", "pic1dp_gpu_launch_timing_stop",
    "pic1dp_gpu_load_markers_kiss64", "pic1dp_gpu_load_markers_counter", "pic1dp_gpu_kiss64_uniforms",
    "pic1dp_host_kiss64_jump", "pic1dp_host_kiss64_fill", "pic1dp_host_counter_uniforms",
    "pic1dp_gpu_load_markers_superkiss64", "pic1dp_gpu_superkiss64_uniforms", "pic1dp_host_superkiss64_fill",
    "pic1dp_host_superkiss64_refill", "pic1dp_gpu_load_markers_maxwellian_kiss64",
    "pic1dp_gpu_load_markers_maxwellian_superkiss64", "pic1dp_gpu_last_gaussian_load",
    "pic1dp_gpu_load_markers_mt19937_64", "pic1dp_gpu_load_markers_maxwellian_mt19937_64",
    "pic1dp_gpu_mt19937_64_uniforms", "pic1dp_host_mt19937_64_jump",
    "pic1dp_gpu_p2p_trace", "pic1dp_gpu_p2p_trace_read", "pic1dp_gpu_output_all", "pic1dp_gpu_set_modes",
]

# RNG call-backs of particle_remove / particle_split (pic1dp_real64_fn, pic1dp_gaussian_array_fn)
REAL64_FN = C.CFUNCTYPE(C.c_double, C.c_void_p)
GAUSSIAN_ARRAY_FN = C.CFUNCTYPE(None, C.c_void_p, C.POINTER(C.c_double), C.c_int32)

_lib = None


def lib_path() -> str:
    return _LIB_PATH


def load() -> C.CDLL:
    """Load libpic1dp_b200.so.  Raises if it has not been built (python -m pic1dp_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise RuntimeError(
            f"{_LIB_PATH} is missing: the CUDA extension has not been built "
            "(run `python -m pic1dp_b200.build` or __graft_entry__.build()); there is no CPU fallback")
    L = C.CDLL(_LIB_PATH)
    vp, dp, i32, i64 = C.c_void_p, C.POINTER(C.c_double), C.c_int32, C.c_int64
    u8p = C.POINTER(C.c_uint8)
    L.pic1dp_gpu_params_default.argtypes = [C.POINTER(Params)]
    L.pic1dp_gpu_params_default.restype = None
    L.pic1dp_gpu_abi_version.restype = C.c_int
    L.pic1dp_gpu_strerror.argtypes = [C.c_int]
    L.pic1dp_gpu_strerror.restype = C.c_char_p
    L.pic1dp_gpu_last_error.argtypes = [vp]
    L.pic1dp_gpu_last_error.restype = C.c_char_p
    L.pic1dp_gpu_create.argtypes = [C.POINTER(Params), C.POINTER(vp)]
    L.pic1dp_gpu_destroy.argtypes = [vp]
    L.pic1dp_gpu_comm_unique_id.argtypes = [u8p]
    L.pic1dp_gpu_comm_init.argtypes = [vp, u8p]
    L.pic1dp_gpu_p2p_export.argtypes = [vp, u8p]
    L.pic1dp_gpu_p2p_import.argtypes = [vp, u8p]
    L.pic1dp_gpu_set_markers.argtypes = [vp, i32, i64, dp, dp, dp, dp]
    L.pic1dp_gpu_load_markers.argtypes = [vp, i32, i64, i64, dp, dp, C.c_double, i32, C.POINTER(i32), dp, dp]
    L.pic1dp_gpu_load_markers_maxwellian.argtypes = [vp, i32, i64, i64, dp, dp, i32, C.POINTER(i32), dp, dp]
    L.pic1dp_gpu_get_markers.argtypes = [vp, i32, dp, dp, dp, dp, C.POINTER(i64)]
    L.pic1dp_gpu_compute_shape_x.argtypes = [vp]
    L.pic1dp_gpu_get_shape_x.argtypes = [vp, i32, C.POINTER(i32), dp, dp]
    L.pic1dp_gpu_collect_charge.argtypes = [vp]
    L.pic1dp_gpu_solve_field.argtypes = [vp]
    L.pic1dp_gpu_push.argtypes = [vp, i32]
    L.pic1dp_gpu_step.argtypes = [vp, i32]
    L.pic1dp_gpu_get_field.argtypes = [vp, dp, dp, dp, dp]
    L.pic1dp_gpu_set_field.argtypes = [vp, dp, dp]
    L.pic1dp_gpu_get_operators.argtypes = [vp, dp, dp, dp]
    L.pic1dp_gpu_set_modes.argtypes = [vp, i32, C.POINTER(i32)]
    L.pic1dp_gpu_field_energy.argtypes = [vp, dp]
    L.pic1dp_gpu_output_field.argtypes = [vp, dp]
    L.pic1dp_gpu_output_ptcldist.argtypes = [vp, i32, i32, i32, C.c_double, dp, dp, dp, dp, dp, dp]
    L.pic1dp_gpu_sync.argtypes = [vp]
    L.pic1dp_gpu_timer_start.argtypes = [vp]
    L.pic1dp_gpu_timer_stop.argtypes = [vp, C.POINTER(C.c_float)]
    L.pic1dp_gpu_get_counters.argtypes = [vp, C.POINTER(Counters)]
    L.pic1dp_gpu_profile_step.argtypes = [vp, C.POINTER(C.c_float)]
    i64p, dbl = C.POINTER(i64), C.c_double
    L.pic1dp_gpu_launch_timing_start.argtypes = [vp]
    L.pic1dp_gpu_launch_timing_stop.argtypes = [vp, dp, i64p]
    L.pic1dp_gpu_compute_dist_pertb_abs_v.argtypes = [vp, i32, dbl, dp]
    L.pic1dp_gpu_particle_merge.argtypes = [vp, dbl, i64p]
    L.pic1dp_gpu_particle_remove.argtypes = [vp, dbl, i32, dbl, REAL64_FN, vp, i64p]
    L.pic1dp_gpu_particle_split.argtypes = [vp, dbl, i32, dbl, GAUSSIAN_ARRAY_FN, vp, i64p]
    L.pic1dp_host_particle_merge.argtypes = [i64, dp, dp, dp, dp, dp, i32, dbl, dbl, i32, dbl]
    L.pic1dp_host_particle_merge.restype = i64
    L.pic1dp_host_particle_remove.argtypes = [i64, dp, dp, dp, dp, dp, i32, dbl, dbl, i32, dbl, REAL64_FN, vp]
    L.pic1dp_host_particle_remove.restype = i64
    L.pic1dp_host_particle_split.argtypes = [i64, i64, dp, dp, dp, dp, dp, i32, dbl, dbl, i32, dbl, i32,
                                             GAUSSIAN_ARRAY_FN, vp]
    L.pic1dp_host_particle_split.restype = i64
    u64p = C.POINTER(C.c_uint64)
    L.pic1dp_gpu_load_markers_kiss64.argtypes = [vp, i32, i64, i64, u64p, i64, i64, dbl, i32, C.POINTER(i32), dp, dp]
    L.pic1dp_gpu_load_markers_counter.argtypes = [vp, i32, i64, i64, C.c_uint64, i64, dbl, i32, C.POINTER(i32), dp, dp]
    L.pic1dp_gpu_kiss64_uniforms.argtypes = [vp, u64p, i64, i64, dp]
    L.pic1dp_host_kiss64_jump.argtypes = [u64p, i64]
    L.pic1dp_host_kiss64_fill.argtypes = [u64p, i64, dp]
    L.pic1dp_host_counter_uniforms.argtypes = [C.c_uint64, i32, i64, i64, dp, dp]
    L.pic1dp_host_counter_uniforms.restype = None
    i32p = C.POINTER(i32)
    L.pic1dp_gpu_load_markers_superkiss64.argtypes = [vp, i32, i64, i64, i64, u64p, i32p, dbl, i32, C.POINTER(i32), dp, dp]
    L.pic1dp_gpu_superkiss64_uniforms.argtypes = [vp, u64p, i32p, i64, dp]
    L.pic1dp_host_superkiss64_fill.argtypes = [u64p, i32p, i64, dp]
    L.pic1dp_host_superkiss64_refill.argtypes = [u64p, i32]
    L.pic1dp_gpu_load_markers_maxwellian_kiss64.argtypes = [vp, i32, i64, i64, i64, u64p, i32p, dp, i32, i32p, dp, dp]
    L.pic1dp_gpu_load_markers_maxwellian_superkiss64.argtypes = [vp, i32, i64, i64, i64, u64p, i32p, i32p, dp, i32, i32p,
                                                                 dp, dp]
    L.pic1dp_gpu_last_gaussian_load.argtypes = [vp, i64p, i64p, i64p]
    L.pic1dp_gpu_load_markers_mt19937_64.argtypes = [vp, i32, i64, i64, i64, u64p, i32p, dbl, i32, i32p, dp, dp]
    L.pic1dp_gpu_load_markers_maxwellian_mt19937_64.argtypes = [vp, i32, i64, i64, i64, u64p, i32p, i32p, dp, i32, i32p,
                                                                dp, dp]
    L.pic1dp_gpu_mt19937_64_uniforms.argtypes = [vp, u64p, i32p, i64, dp]
    L.pic1dp_host_mt19937_64_jump.argtypes = [u64p, i32p, i64]
    L.pic1dp_gpu_output_all.argtypes = [vp, i32, i32, dbl, dp, dp]
    L.pic1dp_gpu_p2p_trace.argtypes = [vp, i32]
    L.pic1dp_gpu_p2p_trace_read.argtypes = [vp, u64p, i64p]
    for name in EXPORTS:
        fn = getattr(L, name)
        if fn.restype is C.c_int and name not in ("pic1dp_gpu_abi_version",):
            fn.restype = C.c_int
    _lib = L
    return L
