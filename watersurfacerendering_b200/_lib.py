"""ctypes binding of the C ABI in include/wsocean.h (libwsocean.so, hand-written sm_100a CUDA).

The library is the only compute path: if it is missing or cannot be loaded this module raises —
there is no CPU or PyTorch fallback.
"""
from __future__ import annotations

import ctypes as C
import os

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
# WSO_LIB_PATH: tuning sweeps point this at a variant build of the same library (tools/tune_build.sh)
LIB_PATH = os.environ.get("WSO_LIB_PATH") or os.path.join(PKG_DIR, "libwsocean.so")

WSO_OK = 0
WSO_ERR_INVALID_ARG = -1
WSO_ERR_BAD_TILE_SIZE = -2
WSO_ERR_NOT_PREPARED = -3
WSO_ERR_CUDA = -4
WSO_ERR_OUT_OF_MEMORY = -5
WSO_ERR_H0_NOT_CONJUGATE = -6

WSO_MAP_DISPLACEMENT = 0
WSO_MAP_NORMAL = 1

# map texel formats (wso_set_map_format)
WSO_MAP_RGBA32F = 0
WSO_MAP_RGBA16F = 1

# struct wso_surface_sample (include/wsocean.h): one 32-byte record per surface query
SURFACE_SAMPLE_DTYPE = [("height", "<f4"), ("normal_x", "<f4"), ("normal_y", "<f4"), ("normal_z", "<f4"),
                        ("offset_x", "<f4"), ("offset_z", "<f4"), ("residual", "<f4"), ("w", "<f4")]

# ray casts (wso_raycast_surface): status of a wso_ray_hit
WSO_RAY_MISS = 0
WSO_RAY_HIT = 1
WSO_RAY_ORIGIN_BELOW = 2
WSO_RAY_UNRESOLVED = 3
WSO_RAY_INVALID = 4

# struct wso_ray_hit (include/wsocean.h): one 48-byte record per ray, the hit's wso_surface_sample flattened into it
RAY_HIT_DTYPE = [("distance", "<f4"), ("x", "<f4"), ("z", "<f4"), ("status", "<u4")] + SURFACE_SAMPLE_DTYPE

STATUS_NAMES = {
    0: "WSO_OK", -1: "WSO_ERR_INVALID_ARG", -2: "WSO_ERR_BAD_TILE_SIZE", -3: "WSO_ERR_NOT_PREPARED",
    -4: "WSO_ERR_CUDA", -5: "WSO_ERR_OUT_OF_MEMORY", -6: "WSO_ERR_H0_NOT_CONJUGATE",
}


class WsoParams(C.Structure):
    """struct wso_params (include/wsocean.h)."""
    _fields_ = [
        ("tile_size", C.c_uint32),
        ("tile_length", C.c_float),
        ("wind_dir_x", C.c_float),
        ("wind_dir_y", C.c_float),
        ("wind_speed", C.c_float),
        ("anim_period", C.c_float),
        ("phillips_const", C.c_float),
        ("damping", C.c_float),
        ("lambda_", C.c_float),
    ]


class WsoRayParams(C.Structure):
    """struct wso_ray_params (include/wsocean.h)."""
    _fields_ = [
        ("step", C.c_float),
        ("max_steps", C.c_uint32),
        ("refine", C.c_uint32),
        ("iterations", C.c_uint32),
    ]


# every symbol include/wsocean.h declares: name -> (restype, argtypes)
_vp, _u32, _f32, _int = C.c_void_p, C.c_uint32, C.c_float, C.c_int
_pp = C.POINTER(WsoParams)
SYMBOLS = {
    "wso_default_params": (_int, [_pp]),
    "wso_create": (_int, [_pp, _int, _u32, _u32, C.POINTER(_vp)]),
    "wso_destroy": (_int, [_vp]),
    "wso_set_params": (_int, [_vp, _u32, _pp]),
    "wso_get_params": (_int, [_vp, _u32, _pp]),
    "wso_set_lambda": (_int, [_vp, _u32, _f32]),
    "wso_set_compute_jacobian": (_int, [_vp, _int]),
    "wso_get_compute_jacobian": (_int, [_vp, _vp]),
    "wso_prepare": (_int, [_vp, _u32, _int, C.c_uint]),
    "wso_prepare_gauss": (_int, [_vp, _u32, _vp]),
    "wso_prepare_gauss_device": (_int, [_vp, _u32, _vp]),
    "wso_prepare_counter": (_int, [_vp, _u32, C.c_uint64]),
    "wso_import_h0": (_int, [_vp, _u32, _vp]),
    "wso_export_h0": (_int, [_vp, _u32, _vp]),
    "wso_import_h0_compact": (_int, [_vp, _u32, _vp]),
    "wso_export_h0_compact": (_int, [_vp, _u32, _vp]),
    "wso_compute_async": (_int, [_vp, _f32, C.POINTER(_vp)]),
    "wso_wait_event": (_int, [_vp, _vp]),
    "wso_compute": (_int, [_vp, _f32, C.POINTER(_f32)]),
    "wso_compute_batch": (_int, [_vp, _u32, _vp, _vp, _u32]),
    "wso_compute_to_host": (_int, [_vp, _u32, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "wso_sync": (_int, [_vp]),
    "wso_read_heights": (_int, [_vp, _u32, _u32, _vp, _vp, _vp]),
    "wso_map_host": (_int, [_vp, _int, C.POINTER(_vp), C.POINTER(C.c_size_t)]),
    "wso_map_device": (_int, [_vp, _int, _u32, C.POINTER(_vp), C.POINTER(C.c_size_t)]),
    "wso_copy_map": (_int, [_vp, _int, _u32, _vp]),
    # map format (RGBA32F / RGBA16F) and the byte-typed map accessors that serve both
    "wso_set_map_format": (_int, [_vp, _int]),
    "wso_get_map_format": (_int, [_vp, C.POINTER(_int)]),
    "wso_map_host_bytes": (_int, [_vp, _int, C.POINTER(_vp), C.POINTER(C.c_size_t)]),
    "wso_copy_map_bytes": (_int, [_vp, _int, _u32, _vp, C.c_size_t]),
    "wso_compute_to_host_bytes": (_int, [_vp, _u32, _vp, _vp, _vp, _vp, C.c_size_t, _vp, _vp, _vp]),
    # surface queries (height / normal / undisplaced origin at world points, 1..4 cascades)
    "wso_query_surface": (_int, [_vp, _u32, _vp, _u32, _u32, _vp, _vp]),
    "wso_query_surface_host": (_int, [_vp, _u32, _vp, _u32, _u32, _vp, _vp]),
    # ray casts (first hit of a segment with the displaced surface, 1..4 cascades)
    "wso_raycast_surface": (_int, [_vp, _u32, _vp, C.POINTER(WsoRayParams), _u32, _vp, _vp]),
    "wso_raycast_surface_host": (_int, [_vp, _u32, _vp, C.POINTER(WsoRayParams), _u32, _vp, _vp]),
    # external-memory interop (Vulkan side of the maps)
    "wso_set_exportable": (_int, [_vp, _int]),
    "wso_export_fd": (_int, [_vp, _int, C.POINTER(_int), C.POINTER(C.c_size_t)]),
    "wso_import_external_fd": (_int, [_vp, _int, _int, C.c_size_t, C.c_size_t]),
    "wso_import_semaphore_fd": (_int, [_vp, _int, _int, _int]),
    "wso_signal_semaphore": (_int, [_vp, _int, C.c_uint64]),
    "wso_wait_semaphore": (_int, [_vp, _int, C.c_uint64]),
    "wso_set_stream": (_int, [_vp, _vp]),
    "wso_alloc_host": (_int, [C.c_size_t, C.POINTER(_vp)]),
    "wso_free_host": (_int, [_vp]),
    "wso_select_kernels": (_int, [_int]),
    "wso_register_host": (_int, [_vp, C.c_size_t]),
    "wso_unregister_host": (_int, [_vp]),
    "wso_get_stats": (_int, [_vp, C.POINTER(C.c_uint64), C.POINTER(_u32)]),
    "wso_set_frame_graph": (_int, [_vp, _int]),
    "wso_get_frame_graph_stats": (_int, [_vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "wso_set_profiling": (_int, [_vp, _int]),
    "wso_get_profile": (_int, [_vp, _vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    # slab-decomposed path (one large grid over several devices)
    "wso_slab_create": (_int, [_pp, _int, _u32, _u32, C.POINTER(_vp)]),
    "wso_slab_destroy": (_int, [_vp]),
    "wso_slab_import_h0": (_int, [_vp, _vp]),
    "wso_slab_prepare_counter": (_int, [_vp, C.c_uint64]),
    "wso_slab_prepare_counter_device": (_int, [_vp, C.c_uint64]),
    "wso_counter_h0": (_int, [_pp, C.c_uint64, _u32, _u32, _vp]),
    "wso_slab_set_lambda": (_int, [_vp, _f32]),
    "wso_slab_set_stream": (_int, [_vp, _vp]),
    "wso_slab_buffers": (_int, [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(C.c_size_t), C.POINTER(_vp)]),
    "wso_slab_ipc_handle": (_int, [_vp, _vp]),
    "wso_slab_open_peer": (_int, [_vp, _u32, _vp]),
    "wso_slab_set_fused": (_int, [_vp, _int]),
    "wso_slab_force_pair": (_int, [_vp, _int]),
    "wso_slab_pass1": (_int, [_vp, _f32]),
    "wso_slab_exchange": (_int, [_vp]),
    "wso_slab_pass1_fields": (_int, [_vp, _f32, _int, _int]),
    "wso_slab_exchange_fields": (_int, [_vp, _int, _int, _vp]),
    "wso_slab_fields_per_group": (_int, [_vp]),
    "wso_slab_heights": (_int, [_vp]),
    "wso_slab_pass2": (_int, [_vp]),
    "wso_slab_sync": (_int, [_vp]),
    "wso_slab_read_heights": (_int, [_vp, C.POINTER(_f32), C.POINTER(_f32), C.POINTER(_f32)]),
    "wso_slab_map_device": (_int, [_vp, _int, C.POINTER(_vp), C.POINTER(_u32)]),
    "wso_slab_copy_rows": (_int, [_vp, _int, _vp]),
    "wso_slab_row_index": (_int, [_vp, _vp]),
    "wso_slab_last_error": (C.c_char_p, [_vp]),
    "wso_last_error": (C.c_char_p, [_vp]),
    "wso_version": (C.c_char_p, []),
}

_lib = None


def load():
    """Load libwsocean.so and bind every declared symbol; raises if the library is absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} not built - run `python -m watersurfacerendering_b200.build` "
                "(there is no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)  # AttributeError if the .so does not export it
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


class WsoError(RuntimeError):
    def __init__(self, status: int, msg: str):
        super().__init__(f"{STATUS_NAMES.get(status, status)}: {msg}")
        self.status = status


def check(status: int, ctx=None):
    if status != WSO_OK:
        msg = load().wso_last_error(ctx)
        raise WsoError(status, msg.decode() if msg else "")


def check_slab(status: int, slab=None):
    if status != WSO_OK:
        msg = load().wso_slab_last_error(slab)
        raise WsoError(status, msg.decode() if msg else "")
