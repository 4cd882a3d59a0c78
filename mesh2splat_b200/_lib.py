"""ctypes binding of libm2s.so (include/m2s.h).  No fallback: if the library is missing or there is
no CUDA device, calls raise."""
from __future__ import annotations

import ctypes as C
import os

from . import _abi

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("M2S_LIB") or os.path.join(_HERE, "libm2s.so")  # M2S_LIB: tuning variants (build.py --out)
_lib = None

# every symbol include/m2s.h declares (tests check the .so exports all of them)
SYMBOLS = [
    "m2s_version", "m2s_last_error", "m2s_status_string", "m2s_record_stride", "m2s_reference_capacity",
    "m2s_params_default", "m2s_ctx_create", "m2s_ctx_destroy", "m2s_ctx_device", "m2s_ctx_sm_count", "m2s_ctx_status",
    "m2s_compute_bboxes", "m2s_scene_upload", "m2s_scene_upload_range", "m2s_scene_h2d_bytes", "m2s_scene_free", "m2s_scene_read_mip",
    "m2s_convert_enqueue", "m2s_convert", "m2s_convert_timed", "m2s_convert_host", "m2s_convert_gather_enqueue",
    "m2s_ply_header", "m2s_ply_encode", "m2s_ply_write", "m2s_convert_file",
    "m2s_glb_load", "m2s_hscene_view", "m2s_hscene_primitive_name", "m2s_hscene_free",
    "m2s_prepass", "m2s_prepass_enqueue",
    "m2s_sort_quads", "m2s_sort_quads_enqueue", "m2s_splat", "m2s_splat_enqueue",
]


class M2SError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"m2s status {status}: {message}")
        self.status = status
        self.message = message


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing — build it with `python -m mesh2splat_b200.build` "
            "(there is no CPU fallback for the conversion path)")
    L = C.CDLL(LIB_PATH)
    missing = [n for n in SYMBOLS if not hasattr(L, n)]
    if missing:
        raise RuntimeError(f"{LIB_PATH} is stale: missing symbols {missing}; rebuild with `python -m mesh2splat_b200.build --force`")
    vp, u32, u64, f32, i32 = C.c_void_p, C.c_uint32, C.c_uint64, C.c_float, C.c_int
    L.m2s_version.restype = i32
    L.m2s_last_error.restype = C.c_char_p
    L.m2s_status_string.restype = C.c_char_p
    L.m2s_status_string.argtypes = [i32]
    L.m2s_record_stride.restype = u32
    L.m2s_record_stride.argtypes = [u32]
    L.m2s_reference_capacity.restype = u64
    L.m2s_reference_capacity.argtypes = [u32, u32]
    L.m2s_params_default.restype = None
    L.m2s_params_default.argtypes = [C.POINTER(_abi.m2s_params)]
    L.m2s_ctx_create.restype = i32
    L.m2s_ctx_create.argtypes = [i32, C.POINTER(vp)]
    L.m2s_ctx_destroy.restype = None
    L.m2s_ctx_destroy.argtypes = [vp]
    L.m2s_ctx_device.restype = i32
    L.m2s_ctx_device.argtypes = [vp]
    L.m2s_ctx_status.restype = i32
    L.m2s_ctx_status.argtypes = [vp]
    L.m2s_ctx_sm_count.restype = i32
    L.m2s_ctx_sm_count.argtypes = [vp]
    L.m2s_compute_bboxes.restype = i32
    L.m2s_compute_bboxes.argtypes = [vp, C.POINTER(_abi.m2s_primitive), u32, i32]
    L.m2s_scene_upload.restype = i32
    L.m2s_scene_upload.argtypes = [vp, C.POINTER(_abi.m2s_scene), C.POINTER(vp)]
    L.m2s_scene_upload_range.restype = i32
    L.m2s_scene_upload_range.argtypes = [vp, C.POINTER(_abi.m2s_scene), u32, u64, u64, C.POINTER(vp)]
    L.m2s_scene_h2d_bytes.restype = u64
    L.m2s_scene_h2d_bytes.argtypes = [vp]
    L.m2s_scene_free.restype = None
    L.m2s_scene_free.argtypes = [vp, vp]
    L.m2s_scene_read_mip.restype = i32
    L.m2s_scene_read_mip.argtypes = [vp, vp, u32, u32, vp, C.POINTER(u32), C.POINTER(u32)]
    L.m2s_convert_enqueue.restype = i32
    L.m2s_convert_enqueue.argtypes = [vp, vp, C.POINTER(_abi.m2s_params), vp, u64, vp, vp, vp]
    L.m2s_convert_gather_enqueue.restype = i32
    L.m2s_convert_gather_enqueue.argtypes = [vp, vp, C.POINTER(_abi.m2s_params), C.POINTER(_abi.m2s_peers), u64, vp, vp]
    L.m2s_convert.restype = i32
    L.m2s_convert.argtypes = [vp, vp, C.POINTER(_abi.m2s_params), vp, u64, vp, C.POINTER(_abi.m2s_result)]
    L.m2s_convert_timed.restype = i32
    L.m2s_convert_timed.argtypes = [vp, vp, C.POINTER(_abi.m2s_params), vp, u64, C.POINTER(f32), C.POINTER(f32)]
    L.m2s_convert_host.restype = i32
    L.m2s_convert_host.argtypes = [vp, C.POINTER(_abi.m2s_scene), C.POINTER(_abi.m2s_params), vp, u64, vp,
                                   C.POINTER(_abi.m2s_result)]
    L.m2s_ply_header.restype = C.c_size_t
    L.m2s_ply_header.argtypes = [u32, u64, C.c_char_p, C.c_size_t]
    L.m2s_ply_encode.restype = i32
    L.m2s_ply_encode.argtypes = [vp, vp, u64, u32, f32, vp, vp]
    L.m2s_ply_write.restype = i32
    L.m2s_ply_write.argtypes = [C.c_char_p, vp, u64, u32, f32]
    L.m2s_convert_file.restype = i32
    L.m2s_convert_file.argtypes = [vp, C.c_char_p, u32, f32, u32, C.c_char_p, C.POINTER(_abi.m2s_result)]
    L.m2s_glb_load.restype = i32
    L.m2s_glb_load.argtypes = [C.c_char_p, i32, C.POINTER(vp)]
    L.m2s_hscene_view.restype = C.POINTER(_abi.m2s_scene)
    L.m2s_hscene_view.argtypes = [vp]
    L.m2s_hscene_primitive_name.restype = C.c_char_p
    L.m2s_hscene_primitive_name.argtypes = [vp, u32]
    L.m2s_hscene_free.restype = None
    L.m2s_hscene_free.argtypes = [vp]
    L.m2s_prepass_enqueue.restype = i32
    L.m2s_prepass_enqueue.argtypes = [vp, vp, u64, vp, C.POINTER(_abi.m2s_prepass_params), vp, vp, vp, vp]
    L.m2s_prepass.restype = i32
    L.m2s_prepass.argtypes = [vp, vp, u64, C.POINTER(_abi.m2s_prepass_params), vp, vp, C.POINTER(u32)]
    L.m2s_sort_quads_enqueue.restype = i32
    L.m2s_sort_quads_enqueue.argtypes = [vp, vp, vp, u64, vp, vp, vp, vp]
    L.m2s_sort_quads.restype = i32
    L.m2s_sort_quads.argtypes = [vp, vp, vp, u64, vp, vp, C.POINTER(f32)]
    L.m2s_splat_enqueue.restype = i32
    L.m2s_splat_enqueue.argtypes = [vp, vp, u64, vp, C.POINTER(_abi.m2s_splat_params), C.POINTER(_abi.m2s_gbuffer), u64, vp]
    L.m2s_splat.restype = i32
    L.m2s_splat.argtypes = [vp, vp, u64, vp, C.POINTER(_abi.m2s_splat_params), C.POINTER(_abi.m2s_gbuffer), C.POINTER(u64), C.POINTER(f32)]
    _lib = L
    return L


def check(status: int, allow=()) -> int:
    if status != _abi.M2S_OK and status not in allow:
        raise M2SError(status, lib().m2s_last_error().decode("utf-8", "replace"))
    return status
