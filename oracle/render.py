"""CPU checker of the viewer passes after the prepass (SURVEY 8 f-5, f-6): ctypes wrappers of
oracle/libm2s_render_oracle.so (oracle/m2s_render_oracle.c) and of the reference's own splatting shaders compiled as
C++ (oracle/_ref/libm2s_refsplat.so).  Both are built by oracle/build_render.py.  TEST INFRASTRUCTURE: only tests/,
__graft_entry__.smoke() and tests/golden/make_golden_splat.py import this module; mesh2splat_b200 never does."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from mesh2splat_b200 import _abi

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        path = os.path.join(_HERE, "libm2s_render_oracle.so")
        if not os.path.exists(path):
            from . import build_render  # noqa: WPS433
            build_render.build_render_oracle()
        _lib = C.CDLL(path)
    return _lib


# ---- viewer: depth sort and splatting pass (SURVEY 8 f-5, f-6) ----------------------------------------------------------
def sort_quads(depths: np.ndarray) -> np.ndarray:
    """orc_sort_quads: the prepass index of each quad in the stable ascending order of floatBitsToUint(depth)."""
    L = lib()
    L.orc_sort_quads.restype = None
    L.orc_sort_quads.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]
    d = np.ascontiguousarray(depths, np.float32)
    order = np.zeros(max(1, len(d)), np.uint32)
    L.orc_sort_quads(d.ctypes.data, len(d), order.ctypes.data)
    return order[: len(d)]


def splat(quads: np.ndarray, width: int, height: int, render_mode: int = 0) -> dict:
    """orc_splat: GaussianSplattingPass of the quads (n x 24 float32, draw order) into a cleared width x height G-buffer.
    Returns {target: (height, width, 4)} with position, normal, depth float16 and albedo, metallic_roughness uint8;
    row 0 = the bottom row."""
    L = lib()
    L.orc_splat.restype = None
    L.orc_splat.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32] + [C.c_void_p] * 5
    q = np.ascontiguousarray(quads, np.float32).reshape(-1, 24)
    out = {name: np.zeros((height, width, 4), np.float16 if kind == "f16" else np.uint8) for name, kind in _abi.GBUFFER_TARGETS}
    L.orc_splat(q.ctypes.data, len(q), width, height, render_mode, *[out[name].ctypes.data for name, _ in _abi.GBUFFER_TARGETS])
    return out


def splat_vertex(quad: np.ndarray, width: float, height: float) -> np.ndarray:
    """gl_Position of the quad's 4 corners (4 x 4) as gaussianSplattingVS.glsl computes them."""
    L = lib()
    L.orc_splat_vertex.restype = None
    L.orc_splat_vertex.argtypes = [C.c_void_p, C.c_float, C.c_float, C.c_void_p]
    q = np.ascontiguousarray(quad, np.float32).reshape(24)
    out = np.zeros((4, 4), np.float32)
    L.orc_splat_vertex(q.ctypes.data, width, height, out.ctypes.data)
    return out


def splat_fragments(quad: np.ndarray, width: float, height: float, render_mode: int, frag_xy: np.ndarray) -> np.ndarray:
    """gaussianSplattingPS.glsl outputs (n x 5 x 4: position, normal, albedo, depth, metallic-roughness) at gl_FragCoord.xy."""
    L = lib()
    L.orc_splat_fragments.restype = None
    L.orc_splat_fragments.argtypes = [C.c_void_p, C.c_float, C.c_float, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p]
    q = np.ascontiguousarray(quad, np.float32).reshape(24)
    f = np.ascontiguousarray(frag_xy, np.float32).reshape(-1, 2)
    out = np.zeros((len(f), 5, 4), np.float32)
    L.orc_splat_fragments(q.ctypes.data, width, height, render_mode, f.ctypes.data, len(f), out.ctypes.data)
    return out


_refsplat = None


def ref_splat_lib():
    """The reference's own splatting shaders compiled as C++ (oracle/_ref/libm2s_refsplat.so), or None."""
    global _refsplat
    if _refsplat is None:
        path = os.path.join(_HERE, "_ref", "libm2s_refsplat.so")
        if not os.path.exists(path):
            return None
        _refsplat = C.CDLL(path)
        _refsplat.ref_splat.restype = None
        _refsplat.ref_splat.argtypes = [C.c_void_p, C.c_float, C.c_float, C.c_int, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]
    return _refsplat


def ref_splat(quad: np.ndarray, width: float, height: float, render_mode: int, frag_xy: np.ndarray):
    """gaussianSplattingVS.glsl + gaussianSplattingPS.glsl themselves: (corners 4 x 4, outputs n x 5 x 4)."""
    L = ref_splat_lib()
    if L is None:
        raise RuntimeError("oracle/_ref/libm2s_refsplat.so is not built")
    q = np.ascontiguousarray(quad, np.float32).reshape(24)
    f = np.ascontiguousarray(frag_xy, np.float32).reshape(-1, 2)
    corners = np.zeros((4, 4), np.float32)
    out = np.zeros((len(f), 5, 4), np.float32)
    L.ref_splat(q.ctypes.data, width, height, render_mode, f.ctypes.data, len(f), corners.ctypes.data, out.ctypes.data)
    return corners, out
