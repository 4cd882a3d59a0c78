"""ctypes mirror of include/m2s.h (structs, enums) and the host-side Scene container.

No compute here: this is the marshalling layer between numpy arrays and the C ABI.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field

import numpy as np

# ---- enums (include/m2s.h) ------------------------------------------------------------------
M2S_OK, M2S_E_INVALID, M2S_E_NOGPU, M2S_E_CUDA, M2S_E_CAPACITY, M2S_E_IO, M2S_E_FORMAT = range(7)
LAYOUT_REF96, LAYOUT_PACKED56, LAYOUT_PLY_STANDARD, LAYOUT_PLY_PBR, LAYOUT_PLY_COMPRESSED = range(5)
FLAG_NONE, FLAG_UNCAPPED = 0, 1
FLOATS_PER_TRIANGLE = 36
MAX_MIP_LEVEL = 4
REFERENCE_MAX_GAUSSIANS = 7_000_000
STRIDES = {LAYOUT_REF96: 96, LAYOUT_PACKED56: 56, LAYOUT_PLY_STANDARD: 248, LAYOUT_PLY_PBR: 76,
           LAYOUT_PLY_COMPRESSED: 48}
# which .ply format (savePlyVector FORMAT, parsers.cpp:631-651) a row layout corresponds to
PLY_FORMAT_LAYOUT = {0: LAYOUT_PLY_STANDARD, 1: LAYOUT_PLY_PBR, 2: LAYOUT_PLY_COMPRESSED}


class m2s_texture(C.Structure):
    _fields_ = [("rgba", C.c_void_p), ("width", C.c_uint32), ("height", C.c_uint32)]


class m2s_primitive(C.Structure):
    _fields_ = [("first_triangle", C.c_uint64), ("triangle_count", C.c_uint64),
                ("bbox_min", C.c_float * 3), ("bbox_max", C.c_float * 3),
                ("base_color_factor", C.c_float * 4),
                ("albedo_texture", C.c_int32), ("normal_texture", C.c_int32),
                ("metallic_roughness_texture", C.c_int32), ("reserved", C.c_int32)]


class m2s_scene(C.Structure):
    _fields_ = [("triangles", C.c_void_p), ("triangle_count", C.c_uint64),
                ("primitives", C.POINTER(m2s_primitive)), ("primitive_count", C.c_uint32),
                ("textures", C.POINTER(m2s_texture)), ("texture_count", C.c_uint32)]


class m2s_params(C.Structure):
    _fields_ = [("resolution", C.c_uint32), ("gaussian_std", C.c_float),
                ("max_gaussians", C.c_uint64), ("layout", C.c_uint32), ("flags", C.c_uint32),
                ("first_triangle", C.c_uint64), ("triangle_count", C.c_uint64),
                ("row_begin", C.c_uint32), ("row_end", C.c_uint32)]


class m2s_result(C.Structure):
    _fields_ = [("total", C.c_uint64), ("written", C.c_uint64), ("cap", C.c_uint64),
                ("device_ms", C.c_float)]


MAX_PEERS = 8


class m2s_prepass_params(C.Structure):
    """include/m2s.h: the uniforms of GaussiansPrepass::execute; matrices column-major (glm::mat4)."""
    _fields_ = [("world_to_view", C.c_float * 16), ("view_to_clip", C.c_float * 16), ("model_to_world", C.c_float * 16),
                ("resolution", C.c_float * 2), ("near_far", C.c_float * 2), ("std_dev", C.c_float), ("render_mode", C.c_uint32),
                ("layout", C.c_uint32), ("reserved", C.c_uint32)]


QUAD_BYTES = 96
MAX_SPLAT_SIZE = 4096


class m2s_splat_params(C.Structure):
    """include/m2s.h: viewport and render mode of GaussianSplattingPass::execute."""
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("render_mode", C.c_uint32), ("reserved", C.c_uint32)]


class m2s_gbuffer(C.Structure):
    """include/m2s.h: the five G-buffer images (device pointers, row-major, row 0 = bottom row)."""
    _fields_ = [("position", C.c_void_p), ("normal", C.c_void_p), ("albedo", C.c_void_p), ("depth", C.c_void_p),
                ("metallic_roughness", C.c_void_p)]


# G-buffer targets: (name, storage) as Renderer::createGBuffer (renderer.cpp:329-379) allocates them
GBUFFER_TARGETS = (("position", "f16"), ("normal", "f16"), ("albedo", "u8"), ("depth", "f16"), ("metallic_roughness", "u8"))


def make_prepass_params(world_to_view, view_to_clip, model_to_world, resolution, near_far, std_dev: float, render_mode: int, layout: int):
    p = m2s_prepass_params()
    for name, m in (("world_to_view", world_to_view), ("view_to_clip", view_to_clip), ("model_to_world", model_to_world)):
        setattr(p, name, (C.c_float * 16)(*[float(v) for v in np.asarray(m, np.float32).ravel()]))
    p.resolution = (C.c_float * 2)(float(resolution[0]), float(resolution[1]))
    p.near_far = (C.c_float * 2)(float(near_far[0]), float(near_far[1]))
    p.std_dev, p.render_mode, p.layout, p.reserved = float(std_dev), int(render_mode), int(layout), 0
    return p


class m2s_peers(C.Structure):
    _fields_ = [("world", C.c_uint32), ("rank", C.c_uint32), ("out", C.c_void_p * MAX_PEERS), ("xch", C.c_void_p * MAX_PEERS)]


def make_params(resolution: int, layout: int = LAYOUT_REF96, gaussian_std: float = 0.65,
                max_gaussians: int = 0, flags: int = 0, first_triangle: int = 0,
                triangle_count: int = 0, row_begin: int = 0, row_end: int = 0) -> m2s_params:
    return m2s_params(int(resolution), float(gaussian_std), int(max_gaussians), int(layout),
                      int(flags), int(first_triangle), int(triangle_count), int(row_begin), int(row_end))


def reference_capacity(resolution: int, primitive_count: int) -> int:
    """min(6 R^2 meshCount, 7e6): ConversionPass.cpp:21-24."""
    return min(6 * resolution * resolution * max(1, primitive_count), REFERENCE_MAX_GAUSSIANS)


@dataclass
class Primitive:
    """One glTF primitive == one utils::Mesh == one draw call of the reference."""
    first_triangle: int
    triangle_count: int
    base_color_factor: tuple = (1.0, 1.0, 1.0, 1.0)
    albedo_texture: int = -1
    normal_texture: int = -1
    metallic_roughness_texture: int = -1
    bbox_min: tuple = (0.0, 0.0, 0.0)
    bbox_max: tuple = (0.0, 0.0, 0.0)
    name: str = "mesh"


@dataclass
class Scene:
    """Host-side scene: what SceneManager::loadModel leaves in RenderContext, minus GL handles.

    triangles: float32 (T, 36) — 3 x {position xyz, normal xyz, tangent xyzw, uv}, world space
    textures:  list of uint8 (H, W, 4), row 0 first
    """
    triangles: np.ndarray
    primitives: list = field(default_factory=list)
    textures: list = field(default_factory=list)

    def __post_init__(self):
        t = np.ascontiguousarray(self.triangles, dtype=np.float32)
        if t.ndim != 2 or t.shape[1] != FLOATS_PER_TRIANGLE:
            t = t.reshape(-1, FLOATS_PER_TRIANGLE)
        self.triangles = t
        self.textures = [np.ascontiguousarray(x, dtype=np.uint8) for x in self.textures]
        for x in self.textures:
            if x.ndim != 3 or x.shape[2] != 4:
                raise ValueError("textures must be (H, W, 4) uint8")
        if not self.primitives:
            self.primitives = [Primitive(0, len(t))]

    @property
    def triangle_count(self) -> int:
        return int(self.triangles.shape[0])

    def compute_bboxes(self, cumulative: bool = True) -> None:
        """Reference rule (SceneManager.cpp:476-477,514-520,527): primitive k gets the union box
        of primitives 0..k when cumulative (the reference's behaviour)."""
        mn = np.full(3, np.finfo(np.float32).max, np.float32)
        mx = -mn
        pos = self.triangles.reshape(-1, 3, 12)[:, :, 0:3]
        for p in self.primitives:
            if not cumulative:
                mn = np.full(3, np.finfo(np.float32).max, np.float32)
                mx = -mn
            sl = pos[p.first_triangle:p.first_triangle + p.triangle_count].reshape(-1, 3)
            if len(sl):
                mn = np.minimum(mn, sl.min(axis=0))
                mx = np.maximum(mx, sl.max(axis=0))
            p.bbox_min = tuple(float(v) for v in mn)
            p.bbox_max = tuple(float(v) for v in mx)

    def c_struct(self):
        """Returns (m2s_scene, keepalive) — keep `keepalive` referenced while the struct is used."""
        prims = (m2s_primitive * max(1, len(self.primitives)))()
        for i, p in enumerate(self.primitives):
            prims[i].first_triangle = p.first_triangle
            prims[i].triangle_count = p.triangle_count
            prims[i].bbox_min = (C.c_float * 3)(*p.bbox_min)
            prims[i].bbox_max = (C.c_float * 3)(*p.bbox_max)
            prims[i].base_color_factor = (C.c_float * 4)(*p.base_color_factor)
            prims[i].albedo_texture = p.albedo_texture
            prims[i].normal_texture = p.normal_texture
            prims[i].metallic_roughness_texture = p.metallic_roughness_texture
        texs = (m2s_texture * max(1, len(self.textures)))()
        for i, t in enumerate(self.textures):
            texs[i].rgba = t.ctypes.data
            texs[i].width = t.shape[1]
            texs[i].height = t.shape[0]
        s = m2s_scene()
        s.triangles = self.triangles.ctypes.data
        s.triangle_count = self.triangle_count
        s.primitives = prims
        s.primitive_count = len(self.primitives)
        s.textures = texs
        s.texture_count = len(self.textures)
        return s, (prims, texs, self.triangles, self.textures)

    def texture_bytes(self) -> int:
        return int(sum(t.nbytes for t in self.textures))


def record_dtype(layout: int) -> np.dtype:
    """numpy view of one output record."""
    if layout == LAYOUT_REF96:
        return np.dtype([("position", "<f4", 4), ("color", "<f4", 4), ("scale", "<f4", 4),
                         ("normal", "<f4", 4), ("rotation", "<f4", 4), ("pbr", "<f4", 4)])
    if layout == LAYOUT_PACKED56:
        return np.dtype([("xyz", "<f4", 3), ("rot", "<f4", 4), ("log_scale", "<f4", 3),
                         ("sh0", "<f4", 3), ("opacity", "<f4")])
    if layout == LAYOUT_PLY_STANDARD:
        return np.dtype([("xyz", "<f4", 3), ("normal", "<f4", 3), ("f_dc", "<f4", 3),
                         ("f_rest", "<f4", 45), ("opacity", "<f4"), ("scale", "<f4", 3),
                         ("rot", "<f4", 4)])
    if layout == LAYOUT_PLY_PBR:
        return np.dtype([("xyz", "<f4", 3), ("normal", "<f4", 3), ("f_dc", "<f4", 3),
                         ("metallic", "<f4"), ("roughness", "<f4"), ("opacity", "<f4"),
                         ("scale", "<f4", 3), ("rot", "<f4", 4)])
    if layout == LAYOUT_PLY_COMPRESSED:
        return np.dtype([("xyz", "<f4", 3), ("rgba", "u1", 4), ("rot", "<f4", 4),
                         ("scale", "<f4", 3), ("octa", "u1", 2), ("roughness", "u1"),
                         ("metallic", "u1")])
    raise ValueError(f"unknown layout {layout}")
