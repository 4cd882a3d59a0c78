"""Host-side mirror of the reference's interface for the conversion path, over the C ABI.

Reference surface (src/utils/SceneManager.hpp:18-20, src/renderer/renderPasses/RenderPass.hpp:10-28,
src/renderer/RenderContext.hpp:28-124):

    SceneManager::loadModel(path, parentFolder)      -> SceneManager.loadModel / .setScene
    ConversionPass::execute(RenderContext&)          -> ConversionPass.execute(renderContext)
    SceneManager::exportPly(outPath, exportFormat)   -> SceneManager.exportPly

plus the plain functional form `Context.convert(...)`.  torch is used only to own device buffers
(torch.empty(..., device="cuda")) and pinned host buffers; every computation is a call into
libm2s.so.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import _abi
from ._lib import M2SError, check, lib


def _torch():
    import torch  # noqa: WPS433 (lazy: the ABI layer itself does not need torch)
    return torch


class DeviceScene:
    """Device-resident scene (triangles, primitive table, mip chains): what loadModel leaves on the
    GPU in the reference (VBOs + GL textures)."""

    def __init__(self, ctx: "Context", handle: int, scene: _abi.Scene):
        self.ctx, self.handle = ctx, handle
        self.primitive_count = len(scene.primitives)
        self.triangle_count = scene.triangle_count
        self.texture_shapes = [t.shape[:2] for t in scene.textures]

    def read_mip(self, texture: int, level: int) -> np.ndarray:
        h, w = self.texture_shapes[texture]
        buf = np.zeros((h, w, 4), np.uint8)
        ow, oh = C.c_uint32(0), C.c_uint32(0)
        check(lib().m2s_scene_read_mip(self.ctx.handle, self.handle, texture, level, buf.ctypes.data,
                                       C.byref(ow), C.byref(oh)))
        return buf.reshape(-1)[: ow.value * oh.value * 4].reshape(oh.value, ow.value, 4).copy()

    def h2d_bytes(self) -> int:
        return int(lib().m2s_scene_h2d_bytes(self.handle))

    def free(self):
        if self.handle:
            lib().m2s_scene_free(self.ctx.handle, self.handle)
            self.handle = 0

    def __del__(self):
        try:
            self.free()
        except Exception:  # noqa: BLE001
            pass


@dataclass
class ConvertOutput:
    data: object            # torch.uint8 tensor on the device, capacity * stride bytes
    keys: object            # torch.int64 tensor (fragment identity) or None
    total: int              # fragments generated (reference: numberOfGaussians)
    written: int            # records stored = min(total, cap)
    cap: int
    device_ms: float
    layout: int
    overflow: bool

    def numpy(self) -> np.ndarray:
        stride = _abi.STRIDES[self.layout]
        raw = self.data[: self.written * stride].cpu().numpy()
        return raw.view(_abi.record_dtype(self.layout))

    def keys_numpy(self):
        return None if self.keys is None else self.keys[: self.written].cpu().numpy().view(np.uint64)


@dataclass
class GBuffer:
    """The five targets of GaussianSplattingPass (renderer.cpp:329-379) as torch device tensors of shape (height, width, 4),
    row 0 = the bottom row (GL's window origin): position, normal, depth float16; albedo, metallic_roughness uint8."""
    position: object
    normal: object
    albedo: object
    depth: object
    metallic_roughness: object
    render_mode: int
    pairs: int = 0              # (tile, quad) pairs the splat walked
    device_ms: float = 0.0      # device time of the splatting pass
    survivors: int = 0          # quads splatted (Context.render: the prepass's count)

    @staticmethod
    def empty(width: int, height: int, render_mode: int, device) -> "GBuffer":
        torch = _torch()
        mk = {"f16": lambda: torch.empty((height, width, 4), dtype=torch.float16, device=device),
              "u8": lambda: torch.empty((height, width, 4), dtype=torch.uint8, device=device)}
        return GBuffer(*[mk[kind]() for _, kind in _abi.GBUFFER_TARGETS], render_mode=render_mode)

    def c_struct(self) -> _abi.m2s_gbuffer:
        return _abi.m2s_gbuffer(*[getattr(self, name).data_ptr() for name, _ in _abi.GBUFFER_TARGETS])

    def numpy(self) -> dict:
        """{target name: numpy array (height, width, 4)}: float16 or uint8."""
        return {name: getattr(self, name).cpu().numpy() for name, _ in _abi.GBUFFER_TARGETS}

    def image(self, mode: int | None = None) -> np.ndarray:
        """The non-lit composite of the deferred pass (gaussianSplattingDeferredPS.glsl:120-131), float32 (height, width, 4):
        mode 5 shows (metallic_roughness.rg, 0, 1), every other mode (albedo.rgb, 1).  Mode 6 (lighting) is not provided."""
        mode = self.render_mode if mode is None else mode
        if mode == 6:
            raise ValueError("render mode 6 needs the lighting of the deferred pass, which is not provided")
        src = (self.metallic_roughness if mode == 5 else self.albedo).cpu().numpy().astype(np.float32) / np.float32(255.0)
        out = np.zeros(src.shape, np.float32)
        out[..., 3] = 1.0
        out[..., 0:2] = src[..., 0:2]
        if mode != 5:
            out[..., 2] = src[..., 2]
        return out


class Context:
    """One per GPU (m2s_ctx)."""

    def __init__(self, device: int = 0):
        h = C.c_void_p(0)
        check(lib().m2s_ctx_create(device, C.byref(h)))
        self.handle = h.value
        self.device = device
        self.sm_count = lib().m2s_ctx_sm_count(self.handle)

    def close(self):
        if getattr(self, "handle", 0):
            lib().m2s_ctx_destroy(self.handle)
            self.handle = 0

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # ---- inputs ----
    def upload(self, scene: _abi.Scene) -> DeviceScene:
        cs, keep = scene.c_struct()
        h = C.c_void_p(0)
        check(lib().m2s_scene_upload(self.handle, C.byref(cs), C.byref(h)))
        del keep
        return DeviceScene(self, h.value, scene)

    def upload_range(self, scene: _abi.Scene, layout: int, first_triangle: int, triangle_count: int, c_scene=None) -> DeviceScene:
        """One shard (m2s_scene_upload_range): the triangle range at its global indices + only the texture rows it samples."""
        cs, keep = c_scene if c_scene is not None else scene.c_struct()
        h = C.c_void_p(0)
        check(lib().m2s_scene_upload_range(self.handle, C.byref(cs), layout, first_triangle, triangle_count, C.byref(h)))
        del keep
        return DeviceScene(self, h.value, scene)

    # ---- the hot path ----
    def default_capacity(self, dscene: DeviceScene, resolution: int, max_gaussians: int, flags: int) -> int:
        if max_gaussians:
            return max_gaussians
        if flags & _abi.FLAG_UNCAPPED:
            return 6 * resolution * resolution * max(1, dscene.primitive_count)
        return _abi.reference_capacity(resolution, dscene.primitive_count)

    def convert(self, dscene: DeviceScene, resolution: int, layout: int = _abi.LAYOUT_REF96,
                gaussian_std: float = 0.65, max_gaussians: int = 0, flags: int = 0, first_triangle: int = 0,
                triangle_count: int = 0, capacity: int | None = None, want_keys: bool = False,
                out=None, keys=None, allow_overflow: bool = True, row_begin: int = 0, row_end: int = 0) -> ConvertOutput:
        torch = _torch()
        stride = _abi.STRIDES[layout]
        if capacity is None:
            capacity = self.default_capacity(dscene, resolution, max_gaussians, flags)
        dev = torch.device("cuda", self.device)
        if out is None:
            out = torch.empty(max(1, capacity) * stride, dtype=torch.uint8, device=dev)
        if want_keys and keys is None:
            keys = torch.empty(max(1, capacity), dtype=torch.int64, device=dev)
        p = _abi.make_params(resolution, layout, gaussian_std, max_gaussians, flags, first_triangle, triangle_count,
                             row_begin, row_end)
        res = _abi.m2s_result()
        st = check(lib().m2s_convert(self.handle, dscene.handle, C.byref(p), out.data_ptr(), capacity,
                                     keys.data_ptr() if keys is not None else None, C.byref(res)),
                   allow=(_abi.M2S_E_CAPACITY,) if allow_overflow else ())
        return ConvertOutput(out, keys, int(res.total), int(res.written), int(res.cap), float(res.device_ms), layout,
                             st == _abi.M2S_E_CAPACITY)

    def convert_enqueue(self, dscene: DeviceScene, params: _abi.m2s_params, out, capacity: int, keys=None,
                        total=None, stream: int = 0) -> None:
        """Enqueue only (no synchronisation); out/keys/total are torch device tensors."""
        check(lib().m2s_convert_enqueue(self.handle, dscene.handle, C.byref(params), out.data_ptr(), capacity,
                                        keys.data_ptr() if keys is not None else None,
                                        total.data_ptr() if total is not None else None, stream or None))

    def prepass(self, records, count: int, layout: int, world_to_view, view_to_clip, model_to_world, resolution, near_far,
                std_dev: float, render_mode: int = 0):
        """GaussiansPrepass::execute on device-resident records (a torch uint8 tensor, e.g. ConvertOutput.data): returns
        (quads [m, 24] float32, depths [m] float32) as numpy arrays, in atomic arrival order (m2s_prepass)."""
        import torch
        dev = records.device
        quads = torch.empty(max(1, count) * _abi.QUAD_BYTES, dtype=torch.uint8, device=dev)
        depths = torch.empty(max(1, count), dtype=torch.float32, device=dev)
        p = _abi.make_prepass_params(world_to_view, view_to_clip, model_to_world, resolution, near_far, std_dev, render_mode, layout)
        valid = C.c_uint32(0)
        check(lib().m2s_prepass(self.handle, records.data_ptr(), count, C.byref(p), quads.data_ptr(), depths.data_ptr(), C.byref(valid)))
        m = int(valid.value)
        return quads[: m * _abi.QUAD_BYTES].cpu().numpy().view(np.float32).reshape(m, 24).copy(), depths[:m].cpu().numpy().copy()

    def sort_quads(self, quads, depths, count: int, d_count=None, order: bool = True):
        """RadixSortPass on device-resident prepass output (torch tensors: quads uint8/float32 of count x 96 B, depths float32):
        the stable ascending order of floatBitsToUint(depth).  d_count: optional int32 device tensor (the prepass's counter)
        that overrides `count` downwards.  Returns (sorted quads as a float32 tensor [count, 24], prepass index of each
        sorted quad as an int32 tensor [count] or None); with d_count only the first *d_count rows are defined."""
        torch = _torch()
        dev = quads.device
        torch.cuda.current_stream(dev).synchronize()   # inputs made on torch's stream; the sort runs on the context stream
        sorted_q = torch.empty((max(1, count), 24), dtype=torch.float32, device=dev)
        idx = torch.empty(max(1, count), dtype=torch.int32, device=dev) if order else None
        check(lib().m2s_sort_quads_enqueue(self.handle, quads.data_ptr(), depths.data_ptr(), count,
                                           d_count.data_ptr() if d_count is not None else None, sorted_q.data_ptr(),
                                           idx.data_ptr() if idx is not None else None, None))
        self.synchronize()
        return sorted_q[:count], (idx[:count] if idx is not None else None)

    def splat(self, sorted_quads, count: int, width: int, height: int, render_mode: int = 0, d_count=None,
              max_pairs: int | None = None) -> GBuffer:
        """GaussianSplattingPass into a fresh G-buffer.  max_pairs None: m2s_splat (counts the pairs and sizes the scratch
        exactly; reports pairs and device time); else m2s_splat_enqueue with that pair capacity, then a synchronise and
        m2s_ctx_status (raises M2SError with M2S_E_CAPACITY if the quads touch more pairs: the G-buffer is then cleared)."""
        torch = _torch()
        dev = sorted_quads.device
        torch.cuda.current_stream(dev).synchronize()
        gb = GBuffer.empty(width, height, render_mode, dev)
        gb.survivors = count
        p = _abi.m2s_splat_params(width, height, render_mode, 0)
        g = gb.c_struct()
        dc = d_count.data_ptr() if d_count is not None else None
        if max_pairs is None:
            pairs, ms = C.c_uint64(0), C.c_float(0)
            check(lib().m2s_splat(self.handle, sorted_quads.data_ptr(), count, dc, C.byref(p), C.byref(g), C.byref(pairs), C.byref(ms)))
            gb.pairs, gb.device_ms = int(pairs.value), float(ms.value)
        else:
            check(lib().m2s_splat_enqueue(self.handle, sorted_quads.data_ptr(), count, dc, C.byref(p), C.byref(g), max_pairs, None))
            self.synchronize()
            check(lib().m2s_ctx_status(self.handle))
        return gb

    def render(self, records, count: int, layout: int, world_to_view, view_to_clip, model_to_world, width: int, height: int,
               std_dev: float, render_mode: int = 0, near_far=(0.01, 100.0)) -> GBuffer:
        """prepass -> sort -> splat on the context stream (GaussiansPrepass, RadixSortPass, GaussianSplattingPass): the
        records (e.g. ConvertOutput.data) seen by the camera at width x height.  The prepass's counter feeds the sort and
        the splat on the device; the only host round trip is the splat's pair count."""
        torch = _torch()
        dev = records.device
        torch.cuda.current_stream(dev).synchronize()
        n = max(1, count)
        quads = torch.empty(n * _abi.QUAD_BYTES, dtype=torch.uint8, device=dev)
        depths = torch.empty(n, dtype=torch.float32, device=dev)
        valid = torch.empty(1, dtype=torch.int32, device=dev)
        sorted_q = torch.empty(n * _abi.QUAD_BYTES, dtype=torch.uint8, device=dev)
        p = _abi.make_prepass_params(world_to_view, view_to_clip, model_to_world, (width, height), near_far, std_dev, render_mode,
                                     layout)
        L = lib()
        check(L.m2s_prepass_enqueue(self.handle, records.data_ptr(), count, None, C.byref(p), quads.data_ptr(), depths.data_ptr(),
                                    valid.data_ptr(), None))
        check(L.m2s_sort_quads_enqueue(self.handle, quads.data_ptr(), depths.data_ptr(), count, valid.data_ptr(),
                                       sorted_q.data_ptr(), None, None))
        gb = GBuffer.empty(width, height, render_mode, dev)
        sp = _abi.m2s_splat_params(width, height, render_mode, 0)
        g = gb.c_struct()
        pairs, ms = C.c_uint64(0), C.c_float(0)
        check(L.m2s_splat(self.handle, sorted_q.data_ptr(), count, valid.data_ptr(), C.byref(sp), C.byref(g), C.byref(pairs), C.byref(ms)))
        gb.pairs, gb.device_ms, gb.survivors = int(pairs.value), float(ms.value), int(valid.item())
        return gb

    def synchronize(self) -> None:
        """Waits for the context stream (through a device-wide synchronise: the stream is not exposed)."""
        _torch().cuda.synchronize(self.device)

    def convert_timed(self, dscene: DeviceScene, params: _abi.m2s_params, out, capacity: int):
        """One conversion with an event between the two kernels (they do not overlap): (raster_ms, fragment_ms)."""
        a, b = C.c_float(0), C.c_float(0)
        check(lib().m2s_convert_timed(self.handle, dscene.handle, C.byref(params), out.data_ptr(), capacity, C.byref(a), C.byref(b)))
        return float(a.value), float(b.value)

    def convert_host(self, scene: _abi.Scene, resolution: int, layout: int = _abi.LAYOUT_REF96,
                     gaussian_std: float = 0.65, max_gaussians: int = 0, flags: int = 0, capacity: int | None = None,
                     want_keys: bool = False, out: np.ndarray | None = None, c_scene=None):
        """Host buffers in, host buffers out (m2s_convert_host). Returns (records, keys, result)."""
        stride = _abi.STRIDES[layout]
        if capacity is None:
            if max_gaussians:
                capacity = max_gaussians
            elif flags & _abi.FLAG_UNCAPPED:
                capacity = 6 * resolution * resolution * max(1, len(scene.primitives))
            else:
                capacity = _abi.reference_capacity(resolution, len(scene.primitives))
        if out is None:
            out = np.empty(max(1, capacity) * stride, np.uint8)
        keys = np.empty(max(1, capacity), np.uint64) if want_keys else None
        cs, keep = c_scene if c_scene is not None else scene.c_struct()
        p = _abi.make_params(resolution, layout, gaussian_std, max_gaussians, flags)
        res = _abi.m2s_result()
        check(lib().m2s_convert_host(self.handle, C.byref(cs), C.byref(p), out.ctypes.data, capacity,
                                     keys.ctypes.data if want_keys else None, C.byref(res)),
              allow=(_abi.M2S_E_CAPACITY,))
        del keep
        rec = out[: res.written * stride].view(_abi.record_dtype(layout))
        return rec, (keys[: res.written] if want_keys else None), res

    # ---- outputs ----
    def ply_encode(self, ref96, count: int, fmt: int, scale_multiplier: float):
        """REF96 device tensor -> device tensor of .ply body rows."""
        torch = _torch()
        layout = _abi.PLY_FORMAT_LAYOUT.get(fmt, _abi.LAYOUT_PLY_STANDARD)
        rows = torch.empty(max(1, count) * _abi.STRIDES[layout], dtype=torch.uint8, device=ref96.device)
        check(lib().m2s_ply_encode(self.handle, ref96.data_ptr(), count, fmt, scale_multiplier, rows.data_ptr(), None))
        torch.cuda.synchronize(ref96.device)
        return rows[: count * _abi.STRIDES[layout]]

    def convert_file(self, glb_path: str, resolution: int, ply_path: str, gaussian_std: float = 0.65, fmt: int = 0):
        res = _abi.m2s_result()
        check(lib().m2s_convert_file(self.handle, glb_path.encode(), resolution, gaussian_std, fmt, ply_path.encode(),
                                     C.byref(res)), allow=(_abi.M2S_E_CAPACITY,))
        return res


def ply_header(fmt: int, count: int) -> bytes:
    buf = C.create_string_buffer(8192)
    n = lib().m2s_ply_header(fmt, count, buf, 8192)
    return buf.raw[:n]


def ply_write(path: str, ref96: np.ndarray, fmt: int, scale_multiplier: float) -> None:
    a = np.ascontiguousarray(ref96)
    count = a.nbytes // 96
    check(lib().m2s_ply_write(path.encode(), a.ctypes.data, count, fmt, scale_multiplier))


# ---------------------------------------------------------------------------------------------
# reference-shaped objects
# ---------------------------------------------------------------------------------------------
class RenderContext:
    """The fields of struct RenderContext (RenderContext.hpp:28-124) the conversion path touches."""

    def __init__(self, device: int = 0):
        self.ctx = Context(device)
        self.resolutionTarget = 520          # ImGuiUI.cpp:512 at the default quality 0.5
        self.gaussianStd = 0.65              # main.cpp:26
        self.scene: _abi.Scene | None = None       # dataMeshAndGlMesh (CPU side)
        self.deviceScene: DeviceScene | None = None  # ... (GPU side) + meshToTextureData
        self.gaussianBuffer = None           # SSBO: torch.uint8 device tensor of GaussianDataSSBO records
        self.numberOfGaussians = 0           # may exceed the buffer capacity (ConversionPass.cpp:56-59)
        self.lastResult: ConvertOutput | None = None


class SceneManager:
    def __init__(self, renderContext: RenderContext):
        self.renderContext = renderContext

    def setScene(self, scene: _abi.Scene) -> bool:
        rc = self.renderContext
        if rc.deviceScene is not None:
            rc.deviceScene.free()
        rc.scene = scene
        rc.deviceScene = rc.ctx.upload(scene)
        return True

    def loadModel(self, filePath: str, parentFolder: str = "") -> bool:
        """SceneManager::loadModel (SceneManager.cpp:22-35): parse .glb, bboxes, textures -> GPU."""
        from .gltf import load_glb  # noqa: WPS433
        try:
            return self.setScene(load_glb(filePath))
        except (OSError, ValueError) as e:  # the reference prints and returns false
            print(f"Failed to parse GLTF file: {filePath}: {e}")
            return False

    def exportPly(self, outputFile: str, exportFormat: int = 0) -> None:
        """SceneManager::exportPly (SceneManager.cpp:651-678): read back, scale by std/R, write."""
        rc = self.renderContext
        out = rc.lastResult
        if out is None:
            raise RuntimeError("exportPly before ConversionPass.execute")
        mult = np.float32(rc.gaussianStd) / np.float32(rc.resolutionTarget)
        ply_write(outputFile, out.numpy(), exportFormat, float(mult))


class ConversionPass:
    """IRenderPass for the conversion (RenderPass.hpp:10-28, ConversionPass.cpp:9-68)."""

    def __init__(self):
        self._enabled = False

    def isEnabled(self) -> bool:
        return self._enabled

    def setIsEnabled(self, isPassEnabled: bool) -> None:
        self._enabled = bool(isPassEnabled)

    def execute(self, renderContext: RenderContext) -> None:
        rc = renderContext
        if rc.deviceScene is None:
            raise RuntimeError("ConversionPass.execute: no model loaded")
        out = rc.ctx.convert(rc.deviceScene, rc.resolutionTarget, _abi.LAYOUT_REF96, rc.gaussianStd)
        rc.gaussianBuffer = out.data
        rc.numberOfGaussians = out.total
        rc.lastResult = out


__all__ = ["Context", "DeviceScene", "ConvertOutput", "GBuffer", "RenderContext", "SceneManager", "ConversionPass",
           "ply_header", "ply_write", "M2SError"]
