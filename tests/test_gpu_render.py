"""The viewer's depth sort and splatting pass on the GPU (SURVEY 8 f-5, f-6) against the oracle."""
import os

import numpy as np
import pytest

from oracle import render as roracle
from mesh2splat_b200 import _abi, synth
from mesh2splat_b200._abi import FLAG_UNCAPPED, LAYOUT_PACKED56, LAYOUT_REF96
from mesh2splat_b200._lib import M2SError
from mesh2splat_b200._lib import lib as lib_
from render_util import assert_gbuffer_equal, synthetic_quads

pytestmark = pytest.mark.gpu

# Tolerances of the real-data renders (non-overdraw targets).  The only source of difference is the ulp gap between CUDA's
# expf and glibc's (the rest of the arithmetic is the same fp32 operations, without contraction, on both sides), carried
# forward through the destination alpha.  If a run exceeds a bound, find the cause on one pixel: replay its fragment list in
# the oracle with g nudged by +-2 ulp.  Do not widen a bound without that evidence.
UNORM_TYPICAL, UNORM_MAX = 1, 4     # in 1/255 steps: <= 1 on >= 99.9 % of the pixels, <= 4 everywhere
HALF_TYPICAL_ULP, HALF_MAX_ULP = 2, 64   # in float16 ulps of the pixel's largest component: <= 2 on >= 99.9 %, <= 64 everywhere
TYPICAL_SHARE = 0.999


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _sorted_on_gpu(ctx, quads, depths, count=None, d_count=None):
    sq, order = ctx.sort_quads(_dev(quads.view(np.uint8).reshape(-1)) if len(quads) else _dev(np.zeros(96, np.uint8)),
                               _dev(depths) if len(depths) else _dev(np.zeros(1, np.float32)),
                               len(quads) if count is None else count, d_count=d_count)
    return sq, order


@pytest.mark.parametrize("n", [0, 1, 1023, 1025, 10_000_000])
def test_sort_is_numpys_stable_argsort_plus_gather(gpu_ctx, n):
    rng = np.random.default_rng(n)
    depths = -rng.integers(1, 200, n).astype(np.float32) * np.float32(0.25)   # a planar mesh facing the camera: many ties
    depths[: n // 7] = rng.uniform(-30, 5, n // 7)
    quads = np.zeros((n, 24), np.float32)
    quads[:, 0] = np.arange(n, dtype=np.float32)
    quads[:, 1:24] = rng.standard_normal((n, 23)).astype(np.float32) if n <= 100_000 else 1.0
    sq, order = _sorted_on_gpu(gpu_ctx, quads, depths)
    want = np.argsort(depths.view(np.uint32), kind="stable")
    assert np.array_equal(order.cpu().numpy().view(np.uint32), want)
    assert np.array_equal(sq.cpu().numpy().view(np.uint32), quads[want].view(np.uint32))


def test_sort_with_a_device_count(gpu_ctx):
    import torch
    rng = np.random.default_rng(3)
    n, m = 5000, 3217
    depths = -rng.integers(1, 50, n).astype(np.float32)
    quads = rng.standard_normal((n, 24)).astype(np.float32)
    dc = torch.tensor([m], dtype=torch.int32, device="cuda")
    sq, order = _sorted_on_gpu(gpu_ctx, quads, depths, d_count=dc)
    want = np.argsort(depths[:m].view(np.uint32), kind="stable")
    assert np.array_equal(order[:m].cpu().numpy().view(np.uint32), want)
    assert np.array_equal(sq[:m].cpu().numpy(), quads[want])


def _bench_scene_output(ctx, layout, R=512):
    scene = synth.helmet_standin(2048)
    ds = ctx.upload(scene)
    out = ctx.convert(ds, R, layout, flags=FLAG_UNCAPPED, capacity=6 * R * R)
    ds.free()
    return out


def _cameras():
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_prepass_vectors.npz"))
    return [(g[f"view{i}"], g[f"proj{i}"]) for i in range(int(g["ncases"]))]


def test_sort_on_the_bench_scene_survivors(gpu_ctx):
    out = _bench_scene_output(gpu_ctx, LAYOUT_REF96)
    V, P = _cameras()[0]
    quads, depths = gpu_ctx.prepass(out.data, out.written, LAYOUT_REF96, V, P, np.eye(4, dtype=np.float32).ravel(), (1280, 720),
                                    (0.01, 100.0), 0.65 / 512, 0)
    assert len(quads) > 10_000
    sq, order = _sorted_on_gpu(gpu_ctx, quads, depths)
    want = np.argsort(depths.view(np.uint32), kind="stable")
    assert np.array_equal(order.cpu().numpy().view(np.uint32), want)
    assert np.array_equal(sq.cpu().numpy().view(np.uint32), quads[want].view(np.uint32))


@pytest.mark.parametrize("size", [(1283, 719), (16, 16), (1, 1), (4096, 4096)])
@pytest.mark.parametrize("mode", [0, 4])
def test_splat_synthetic_quads_bit_identical_to_the_oracle(gpu_ctx, size, mode):
    """conic = 0 (g = 1 exactly): every target bit-identical to the oracle.  Quads from sub-pixel to the 1024-pixel axis
    limit, rotated, straddling tiles and screen edges, equal depths, and a stack about 1000 deep."""
    W, H = size
    if (W, H) == (4096, 4096) and mode == 4:
        pytest.skip("4096 x 4096 runs once, in mode 0")
    q = synthetic_quads(W, H, seed=W * 7 + H + mode, n=300 if W > 16 else 60, deep=1000)
    gb = gpu_ctx.splat(_dev(q), len(q), W, H, mode)
    want = roracle.splat(q, W, H, mode)
    assert_gbuffer_equal(gb.numpy(), want)
    assert np.count_nonzero(want["albedo"][..., 3]) > 0


def _ulp16(x):
    """Spacing of float16 at |x|."""
    a = np.abs(x.astype(np.float32))
    e = np.floor(np.log2(np.maximum(a, np.float32(2.0 ** -14))))
    return np.float32(2.0) ** (e - 10)


def _assert_close(got: dict, want: dict, tag):
    for name, kind in _abi.GBUFFER_TARGETS:
        g, w = got[name], want[name]
        if kind == "u8":
            d = np.abs(g.astype(np.int32) - w.astype(np.int32)).max(axis=-1)
            assert d.max() <= UNORM_MAX, (tag, name, int(d.max()))
            assert np.mean(d <= UNORM_TYPICAL) >= TYPICAL_SHARE, (tag, name, float(np.mean(d <= UNORM_TYPICAL)))
        else:
            gf, wf = g.astype(np.float32), w.astype(np.float32)
            assert np.array_equal(np.isfinite(gf), np.isfinite(wf)), (tag, name)
            fin = np.isfinite(wf)
            # ulps of the pixel's largest component: a component that cancels to near 0 (world positions either side of
            # the origin) is compared on the scale of the sums that produced it
            scale = np.where(fin, np.abs(wf), 0).max(axis=-1, keepdims=True)
            d = np.where(fin, np.abs(gf - wf) / _ulp16(scale), 0).max(axis=-1)
            assert d.max() <= HALF_MAX_ULP, (tag, name, float(d.max()))
            assert np.mean(d <= HALF_TYPICAL_ULP) >= TYPICAL_SHARE, (tag, name, float(np.mean(d <= HALF_TYPICAL_ULP)))


@pytest.mark.parametrize("layout", [LAYOUT_REF96, LAYOUT_PACKED56])
def test_render_the_bench_scene_against_the_oracle(gpu_ctx, layout):
    """convert -> prepass -> sort -> splat on the device for the five golden cameras at 1280 x 720.  Ties in depth make the
    render depend on the prepass arrival order, so the oracle splats the GPU's own sorted quads (the sort is checked above).
    Overdraw albedo is exact; the other targets within the tolerances at the top of this file."""
    out = _bench_scene_output(gpu_ctx, layout)
    W, H = 1280, 720
    M = np.eye(4, dtype=np.float32).ravel()
    for i, (V, P) in enumerate(_cameras()):
        for mode in (0, 4) if i < 2 else (0,):
            gb = gpu_ctx.render(out.data, out.written, layout, V, P, M, W, H, 0.65 / 512, mode)
            assert gb.survivors > 1000 and gb.pairs >= gb.survivors // 4
            # the same chain step by step: the sorted quads the G-buffer was made from
            qn, dn = gpu_ctx.prepass(out.data, out.written, layout, V, P, M, (W, H), (0.01, 100.0), 0.65 / 512, mode)
            assert len(qn) == gb.survivors
            sq, _ = _sorted_on_gpu(gpu_ctx, qn, dn)
            step = gpu_ctx.splat(sq, len(qn), W, H, mode)
            want = roracle.splat(sq.cpu().numpy(), W, H, mode)
            got = step.numpy()
            if mode == 4:
                assert np.array_equal(got["albedo"], want["albedo"]), i
            _assert_close(got, want, (layout, i, mode))


def test_enqueue_chain_equals_the_synchronous_calls_and_capacity_is_reported(gpu_ctx):
    """prepass -> sort -> splat enqueued on one stream with device counts only (Context.render) equals the step-by-step
    synchronous calls, byte for byte when the prepass order matches; a max_pairs below the pair count leaves the G-buffer
    cleared and m2s_ctx_status reports M2S_E_CAPACITY."""
    q = synthetic_quads(256, 128, seed=11, n=200, deep=50)
    d = _dev(q)
    a = gpu_ctx.splat(d, len(q), 256, 128, 0)
    b = gpu_ctx.splat(d, len(q), 256, 128, 0, max_pairs=a.pairs)
    assert_gbuffer_equal(a.numpy(), b.numpy())
    with pytest.raises(M2SError) as e:
        gpu_ctx.splat(d, len(q), 256, 128, 0, max_pairs=a.pairs - 1)
    assert e.value.status == _abi.M2S_E_CAPACITY
    import ctypes as C
    from mesh2splat_b200.api import GBuffer
    gb = GBuffer.empty(256, 128, 0, d.device)
    for t in (gb.position, gb.normal, gb.albedo, gb.depth, gb.metallic_roughness):
        t.fill_(7)
    import torch
    torch.cuda.synchronize()
    p, g = _abi.m2s_splat_params(256, 128, 0, 0), gb.c_struct()
    assert lib_().m2s_splat_enqueue(gpu_ctx.handle, d.data_ptr(), len(q), None, C.byref(p), C.byref(g), a.pairs // 2, None) == _abi.M2S_OK
    gpu_ctx.synchronize()
    assert lib_().m2s_ctx_status(gpu_ctx.handle) == _abi.M2S_E_CAPACITY
    for name, arr in gb.numpy().items():
        assert not np.any(arr), name   # left cleared
    from mesh2splat_b200._lib import lib
    assert lib().m2s_ctx_status(gpu_ctx.handle) == _abi.M2S_OK   # reading the condition cleared it
    ample = gpu_ctx.splat(d, len(q), 256, 128, 0, max_pairs=10 ** 6)   # more capacity than needed: the same image
    assert_gbuffer_equal(a.numpy(), ample.numpy())

    # the device-count chain on a real scene: Context.render against prepass + sort + splat called one by one
    out = _bench_scene_output(gpu_ctx, LAYOUT_PACKED56, R=256)
    V, P = _cameras()[3]
    M = np.eye(4, dtype=np.float32).ravel()
    chain = gpu_ctx.render(out.data, out.written, LAYOUT_PACKED56, V, P, M, 640, 360, 1.0, 0)
    qn, dn = gpu_ctx.prepass(out.data, out.written, LAYOUT_PACKED56, V, P, M, (640, 360), (0.01, 100.0), 1.0, 0)
    assert len(qn) == chain.survivors
    sq, _ = _sorted_on_gpu(gpu_ctx, qn, dn)
    step = gpu_ctx.splat(sq, len(qn), 640, 360, 0)
    # both are exact functions of the sorted quads; the prepass order may differ between runs only among equal depths
    _assert_close(chain.numpy(), step.numpy(), "chain")
    assert chain.pairs == step.pairs
