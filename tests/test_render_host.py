"""The viewer's depth sort and splatting pass (SURVEY 8 f-5, f-6) on the CPU: the oracle against the reference's own shaders,
known-answer tests of the rasterisation and the blend, and the C ABI's argument checks (no GPU needed)."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import render as roracle
from mesh2splat_b200 import _abi
from render_util import quad

HERE = os.path.dirname(os.path.abspath(__file__))


def _golden():
    return np.load(os.path.join(HERE, "golden", "ref_splat_vectors.npz"))


def test_splat_oracle_matches_reference_shaders_bit_for_bit():
    """tests/golden/ref_splat_vectors.npz holds gaussianSplattingVS/PS.glsl's own corner positions and outputs (made by
    tests/golden/make_golden_splat.py from the reference's sources) for the prepass golden quads: both sides are C on the
    same libm expf, so they agree bit for bit, in and far outside each quad, in modes 0 and 4."""
    g = _golden()
    n = 0
    for i in range(int(g["ncases"])):
        W, H = (float(v) for v in g[f"size{i}"])
        for k, q in enumerate(g[f"quads{i}"]):
            assert np.array_equal(roracle.splat_vertex(q, W, H).view(np.uint32), g[f"corners{i}"][k].view(np.uint32))
            for m, mode in enumerate(g["modes"]):
                got = roracle.splat_fragments(q, W, H, int(mode), g[f"frags{i}"][k])
                assert np.array_equal(got.view(np.uint32), g[f"out{i}"][m, k].view(np.uint32)), (i, k, int(mode))
                n += 1
    assert n >= 300


@pytest.mark.parametrize("n,levels", [(1, 5), (1000, 3), (5000, 20000), (20000, 7)])
def test_oracle_sort_is_the_stable_sort_of_the_key_bits(n, levels):
    rng = np.random.default_rng(n)
    d = -rng.integers(1, levels + 1, n).astype(np.float32) * np.float32(0.37)   # many equal depths
    d[: n // 10] = rng.uniform(-50, 50, n // 10)                               # and some of either sign
    want = np.argsort(d.view(np.uint32), kind="stable")
    assert np.array_equal(roracle.sort_quads(d), want)


def _covered(W, H, q, mode=4):
    return roracle.splat(q[None] if q.ndim == 1 else q, W, H, mode)


def test_axis_aligned_quad_covers_the_expected_pixel_rectangle():
    W, H = 40, 30
    q = quad(10.0, 12.0, 4.0, 0.0, 0.0, 3.0, W, H)   # window x in [6, 14], y in [9, 15]: pixel centres 6..13, 9..14
    gb = _covered(W, H, q, 0)
    a = gb["albedo"][..., 3]
    ys, xs = np.nonzero(a)
    assert (xs.min(), xs.max(), ys.min(), ys.max()) == (6, 13, 9, 14)
    assert np.count_nonzero(a) == 8 * 6


def test_rotated_quad_shared_diagonal_is_owned_once():
    """Mode 4 (ONE, ONE) counts fragments: one fragment gives albedo (3, 1, 0, 3) (rint(.01 * 255), rint(.005 * 255))."""
    W, H = 64, 64
    for ang in np.linspace(0.05, 1.5, 7):
        r = 13.3
        q = quad(31.7, 30.2, r * np.cos(ang), r * np.sin(ang), -0.6 * r * np.sin(ang), 0.6 * r * np.cos(ang), W, H)
        a = _covered(W, H, q, 4)["albedo"]
        hit = a[..., 3] > 0
        assert hit.sum() > 100
        assert np.all(a[hit] == [3, 1, 0, 3]), np.unique(a[hit].reshape(-1, 4), axis=0)


@pytest.mark.parametrize("k", [1, 2, 5, 40, 84, 85, 86, 300])
def test_overdraw_unorm_steps(k):
    """k fragments in mode 4 give min(255, 3k) and min(255, k): the target is quantised after every fragment."""
    W, H = 8, 8
    q = np.stack([quad(4.0, 4.0, 2.0, 0.0, 0.0, 2.0, W, H)] * k)
    a = _covered(W, H, q, 4)["albedo"][4, 4]
    assert a.tolist() == [min(255, 3 * k), min(255, k), 0, min(255, 3 * k)]


def test_equal_depth_quads_compose_in_arrival_order():
    W, H = 16, 16
    red = quad(8.0, 8.0, 6.0, 0.0, 0.0, 6.0, W, H, color=(1.0, 0.0, 0.0, 0.6))
    blue = quad(8.0, 8.0, 6.0, 0.0, 0.0, 6.0, W, H, color=(0.0, 0.0, 1.0, 0.6))
    rb = _covered(W, H, np.stack([red, blue]), 0)["albedo"][8, 8]
    br = _covered(W, H, np.stack([blue, red]), 0)["albedo"][8, 8]
    # first: rint(0.6 * 255) = 153; the second adds 0.6 * (1 - 153/255)
    assert rb[0] == 153 and rb[2] == 61 and br[2] == 153 and br[0] == 61
    assert rb[3] == br[3] == 214


def test_offscreen_quads_are_clipped_and_nan_quads_produce_nothing():
    W, H = 32, 32
    off = [quad(-20.0, 10.0, 5.0, 0.0, 0.0, 5.0, W, H), quad(10.0, 50.0, 5.0, 0.0, 0.0, 5.0, W, H)]
    nan = quad(10.0, 10.0, 5.0, 0.0, 0.0, 5.0, W, H)
    nan[4:8] = np.nan   # what the prepass writes for a perfectly round splat (0/0 direction)
    gb = _covered(W, H, np.stack(off + [nan]), 0)
    for name in gb:
        assert not np.any(gb[name]), name
    edge = _covered(W, H, quad(-2.0, 3.0, 5.0, 0.0, 0.0, 2.0, W, H), 4)["albedo"][..., 3]
    ys, xs = np.nonzero(edge)
    assert xs.min() == 0 and xs.max() == 2 and (ys.min(), ys.max()) == (1, 4)


def test_render_entry_points_reject_bad_arguments_without_a_gpu():
    """m2s_sort_quads* / m2s_splat*: M2S_E_INVALID before any CUDA call; struct sizes as include/m2s.h states."""
    from mesh2splat_b200._lib import lib
    L = lib()
    assert C.sizeof(_abi.m2s_splat_params) == 16 and C.sizeof(_abi.m2s_gbuffer) == 5 * 8
    fake = C.c_void_p(0x1000)   # never dereferenced: validation fails first
    buf = 0x100000
    gb = _abi.m2s_gbuffer(buf, buf, buf, buf, buf)
    ok = _abi.m2s_splat_params(64, 64, 0, 0)
    assert L.m2s_sort_quads(None, None, None, 0, None, None, None) == _abi.M2S_E_INVALID
    assert L.m2s_sort_quads_enqueue(None, None, None, 0, None, None, None, None) == _abi.M2S_E_INVALID
    assert L.m2s_sort_quads_enqueue(fake, None, None, 10, None, None, None, None) == _abi.M2S_E_INVALID
    assert L.m2s_sort_quads_enqueue(fake, buf, buf, 1 << 32, None, buf, None, None) == _abi.M2S_E_INVALID
    assert L.m2s_sort_quads_enqueue(fake, buf + 8, buf, 10, None, buf, None, None) == _abi.M2S_E_INVALID
    assert L.m2s_splat(None, buf, 1, None, C.byref(ok), C.byref(gb), None, None) == _abi.M2S_E_INVALID
    assert L.m2s_splat_enqueue(fake, buf, 1, None, None, C.byref(gb), 10, None) == _abi.M2S_E_INVALID
    assert L.m2s_splat_enqueue(fake, buf, 1, None, C.byref(ok), None, 10, None) == _abi.M2S_E_INVALID
    assert L.m2s_splat_enqueue(fake, None, 1, None, C.byref(ok), C.byref(gb), 10, None) == _abi.M2S_E_INVALID
    for w, h, mode in ((0, 64, 0), (64, 0, 0), (4097, 64, 0), (64, 4097, 0), (64, 64, 3), (64, 64, 7)):
        p = _abi.m2s_splat_params(w, h, mode, 0)
        assert L.m2s_splat_enqueue(fake, buf, 1, None, C.byref(p), C.byref(gb), 10, None) == _abi.M2S_E_INVALID, (w, h, mode)
        assert L.m2s_splat(fake, buf, 1, None, C.byref(p), C.byref(gb), None, None) == _abi.M2S_E_INVALID, (w, h, mode)
    assert L.m2s_splat_enqueue(fake, buf, 1 << 32, None, C.byref(ok), C.byref(gb), 10, None) == _abi.M2S_E_INVALID
    for field in ("position", "normal", "albedo", "depth", "metallic_roughness"):
        bad = _abi.m2s_gbuffer(buf, buf, buf, buf, buf)
        setattr(bad, field, buf + 4)
        assert L.m2s_splat_enqueue(fake, buf, 1, None, C.byref(ok), C.byref(bad), 10, None) == _abi.M2S_E_INVALID, field
        setattr(bad, field, None)
        assert L.m2s_splat_enqueue(fake, buf, 1, None, C.byref(ok), C.byref(bad), 10, None) == _abi.M2S_E_INVALID, field
    assert L.m2s_splat_enqueue(fake, buf + 8, 1, None, C.byref(ok), C.byref(gb), 10, None) == _abi.M2S_E_INVALID
