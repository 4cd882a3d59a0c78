"""CPU tests: pin the oracle against (a) golden vectors produced by the reference's own GLSL,
(b) what the reference build made of the inputs of the *live_reference* tests (tests/golden/ref_live_vectors.npz,
tests/golden/make_golden_live.py), (c) the analytic KATs of SURVEY.md 8c."""
from __future__ import annotations

import os

import numpy as np
import pytest

import oracle
from mesh2splat_b200 import _abi, synth
from mesh2splat_b200._abi import LAYOUT_PACKED56, LAYOUT_REF96, Primitive, Scene

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_shader_vectors.npz")
LIVE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_live_vectors.npz")


@pytest.fixture(scope="module")
def golden():
    return np.load(GOLDEN)


@pytest.fixture(scope="module")
def live():
    return np.load(LIVE)


def _same(a, b):  # bit-equal, NaN == NaN
    a = np.asarray(a, np.float32); b = np.asarray(b, np.float32)
    return np.array_equal(a.view(np.uint32), b.view(np.uint32)) or np.array_equal(a, b, equal_nan=True)


def test_triangle_stage_matches_reference_gs_golden(golden):
    """oracle per-triangle stage == converterGS.glsl main, bit for bit, on 256 seeded triangles."""
    n = len(golden["gs_tris"])
    for i in range(n):
        s = oracle.triangle_setup(golden["gs_tris"][i], golden["gs_bmin"][i], golden["gs_bmax"][i], 512)
        ouv = np.array(s.ouv, np.float32)
        ndc = ouv * np.float32(2.0) - np.float32(1.0)
        assert _same(ndc, golden["gs_glpos"][i][:, :2]), f"gl_Position.xy differs for triangle {i}"
        assert np.all(golden["gs_glpos"][i][:, 2] == 0) and np.all(golden["gs_glpos"][i][:, 3] == 1)
        assert _same(np.array(s.scale, np.float32), golden["gs_scale"][i]), f"Scale differs for triangle {i}"
        assert _same(np.array(s.quat, np.float32), golden["gs_quat"][i]), f"Quaternion differs for triangle {i}"


def test_fragment_stage_matches_reference_fs_golden(golden):
    """oracle per-fragment stage == converterFS.glsl main (incl. the overflow discard)."""
    m = len(golden["fs_varyings"])
    seen_discard = False
    for i in range(m):
        v = golden["fs_varyings"][i]
        tx = golden["fs_texels"][i]
        start, maxg = int(golden["fs_counter_start"][i]), int(golden["fs_max_gaussians"][i])
        assert golden["fs_counter_after"][i] == start + 1          # the counter always advances (:46)
        written = start < maxg                                       # :49-51
        assert bool(golden["fs_written"][i]) == written
        if not written:
            seen_discard = True
            continue
        rec = oracle.fragment(v[0:3], v[3:6], v[6:10], v[12:15], v[15:19], tx[0], tx[1], tx[2],
                              int(golden["fs_flags"][i]), golden["fs_factor"][i])
        assert _same(rec, golden["fs_rec"][i]), f"record differs for fragment {i}"
    assert seen_discard


def test_triangle_stage_matches_live_reference_build(live):
    """500 triangles of a random soup (one bbox around all of them): converterGS.glsl's gl_Position.xy, Scale and
    Quaternion as the reference build computed them, bit for bit."""
    mn, mx = live["gs_bmin"], live["gs_bmax"]
    for i, t in enumerate(live["gs_tris"]):
        s = oracle.triangle_setup(t, mn, mx, 256)
        assert _same(np.array(s.ouv, np.float32) * np.float32(2) - np.float32(1), live["gs_glpos_xy"][i]), i
        assert _same(np.array(s.scale, np.float32), live["gs_scale"][i]) and _same(np.array(s.quat, np.float32), live["gs_quat"][i]), i


# ---- analytic KATs (SURVEY 8c) --------------------------------------------------------------------
def test_kat_unit_quad():
    s = synth.unit_quad()
    rec, keys, total = oracle.convert(s, 64)
    assert total == 4096 and len(rec) == 4096
    tri = (keys >> np.uint64(24)).astype(int)
    assert np.bincount(tri).tolist() == [2080, 2016]
    px = (keys & np.uint64(0xfff)).astype(np.float32); py = ((keys >> np.uint64(12)) & np.uint64(0xfff)).astype(np.float32)
    assert np.array_equal(rec["position"][:, 0], (px + 0.5) / 64) and np.array_equal(rec["position"][:, 1], (py + 0.5) / 64)
    assert len(set(zip(px.tolist(), py.tolist()))) == 4096       # every pixel centre exactly once
    diag = px == py
    assert np.all(tri[diag] == 0)                                # shared diagonal: left edge of triangle 0 owns it
    np.testing.assert_allclose(rec["rotation"][tri == 0][0], [0, 0.9238795, 0.38268343, 0], atol=1e-7)
    np.testing.assert_allclose(rec["rotation"][tri == 1][0], [0.9238795, 0, 0, 0.38268343], atol=1e-7)
    assert np.all(rec["scale"] == np.array([1, 1, 1e-7, 0], np.float32))
    assert np.all(rec["pbr"] == np.array([0.1, 0.5, 0, 1], np.float32))
    assert np.all(rec["color"] == 1) and np.all(rec["normal"] == np.array([0, 0, 1, 0], np.float32))
    # exported values (parsers.cpp:484-499)
    p56, _, _ = oracle.convert(s, 64, LAYOUT_PACKED56)
    np.testing.assert_allclose(p56["log_scale"][0], np.log(np.array([0.65 / 64, 0.65 / 64, 1e-7 * 0.65 / 64])), rtol=1e-6)
    np.testing.assert_allclose(p56["sh0"][0], (1 - 0.5) / 0.28209479177387814, rtol=1e-6)
    assert np.all(np.isposinf(p56["opacity"]))                   # alpha 1 -> +inf in fp32 (utils.hpp:270)


def test_kat_box_face_axes_and_partial_grid():
    s = synth.box((1.0, 2.0, 3.0))
    rec, keys, total = oracle.convert(s, 60)
    tri = (keys >> np.uint64(24)).astype(int)
    # faces: z- z+ (X x Y, range max(1,2)=2), y- y+ (X x Z, range 3), x- x+ (Y x Z, range 3)
    n = np.bincount(tri, minlength=12)
    assert n[0] + n[1] == 30 * 60 and n[2] + n[3] == n[0] + n[1]            # 1x2 on a range-2 grid: 30 x 60 px
    assert n[4] + n[5] == 20 * 60 and n[8] + n[9] == 40 * 60                # 1x3 / 2x3 on a range-3 grid
    assert total == 2 * (1800 + 1200 + 2400)
    # scale = range / 1 in the projection plane (|J_u| = max range), e.g. z faces: 2
    z = rec[tri < 4]
    np.testing.assert_allclose(z["scale"][:, :2], 2.0, rtol=1e-6)


def test_kat_tilted_triangle_scale():
    # triangle in the plane z = x (tilted 45 deg about y), Y-dominant? no: normal (1,0,-1)/sqrt2 -> |nx|==|nz| -> falls to Z
    tri = np.zeros((1, 36), np.float32)
    v = tri.reshape(3, 12)
    v[0, :3] = (0, 0, 0); v[1, :3] = (1, 0, 1); v[2, :3] = (0, 1, 0)
    s = Scene(tri)
    s.primitives[0].bbox_min = (0.0, 0.0, 0.0); s.primitives[0].bbox_max = (1.0, 1.0, 1.0)
    st = oracle.triangle_setup(tri[0], (0, 0, 0), (1, 1, 1), 64)
    assert st.axis == 2                                              # tie |nx| == |nz|: not X (strict >), not Y -> Z
    np.testing.assert_allclose(st.scale[0], np.sqrt(2.0), rtol=1e-6)  # |J_u| = range * sqrt 2
    np.testing.assert_allclose(st.scale[1], 1.0, rtol=1e-6)


def test_kat_degenerate_projection_emits_nothing():
    tri = np.zeros((1, 36), np.float32)
    v = tri.reshape(3, 12)
    v[0, :3] = (0.1, 0.1, 0.1); v[1, :3] = (0.5, 0.5, 0.1); v[2, :3] = (0.9, 0.9, 0.1)   # collinear
    st = oracle.triangle_setup(tri[0], (0, 0, 0), (1, 1, 1), 64)
    assert st.area2 == 0 and st.scale[0] == 0 and st.scale[1] == 0
    s = Scene(tri); s.primitives[0].bbox_max = (1.0, 1.0, 1.0)
    assert oracle.convert(s, 64)[2] == 0


def test_kat_capacity_overflow_and_reference_rule():
    s = synth.unit_quad()
    rec, keys, total = oracle.convert(s, 64, max_gaussians=100)
    assert total == 4096 and len(rec) == 100                         # counter keeps counting (ConversionPass.cpp:56-59)
    assert _abi.reference_capacity(64, 1) == 24576 and _abi.reference_capacity(2048, 1) == 7_000_000
    assert _abi.reference_capacity(1024, 100) == 7_000_000


def test_sampler_kats():
    img = np.zeros((4, 4, 4), np.uint8)
    img[..., 0] = np.arange(16).reshape(4, 4) * 16
    # texel centres reproduce the texel; REPEAT wraps
    for y in range(4):
        for x in range(4):
            c = oracle.sample(img, (x + 0.5) / 4, (y + 0.5) / 4, -1.0)
            assert abs(c[0] - np.float32(img[y, x, 0]) / np.float32(255)) < 1e-7
    a = oracle.sample(img, 0.125, 0.125, 0.0); b = oracle.sample(img, 1.125, -0.875, 0.0)
    assert np.array_equal(a, b)
    # u = 0: halfway between last and first column (wrap)
    c = oracle.sample(img, 0.0, 0.125, 0.0)
    assert abs(c[0] - (img[0, 3, 0] / 255 + img[0, 0, 0] / 255) / 2) < 1e-6
    # mip chain: 4x4 -> 2x2 -> 1x1, box with round-half-up; lambda beyond q clamps to the last level
    l1 = oracle.mip_level(img, 1)
    assert l1[0, 0, 0] == (0 + 16 + 64 + 80 + 2) // 4 and oracle.mip_count(4, 4) == 3
    top = oracle.sample(img, 0.3, 0.7, 9.0)
    assert abs(top[0] - np.float32(oracle.mip_level(img, 2)[0, 0, 0]) / np.float32(255)) < 1e-7
    # trilinear halfway between level 0 and 1
    h = oracle.sample(img, 0.375, 0.375, 0.5)
    l0v = oracle.sample(img, 0.375, 0.375, 0.0)[0]
    l1v = np.float32(l1[0, 0, 0]) / 255 * 0.5625 + np.float32(l1[0, 1, 0]) / 255 * 0.1875 + np.float32(l1[1, 0, 0]) / 255 * 0.1875 + np.float32(l1[1, 1, 0]) / 255 * 0.0625
    assert abs(h[0] - (l0v + l1v) / 2) < 1e-6
    assert oracle.mip_count(2048, 2048) == 5 and oracle.mip_count(1, 1) == 1 and oracle.mip_count(100, 37) == 5


def test_cumulative_bbox_rule():
    a = synth.displaced_sphere(8, 4, seed=1, center=(0, 0, 0))
    b = synth.displaced_sphere(8, 4, seed=2, center=(5, 0, 0))
    s = Scene(np.concatenate([a, b]), [Primitive(0, len(a)), Primitive(len(a), len(b))])
    s.compute_bboxes(cumulative=True)
    assert s.primitives[1].bbox_min[0] == s.primitives[0].bbox_min[0]   # union of 0..k (SceneManager.cpp:476-527)
    assert s.primitives[1].bbox_max[0] > s.primitives[0].bbox_max[0]
    s2 = Scene(np.concatenate([a, b]), [Primitive(0, len(a)), Primitive(len(a), len(b))])
    s2.compute_bboxes(cumulative=False)
    assert s2.primitives[1].bbox_min[0] > 3.0


def test_oracle_thread_count_does_not_change_output():
    tri = synth.displaced_sphere(24, 12, seed=5)
    s = Scene(tri, [Primitive(0, len(tri), (1, 1, 1, 1), 0, 1, 2)], synth.make_material_textures(64, 3))
    s.compute_bboxes()
    r1, k1, t1 = oracle.convert(s, 96, threads=1)
    r8, k8, t8 = oracle.convert(s, 96, threads=8)
    assert t1 == t8 and np.array_equal(k1, k8) and r1.tobytes() == r8.tobytes()


@pytest.mark.parametrize("R,n", [(97, 300), (256, 5000)])
def test_watertight_tiling_covers_every_pixel_exactly_once(R, n):
    """GL 4.6 14.6.1: of two polygons sharing an edge exactly one produces the fragment (top-left rule here).
    A Delaunay tiling of the unit square must therefore emit each of the R*R pixel centres exactly once."""
    from util import planar_triangulation
    s = planar_triangulation(n, seed=R)
    rec, keys, total = oracle.convert(s, R, _abi.LAYOUT_REF96, flags=_abi.FLAG_UNCAPPED)
    assert total == R * R
    pix = keys & np.uint64(0xFFFFFF)
    assert len(np.unique(pix)) == R * R


# ---- export arithmetic pinned to the reference's own writer ---------------------------------------------------
def _ply_golden():
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_ply_vectors.npz"))


@pytest.mark.parametrize("fmt", [0, 1, 2, 9])
def test_ply_bytes_match_reference_savePlyVector_golden(fmt):
    """tests/golden/ref_ply_vectors.npz holds the files the REFERENCE's parsers::savePlyVector wrote for 200
    records (parsers.cpp + utils.cpp compiled from /root/reference by oracle/build.py; make_golden.py).  The
    restatement must reproduce them byte for byte — header, field order, SH0, logit (+inf), log-scale, the
    compressed format's octahedral normal and byte packing, and the default branch for unknown formats."""
    g = _ply_golden()
    rec = g["records"].view(_abi.record_dtype(LAYOUT_REF96)).reshape(-1)
    got = oracle.ply_bytes(rec, fmt, float(g["scale_multiplier"]))
    want = g[f"ply_format_{fmt}"].tobytes()
    assert len(got) == len(want)
    assert got == want


def test_ply_bytes_match_live_reference_writer(live):
    """Same check on other records (uniform random, small scales, some alpha 1) and another multiplier: the files the
    reference's savePlyVector wrote for them, byte for byte."""
    rec = live["ply_records"]
    mult = float(live["ply_scale_multiplier"])
    for fmt in (0, 1, 2):
        assert live[f"ply_format_{fmt}"].tobytes() == oracle.ply_bytes(rec.view(_abi.record_dtype(LAYOUT_REF96)).reshape(-1), fmt, mult)


def test_loader_matches_live_reference_parser(tmp_path, live):
    """Random node transforms / attribute combinations (util.loader_transform_cases) through m2s_glb_load: the
    triangle data the reference's own parser produced for the same files, bit for bit."""
    from test_abi_host import _make_glb
    from util import loader_transform_cases
    from mesh2splat_b200.gltf import load_glb
    cases = loader_transform_cases()
    counts = live["loader_face_counts"]
    assert len(counts) == len(cases)
    wants = np.split(live["loader_faces"], np.cumsum(counts)[:-1])
    for k, kw in enumerate(cases):
        p = tmp_path / f"c{k}.glb"
        _make_glb(str(p), **kw)
        s = load_glb(str(p))
        assert wants[k].shape == s.triangles.shape and np.array_equal(wants[k].view(np.uint32), s.triangles.view(np.uint32)), k


def test_loader_matches_live_reference_parser_on_random_scene_graphs(tmp_path, live):
    """Differential test on 120 random multi-mesh .glb files (util.make_complex_glb): nested matrix / TRS nodes,
    instanced meshes, shared images, every index type, skipped primitives, two scenes — m2s_glb_load vs what the
    reference's own parser made of them: identical triangles (bitwise), names, base colours, texture slots and texels
    (triangles and texels through their recorded SHA-256 digests)."""
    from util import array_digest, make_complex_glb
    from mesh2splat_b200.gltf import load_glb
    seeds = [int(x) for x in live["graph_seeds"]]
    first = np.concatenate([[0], np.cumsum(live["graph_mesh_counts"])])
    compared = 0
    for seed in range(5000, 5120):
        p = tmp_path / "g.glb"
        make_complex_glb(str(p), seed)
        if seed not in seeds:   # the reference rejects the file or finds no mesh in it
            continue
        j = seeds.index(seed)
        m0, m1 = int(first[j]), int(first[j + 1])
        s = load_glb(str(p))
        assert array_digest([s.triangles]) == live["graph_faces_sha256"][j], seed
        assert [str(x) for x in live["graph_mesh_names"][m0:m1]] == [q.name for q in s.primitives], seed
        texels = []
        for q, bc, present in zip(s.primitives, live["graph_base_color"][m0:m1], live["graph_tex_present"][m0:m1]):
            assert np.array_equal(bc, np.asarray(q.base_color_factor, np.float32)), seed
            for which, idx in ((0, q.albedo_texture), (1, q.normal_texture), (2, q.metallic_roughness_texture)):
                assert bool(present[which]) == (idx >= 0), (seed, q.name, which)
                if idx >= 0:
                    texels.append(s.textures[idx])
        assert array_digest(texels) == live["graph_texels_sha256"][j], seed
        compared += 1
    assert compared >= 100


# ---- viewer prepass (SURVEY 8 f-4): the C restatement against the reference's own compute shader --------------------
def _prepass_golden():
    import os
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_prepass_vectors.npz"))
    for i in range(int(g["ncases"])):
        p = g[f"params{i}"]
        yield dict(gaussians=g[f"g{i}"], view=g[f"view{i}"], proj=g[f"proj{i}"], model=g[f"model{i}"], resolution=(float(p[0]), float(p[1])),
                   near_far=(float(p[2]), float(p[3])), std_dev=float(p[4]), render_mode=int(p[5]), fmt=int(p[6]), quads=g[f"quads{i}"], depths=g[f"depths{i}"])


def test_prepass_oracle_matches_reference_shader_golden_vectors():
    """tests/golden/ref_prepass_vectors.npz holds gaussianSplattingPrepassCS.glsl's own outputs (made by
    tests/golden/make_golden_prepass.py from /root/reference): same survivors in the same order, values as
    util.assert_prepass_match states."""
    from util import assert_prepass_match
    n = 0
    for c in _prepass_golden():
        quads, depths = oracle.prepass(c["gaussians"], c["view"], c["proj"], c["model"], c["resolution"], c["near_far"], c["std_dev"],
                                       c["render_mode"], c["fmt"], 0)
        assert_prepass_match(quads, depths, c["quads"], c["depths"], c["resolution"], ordered=True)
        n += 1
    assert n == 5


def test_prepass_live_reference_build_when_available(live):
    """The golden cameras and formats on other gaussians (64 of each case, moved by up to 0.15): the reference shader's
    outputs for them, recorded by tests/golden/make_golden_live.py."""
    from util import assert_prepass_match
    n = 0
    for i, c in enumerate(_prepass_golden()):
        g = live[f"prepass_g{i}"]
        a = oracle.prepass(g, c["view"], c["proj"], c["model"], c["resolution"], c["near_far"], c["std_dev"], c["render_mode"], c["fmt"], 0)
        assert_prepass_match(a[0], a[1], live[f"prepass_quads{i}"], live[f"prepass_depths{i}"], c["resolution"], ordered=True)
        n += len(a[0])
    assert n > 0


def test_packed56_decodes_to_the_gaussian_vertex_it_was_encoded_from():
    """oracle.packed56_as_gaussian_vertex (what the prepass sees for a PACKED56 record, = what the reference's .ply loader
    builds) inverts the export arithmetic of parsers.cpp:484-499: scale * sigma/R, colour, alpha and rotation come back."""
    rng = np.random.default_rng(3)
    n = 300
    rec = np.zeros((n, 24), np.float32)
    rec[:, 0:3] = rng.random((n, 3)) * 4 - 2; rec[:, 3] = 1
    rec[:, 4:8] = rng.random((n, 4)) * 0.98 + 0.01
    rec[:, 8:10] = rng.random((n, 2)) * 3 + 0.01; rec[:, 10] = 1e-7
    q = rng.normal(size=(n, 4)); rec[:, 16:20] = q / np.linalg.norm(q, axis=1, keepdims=True)
    mult = 0.65 / 512
    packed = np.stack([oracle.encode(LAYOUT_PACKED56, rec[i], mult) for i in range(n)])   # one record per call
    g = oracle.packed56_as_gaussian_vertex(np.ascontiguousarray(packed).view(np.uint8).reshape(n, -1))
    assert np.allclose(g[:, 0:3], rec[:, 0:3], rtol=0, atol=0)
    assert np.allclose(g[:, 8:11], rec[:, 8:11] * np.float32(mult), rtol=2e-6)
    assert np.allclose(g[:, 4:7], rec[:, 4:7], atol=2e-7) and np.allclose(g[:, 7], rec[:, 7], atol=1e-6)
    assert np.array_equal(g[:, 16:20], rec[:, 16:20])
