"""Shared helpers for the parity tests: order-independent comparison keyed on fragment identity.

Tolerances (stated once, used everywhere):
  coverage (which (triangle, pixel) pairs emit a gaussian) ........ bit-exact (integer edge functions)
  position ........................................................ 1e-5 * bbox diagonal (absolute)
  raw scale / log-scale, quaternion (same sign convention) ........ 1e-5 relative (+1e-7 abs)
  colour / SH0 / opacity (compared as sigmoid(logit)) / metallic-roughness  1e-4 abs vs the oracle's fp32 sampler
                                                                    (2/255 is the bound vs a real GL driver)
  normal (TBN path) ............................................... 1e-3 abs
"""
from __future__ import annotations

import numpy as np

from mesh2splat_b200 import _abi

POS_TOL_REL_DIAG = 1e-5
REL_TOL = 1e-5
COLOR_TOL = 1e-4
NORMAL_TOL = 1e-3  # FMA-order noise is amplified by ill-conditioned TBN bases in the fuzz inputs
# ... and by normal-map texels near (0.5, 0.5, 0.5): normalize(tex * 2 - 1) of an almost-zero vector multiplies the fp32
# rounding of the interpolated uv (1 ulp = 1e-7 = 3e-5 texel of a 256^2 white-noise map) by up to 1/|v|.  At most this
# fraction of the records may exceed NORMAL_TOL, and then by no more than the contract's bound (SURVEY 8c: 1e-2)
NORMAL_OUTLIER_FRACTION = 2e-4
NORMAL_TOL_OUTLIER = 1e-2


def scene_diag(scene: _abi.Scene) -> float:
    pos = scene.triangles.reshape(-1, 3, 12)[:, :, :3].reshape(-1, 3)
    if len(pos) == 0:
        return 1.0
    pos = pos[np.isfinite(pos).all(axis=1)]
    if len(pos) == 0:
        return 1.0
    return float(np.linalg.norm(pos.max(axis=0) - pos.min(axis=0))) or 1.0


def sort_by_key(rec: np.ndarray, keys: np.ndarray):
    order = np.argsort(keys, kind="stable")
    return rec[order], keys[order]


def _close(a, b, rtol, atol, what, outlier_fraction=0.0, outlier_atol=0.0):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    both_nan = np.isnan(a) & np.isnan(b)
    both_inf = np.isinf(a) & np.isinf(b) & (np.sign(a) == np.sign(b))
    ok = both_nan | both_inf | (np.abs(a - b) <= atol + rtol * np.abs(b))
    if outlier_fraction and not ok.all():
        rows_bad = np.count_nonzero(~ok.reshape(len(ok), -1).all(axis=1))
        if rows_bad <= outlier_fraction * len(ok):
            ok = both_nan | both_inf | (np.abs(a - b) <= outlier_atol + rtol * np.abs(b))
    if not ok.all():
        bad = np.argwhere(~ok)[0]
        raise AssertionError(f"{what}: {np.count_nonzero(~ok)} mismatches, first at {tuple(bad)}: "
                             f"got {a[tuple(bad)]!r} want {b[tuple(bad)]!r}; max abs err "
                             f"{np.nanmax(np.abs(np.where(np.isfinite(a - b), a - b, 0)))}")


def _sigmoid(x):
    x = np.asarray(x, np.float64)
    with np.errstate(over="ignore"):
        return 1.0 / (1.0 + np.exp(-x))


def assert_records_match(scene: _abi.Scene, layout: int, got, got_keys, want, want_keys):
    """Set comparison: same fragment identities (exact), same values (tolerances above)."""
    assert len(got) == len(want), f"count {len(got)} != {len(want)}"
    g, gk = sort_by_key(got, np.asarray(got_keys, np.uint64))
    w, wk = sort_by_key(want, np.asarray(want_keys, np.uint64))
    assert np.array_equal(gk, wk), "coverage differs (fragment identity sets are not equal)"
    assert len(np.unique(gk)) == len(gk), "duplicate fragment identities"
    diag = scene_diag(scene)
    if layout == _abi.LAYOUT_REF96:
        _close(g["position"][:, :3], w["position"][:, :3], 0, POS_TOL_REL_DIAG * diag, "position")
        assert np.all(g["position"][:, 3] == 1.0)
        _close(g["scale"], w["scale"], REL_TOL, 1e-12, "scale")
        _close(g["rotation"], w["rotation"], REL_TOL, 1e-6, "rotation")
        _close(g["color"], w["color"], 0, COLOR_TOL, "color")
        _close(g["normal"], w["normal"], 0, NORMAL_TOL, "normal", NORMAL_OUTLIER_FRACTION, NORMAL_TOL_OUTLIER)
        _close(g["pbr"], w["pbr"], 0, COLOR_TOL, "pbr")
    elif layout == _abi.LAYOUT_PACKED56:
        _close(g["xyz"], w["xyz"], 0, POS_TOL_REL_DIAG * diag, "xyz")
        _close(g["rot"], w["rot"], REL_TOL, 1e-6, "rot")
        _close(g["log_scale"], w["log_scale"], REL_TOL, 1e-5, "log_scale")
        _close(g["sh0"], w["sh0"], 0, COLOR_TOL / 0.28209479177387814, "sh0")
        _close(_sigmoid(g["opacity"]), _sigmoid(w["opacity"]), 0, COLOR_TOL, "sigmoid(opacity)")
    elif layout in (_abi.LAYOUT_PLY_STANDARD, _abi.LAYOUT_PLY_PBR):
        _close(g["xyz"], w["xyz"], 0, POS_TOL_REL_DIAG * diag, "xyz")
        _close(g["normal"], w["normal"], 0, NORMAL_TOL, "normal", NORMAL_OUTLIER_FRACTION, NORMAL_TOL_OUTLIER)
        _close(g["f_dc"], w["f_dc"], 0, COLOR_TOL / 0.28209479177387814, "f_dc")
        _close(_sigmoid(g["opacity"]), _sigmoid(w["opacity"]), 0, COLOR_TOL, "sigmoid(opacity)")
        _close(g["scale"], w["scale"], REL_TOL, 1e-5, "scale")
        _close(g["rot"], w["rot"], REL_TOL, 1e-6, "rot")
        if layout == _abi.LAYOUT_PLY_STANDARD:
            assert not g["f_rest"].any()
        else:
            _close(g["metallic"], w["metallic"], 0, COLOR_TOL, "metallic")
            _close(g["roughness"], w["roughness"], 0, COLOR_TOL, "roughness")
    elif layout == _abi.LAYOUT_PLY_COMPRESSED:
        _close(g["xyz"], w["xyz"], 0, POS_TOL_REL_DIAG * diag, "xyz")
        _close(g["rot"], w["rot"], REL_TOL, 1e-6, "rot")
        _close(g["scale"], w["scale"], REL_TOL, 1e-5, "scale")
        for f in ("rgba", "octa", "roughness", "metallic"):  # u8 quantisation: off by one at rounding boundaries
            d = np.abs(g[f].astype(np.int32) - w[f].astype(np.int32))
            assert d.max(initial=0) <= 1, f"{f}: max byte diff {d.max()}"
            # a value within COLOR_TOL of a rounding boundary may round either way: that is 2 * COLOR_TOL * 255 of all values
            assert np.count_nonzero(d) <= max(4, 2 * COLOR_TOL * 255 * d.size), f"{f}: too many byte diffs"
    else:
        raise ValueError(layout)


def png_bytes(img: np.ndarray) -> bytes:
    """Minimal PNG writer (RGBA8 / RGB8 / gray8, filter 0) for loader tests."""
    import struct
    import zlib

    img = np.ascontiguousarray(img, np.uint8)
    if img.ndim == 2:
        ctype, ch = 0, 1
    else:
        ch = img.shape[2]
        ctype = {1: 0, 2: 4, 3: 2, 4: 6}[ch]
    h, w = img.shape[:2]
    raw = b"".join(b"\x00" + img[y].tobytes() for y in range(h))

    def chunk(t, d):
        return struct.pack(">I", len(d)) + t + d + struct.pack(">I", zlib.crc32(t + d) & 0xffffffff)

    return (b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, 8, ctype, 0, 0, 0))
            + chunk(b"IDAT", zlib.compress(raw, 6)) + chunk(b"IEND", b""))


def planar_triangulation(n_points: int, seed: int) -> _abi.Scene:
    """Delaunay triangulation of the unit square (4 corners + seeded random interior points), z = 0, uv = xy.
    The triangles tile the square with shared edges, so a watertight rasteriser (top-left rule) must emit every
    pixel centre of the R x R grid exactly once — a size-independent property of the coverage rules."""
    from scipy.spatial import Delaunay
    rng = np.random.default_rng(seed)
    pts = np.vstack([[[0, 0], [1, 0], [1, 1], [0, 1]], rng.random((n_points, 2))]).astype(np.float32)
    tri = Delaunay(pts.astype(np.float64)).simplices
    v = np.zeros((len(tri), 3, 12), np.float32)
    v[:, :, 0:2] = pts[tri]
    v[:, :, 5] = 1.0            # normal (0,0,1)
    v[:, :, 6] = 1.0; v[:, :, 9] = 1.0   # tangent (1,0,0,1)
    v[:, :, 10:12] = pts[tri]
    s = _abi.Scene(v.reshape(len(tri), 36), [_abi.Primitive(0, len(tri), (1, 1, 1, 1), -1, -1, -1)], [])
    s.compute_bboxes()
    return s


def png_encode(samples: np.ndarray, ctype: int, depth: int, interlace: bool = False, plte: bytes | None = None,
               trns: bytes | None = None) -> bytes:
    """General PNG writer for loader tests.  samples: (h, w, channels) integers < 2**depth (channels: 1 gray/palette,
    2 gray+alpha, 3 rgb, 4 rgba).  Rows cycle through the five filter types; Adam7 when interlace."""
    import struct
    import zlib
    smp = np.asarray(samples)
    h, w, ch = smp.shape
    assert ch == {0: 1, 2: 3, 3: 1, 4: 2, 6: 4}[ctype]

    def pack_row(row):  # (pw, ch) -> bytes
        flat = row.reshape(-1).astype(np.uint32)
        if depth == 8:
            return flat.astype(np.uint8).tobytes()
        if depth == 16:
            return flat.astype(">u2").tobytes()
        bits = np.zeros(len(flat) * depth, np.uint8)
        for b in range(depth):
            bits[b::depth] = (flat >> (depth - 1 - b)) & 1
        return np.packbits(bits).tobytes()

    fb = max(1, ch * depth // 8)

    def filt(rows):  # list of bytes -> filtered stream
        out = bytearray()
        prev = bytes(len(rows[0])) if rows else b""
        for y, r in enumerate(rows):
            ft = y % 5
            cur = bytearray(len(r))
            for i in range(len(r)):
                a = r[i - fb] if i >= fb else 0
                b = prev[i]
                c = prev[i - fb] if i >= fb else 0
                if ft == 0: pred = 0
                elif ft == 1: pred = a
                elif ft == 2: pred = b
                elif ft == 3: pred = (a + b) >> 1
                else:
                    pp = a + b - c
                    pa, pb, pc = abs(pp - a), abs(pp - b), abs(pp - c)
                    pred = a if (pa <= pb and pa <= pc) else (b if pb <= pc else c)
                cur[i] = (r[i] - pred) & 0xff
            out.append(ft); out += cur
            prev = r
        return bytes(out)

    passes = [(0, 0, 8, 8), (4, 0, 8, 8), (0, 4, 4, 8), (2, 0, 4, 4), (0, 2, 2, 4), (1, 0, 2, 2), (0, 1, 1, 2)] if interlace else [(0, 0, 1, 1)]
    raw = b""
    for x0, y0, dx, dy in passes:
        sub = smp[y0::dy, x0::dx]
        if sub.shape[0] == 0 or sub.shape[1] == 0:
            continue
        raw += filt([pack_row(sub[y]) for y in range(sub.shape[0])])

    def chunk(t, d):
        return struct.pack(">I", len(d)) + t + d + struct.pack(">I", zlib.crc32(t + d) & 0xffffffff)

    out = b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, depth, ctype, 0, 0, 1 if interlace else 0))
    if plte is not None:
        out += chunk(b"PLTE", plte)
    if trns is not None:
        out += chunk(b"tRNS", trns)
    half = len(raw) // 2 or 1
    z = zlib.compress(raw, 6)
    return out + chunk(b"IDAT", z[:half]) + chunk(b"IDAT", z[half:]) + chunk(b"IEND", b"")


def make_complex_glb(path: str, seed: int) -> None:
    """Random multi-mesh .glb for differential loader tests: node hierarchy up to depth 3 mixing `matrix` and TRS
    nodes, 2-4 meshes of 1-3 primitives (index types u8 / u16 / u32 / none; optional NORMAL / TANGENT / TEXCOORD_0;
    a LINES primitive and a POSITION-less one that must be skipped), several materials sharing images, a primitive
    without a material, a mesh instanced by two nodes, an unnamed mesh, optionally two scenes with `scene` set."""
    import json
    import struct
    rng = np.random.default_rng(seed)
    blobs, views, accessors = [], [], []

    def add_view(b):
        off = sum(len(x) for x in blobs)
        blobs.append(b + b"\x00" * ((-len(b)) % 4))
        views.append({"buffer": 0, "byteOffset": off, "byteLength": len(b)})
        return len(views) - 1

    def add_acc(arr, ctype, typ):
        accessors.append({"bufferView": add_view(np.ascontiguousarray(arr).tobytes()), "componentType": ctype, "count": len(arr), "type": typ})
        return len(accessors) - 1

    nimg = int(rng.integers(1, 4))
    images = []
    for i in range(nimg):
        w, h = int(rng.integers(2, 9)), int(rng.integers(2, 9))
        ch = int(rng.choice([3, 4]))
        images.append({"bufferView": add_view(png_bytes(rng.integers(0, 256, size=(h, w, ch), dtype=np.uint8))), "mimeType": "image/png"})
    textures = [{"source": int(rng.integers(0, nimg))} for _ in range(int(rng.integers(1, 5)))]
    materials = []
    for m in range(int(rng.integers(1, 4))):
        pbr = {}
        if rng.random() < 0.8: pbr["baseColorFactor"] = [float(v) for v in rng.random(4)]
        if rng.random() < 0.7: pbr["baseColorTexture"] = {"index": int(rng.integers(0, len(textures)))}
        if rng.random() < 0.5: pbr["metallicRoughnessTexture"] = {"index": int(rng.integers(0, len(textures)))}
        mat = {"name": f"mat{m}", "pbrMetallicRoughness": pbr}
        if rng.random() < 0.5: mat["normalTexture"] = {"index": int(rng.integers(0, len(textures))), "scale": 1.5}
        if rng.random() < 0.2: del mat["pbrMetallicRoughness"]
        materials.append(mat)
    meshes = []
    for mi in range(int(rng.integers(2, 5))):
        prims = []
        for pi in range(int(rng.integers(1, 4))):
            nv = int(rng.integers(3, 12))
            pos = (rng.normal(size=(nv, 3)) * 2).astype(np.float32)
            attrs = {"POSITION": add_acc(pos, 5126, "VEC3")}
            if rng.random() < 0.6:
                n = rng.normal(size=(nv, 3)); attrs["NORMAL"] = add_acc((n / np.linalg.norm(n, axis=1, keepdims=True)).astype(np.float32), 5126, "VEC3")
            if rng.random() < 0.5:
                t = rng.normal(size=(nv, 3)); t /= np.linalg.norm(t, axis=1, keepdims=True)
                attrs["TANGENT"] = add_acc(np.concatenate([t, np.where(rng.random((nv, 1)) < 0.5, -1.0, 1.0)], axis=1).astype(np.float32), 5126, "VEC4")
            if rng.random() < 0.7:
                attrs["TEXCOORD_0"] = add_acc(rng.random((nv, 2)).astype(np.float32), 5126, "VEC2")
            prim = {"attributes": attrs}
            kind = int(rng.integers(0, 4))
            ntri = int(rng.integers(1, 6))
            if kind < 3:
                idx = rng.integers(0, nv, size=ntri * 3)
                dt, ct = [(np.uint8, 5121), (np.uint16, 5123), (np.uint32, 5125)][kind]
                prim["indices"] = add_acc(idx.astype(dt), ct, "SCALAR")
            elif nv % 3:   # non-indexed needs a multiple of 3 vertices, else the reference skips the primitive: keep both cases
                if rng.random() < 0.5:
                    prim["attributes"]["POSITION"] = add_acc(pos[: nv - nv % 3], 5126, "VEC3")
                    for k in ("NORMAL", "TANGENT", "TEXCOORD_0"):
                        prim["attributes"].pop(k, None)
            if rng.random() < 0.8: prim["material"] = int(rng.integers(0, len(materials)))
            if rng.random() < 0.15: prim["mode"] = 1
            if rng.random() < 0.1: del prim["attributes"]["POSITION"]
            prims.append(prim)
        mesh = {"primitives": prims}
        if rng.random() < 0.8: mesh["name"] = f"part{mi}"
        meshes.append(mesh)

    def xform(node):
        r = rng.random()
        if r < 0.35:
            M = np.eye(4, dtype=np.float32); M[:3, :3] = rng.normal(size=(3, 3)); M[:3, 3] = rng.normal(size=3) * 3
            node["matrix"] = [float(v) for v in M.T.reshape(-1)]
        elif r < 0.8:
            if rng.random() < 0.8: node["translation"] = [float(v) for v in rng.normal(size=3) * 2]
            if rng.random() < 0.8:
                q = rng.normal(size=4); node["rotation"] = [float(v) for v in q / np.linalg.norm(q)]
            if rng.random() < 0.8: node["scale"] = [float(v) for v in rng.random(3) * 2 + 0.2]

    nodes = []
    def add_node(depth):
        node = {}
        xform(node)
        if rng.random() < 0.7: node["mesh"] = int(rng.integers(0, len(meshes)))
        nodes.append(node)
        me = len(nodes) - 1
        if depth < 3:
            kids = [add_node(depth + 1) for _ in range(int(rng.integers(0, 3)))]
            if kids: nodes[me]["children"] = kids
        return me
    roots = [add_node(1) for _ in range(int(rng.integers(1, 3)))]
    scenes = [{"nodes": roots}]
    gltf = {"asset": {"version": "2.0"}, "scenes": scenes, "nodes": nodes, "meshes": meshes, "materials": materials,
            "textures": textures, "images": images, "bufferViews": views, "accessors": accessors}
    if rng.random() < 0.3:
        other = add_node(1)
        gltf["scenes"] = [{"nodes": [other]}, {"nodes": roots}]
        gltf["scene"] = 1
    elif rng.random() < 0.7:
        gltf["scene"] = 0
    binblob = b"".join(blobs)
    gltf["buffers"] = [{"byteLength": len(binblob)}]
    js = json.dumps(gltf).encode(); js += b" " * ((-len(js)) % 4)
    with open(path, "wb") as f:
        f.write(struct.pack("<4sII", b"glTF", 2, 12 + 8 + len(js) + 8 + len(binblob)))
        f.write(struct.pack("<I4s", len(js), b"JSON")); f.write(js)
        f.write(struct.pack("<I4s", len(binblob), b"BIN\x00")); f.write(binblob)


def loader_transform_cases(n: int = 24, seed: int = 99) -> list:
    """Keyword arguments of test_abi_host._make_glb for n quads under random node transforms (even k: a `matrix` node,
    odd k: TRS) and varying attribute sets.  Shared by the loader test and tests/golden/make_golden_live.py."""
    rng = np.random.default_rng(seed)
    cases = []
    for k in range(n):
        if k % 2 == 0:
            M = np.eye(4, dtype=np.float32); M[:3, :3] = rng.normal(size=(3, 3)); M[:3, 3] = rng.normal(size=3) * 5
            kw = dict(matrix=M)
        else:
            q = rng.normal(size=4); q /= np.linalg.norm(q)
            kw = dict(trs=([float(v) for v in rng.normal(size=3)], [float(v) for v in q], [float(v) for v in rng.random(3) * 2 + 0.2]))
        kw.update(with_normals=bool(k % 3), with_tangents=bool(k % 5), indexed=bool(k % 4))
        cases.append(kw)
    return cases


def array_digest(arrays) -> str:
    """SHA-256 over the shapes, dtypes and bytes of a sequence of arrays: equal digests <=> equal arrays (for golden
    data too large to store whole)."""
    import hashlib
    h = hashlib.sha256()
    for a in arrays:
        a = np.ascontiguousarray(a)
        h.update(f"{a.dtype.str}{a.shape};".encode())
        h.update(a.tobytes())
    return h.hexdigest()


# ---- viewer prepass (SURVEY 8 f-4) --------------------------------------------------------------------------------
def assert_prepass_match(got_quads, got_depths, want_quads, want_depths, resolution, ordered: bool):
    """QuadNdcTransformation arrays [n, 24] + view depths.  ordered = False: the GPU appends in atomic arrival order, both
    sides are sorted by world position first.  Two outputs of the shader are ill-conditioned BY CONSTRUCTION and are
    compared through what they represent: the conic (inverse of the 2-D covariance: its off-diagonal is a difference of
    almost equal numbers for round splats) through the covariance itself, and the screen axes (eigenvectors: arbitrary —
    in the reference even 0/0 = NaN — when the two eigenvalues coincide) through the ellipse matrix they span."""
    g, w = np.asarray(got_quads, np.float64).reshape(-1, 24), np.asarray(want_quads, np.float64).reshape(-1, 24)
    gd, wd = np.asarray(got_depths, np.float64), np.asarray(want_depths, np.float64)
    assert len(g) == len(w) == len(gd) == len(wd), (len(g), len(w))
    if not ordered:   # pair every expected quad with the produced quad at the same world position (a bijection, or the sets differ)
        from scipy.spatial import cKDTree
        dist, idx = cKDTree(g[:, 20:23]).query(w[:, 20:23])
        scale = max(1.0, float(np.abs(w[:, 20:23]).max(initial=0.0)))
        assert (dist <= 1e-5 * scale).all(), f"{np.count_nonzero(dist > 1e-5 * scale)} expected gaussians have no counterpart (max distance {dist.max()})"
        if len(np.unique(idx)) != len(idx):   # coincident positions: fall back to a full sort of both sides on rounded keys
            key = lambda q: np.lexsort((np.round(q[:, 9], 5), np.round(q[:, 8], 5), np.round(q[:, 22], 5), np.round(q[:, 21], 5), np.round(q[:, 20], 5)))
            og, ow = key(g), key(w)
            g, gd, w, wd = g[og], gd[og], w[ow], wd[ow]
        else:
            g, gd = g[idx], gd[idx]
    _close(g[:, 20:24], w[:, 20:24], 1e-6, 1e-6, "wsPos / pbr.y")
    _close(gd, wd, 1e-5, 1e-6, "view depth")
    _close(g[:, 0:4], w[:, 0:4], 1e-5, 2e-5, "gaussianMean2dNdc")
    _close(g[:, 8:12], w[:, 8:12], 1e-5, 1e-6, "color")
    _close(g[:, 16:20], w[:, 16:20], 1e-5, 2e-5, "normal / pbr.x")
    _close(g[:, 15], w[:, 15], 1e-5, 1e-6, "conic.w (view depth)")

    def cov(q):
        a, b, c = q[:, 12], q[:, 13], q[:, 14]
        det = a * c - b * b
        return np.stack([c / det, -b / det, a / det], 1)
    cg, cw = cov(g), cov(w)
    _close(cg, cw, 2e-4, 1e-5, "2-D covariance (from the conic)")
    hx, hy = resolution[0] * 0.5, resolution[1] * 0.5

    def ellipse(q):
        mx, my, nx, ny = q[:, 4] * hx, q[:, 5] * hy, q[:, 6] * hx, q[:, 7] * hy
        return np.stack([mx * mx + nx * nx, mx * my + nx * ny, my * my + ny * ny], 1)
    eg, ew = ellipse(g), ellipse(w)
    # the shader's eigenvector is normalize(1, (l1 - a + b) / (l1 - c + b)) for cov = [[a, b], [b, c]]: numerator and denominator
    # both vanish for a round splat (0/0 = NaN in the reference itself) and, more generally, whenever a ~ c and b < 0
    # (l1 = a + |b|): there the direction is rounding noise on both sides and is not compared
    mid, dlt = cw[:, 0] + cw[:, 2], np.hypot(cw[:, 0] - cw[:, 2], 2 * cw[:, 1])
    l1 = 0.5 * (mid + dlt)
    num, den = -cw[:, 0] + cw[:, 1] + l1, cw[:, 1] - cw[:, 2] + l1
    ok = (np.abs(num) + np.abs(den)) > 5e-3 * l1
    assert not np.isnan(eg[ok]).any() and not np.isnan(ew[ok]).any(), "NaN axes for a splat that is not round"
    _close(eg[ok], ew[ok], 2e-3, 1e-3, "ellipse spanned by the screen axes (pixels^2)")
