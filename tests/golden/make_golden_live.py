#!/usr/bin/env python3
"""Generates tests/golden/ref_live_vectors.npz: what the REFERENCE's own code makes of the inputs of the tests in
tests/test_oracle.py named *live_reference*: its geometry shader on a random triangle soup, its .ply writer on random
records, its .glb parser on transformed quads and on random multi-mesh scene graphs, its viewer prepass on moved
gaussians.

Needs the reference sources, which oracle/build.py compiles into oracle/_ref/ (as for make_golden.py).  The tests
read only the committed .npz, so they run wherever the repository does.  Numeric inputs are stored next to the
outputs; the .glb inputs are rebuilt by the seeded writers in tests/ (util.loader_transform_cases + _make_glb,
util.make_complex_glb).  Per scene graph the triangles and the decoded texels are stored as SHA-256 digests
(util.array_digest): the whole arrays would be several hundred kB, the digests compare them just as exactly.

    python tests/golden/make_golden_live.py
"""
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))

import oracle  # noqa: E402
from oracle import build as obuild  # noqa: E402
from mesh2splat_b200 import synth  # noqa: E402

OUT = os.path.join(HERE, "ref_live_vectors.npz")
PLY_RECORDS = 128
GRAPH_SEEDS = range(5000, 5120)
PREPASS_PER_CASE = 64    # a seeded sample of the 500 gaussians of each ref_prepass_vectors.npz case


def gs_vectors(out):
    rng = np.random.default_rng(7)
    tris = synth.random_soup(500, seed=11, extent=3.0, tri_size=1.0)
    pos = tris.reshape(-1, 3, 12)[:, :, :3].reshape(-1, 3)
    mn = pos.min(axis=0) - 0.1
    mx = pos.max(axis=0) + rng.random(3).astype(np.float32)
    glpos = np.zeros((len(tris), 3, 2), np.float32); scale = np.zeros((len(tris), 3), np.float32); quat = np.zeros((len(tris), 4), np.float32)
    for i, t in enumerate(tris):
        p, scale[i], quat[i] = oracle.ref_gs(t, mn, mx)
        glpos[i] = p[:, :2]
    out.update(gs_tris=tris, gs_bmin=mn.astype(np.float32), gs_bmax=mx.astype(np.float32), gs_glpos_xy=glpos, gs_scale=scale, gs_quat=quat)


def ply_vectors(out, d):
    rng = np.random.default_rng(77)
    rec = rng.random((PLY_RECORDS, 24)).astype(np.float32)
    rec[:, 8:11] *= np.float32(0.01); rec[:PLY_RECORDS // 10, 7] = 1.0     # alpha 1: opacity +inf
    mult = np.float32(0.65) / np.float32(300)
    out.update(ply_records=rec, ply_scale_multiplier=np.float32(mult))
    for fmt in (0, 1, 2):
        path = os.path.join(d, f"live{fmt}.ply")
        assert oracle.ref_save_ply(path, rec, fmt, float(mult))
        out[f"ply_format_{fmt}"] = np.frombuffer(open(path, "rb").read(), np.uint8)


def loader_vectors(out, d):
    from test_abi_host import _make_glb
    from util import loader_transform_cases
    faces, counts = [], []
    for k, kw in enumerate(loader_transform_cases()):
        p = os.path.join(d, f"c{k}.glb")
        _make_glb(p, **kw)
        ok, meshes = oracle.ref_load_glb(p)
        assert ok
        faces.append(np.vstack([m["faces"] for m in meshes]))
        counts.append(len(faces[-1]))
    out.update(loader_faces=np.vstack(faces), loader_face_counts=np.array(counts, np.int64))


def graph_vectors(out, d):
    from util import array_digest, make_complex_glb
    seeds, mesh_counts, names, colors, present, face_dig, tex_dig = [], [], [], [], [], [], []
    for seed in GRAPH_SEEDS:
        p = os.path.join(d, "g.glb")
        make_complex_glb(p, seed)
        ok, meshes = oracle.ref_load_glb(p)
        if not ok or not meshes:
            continue
        seeds.append(seed)
        mesh_counts.append(len(meshes))
        for m in meshes:
            names.append(m["name"]); colors.append(m["base_color"])
            present.append([int(w in m["textures"]) for w in range(3)])
        face_dig.append(array_digest([np.vstack([m["faces"] for m in meshes])]))
        tex_dig.append(array_digest([m["textures"][w] for m in meshes for w in range(3) if w in m["textures"]]))
    out.update(graph_seeds=np.array(seeds, np.int64), graph_mesh_counts=np.array(mesh_counts, np.int64), graph_mesh_names=np.array(names),
               graph_base_color=np.stack(colors), graph_tex_present=np.array(present, np.uint8), graph_faces_sha256=np.array(face_dig),
               graph_texels_sha256=np.array(tex_dig))


def prepass_vectors(out):
    g = np.load(os.path.join(HERE, "ref_prepass_vectors.npz"))
    rng, pick = np.random.default_rng(77), np.random.default_rng(1)
    for i in range(int(g["ncases"])):
        p = g[f"params{i}"]
        gs = g[f"g{i}"].copy()
        gs[:, 0:3] += (rng.random((len(gs), 3)).astype(np.float32) - 0.5) * 0.3
        gs = gs[np.sort(pick.choice(len(gs), PREPASS_PER_CASE, replace=False))]
        quads, depths = oracle.ref_prepass(gs, g[f"view{i}"], g[f"proj{i}"], g[f"model{i}"], (float(p[0]), float(p[1])),
                                           (float(p[2]), float(p[3])), float(p[4]), int(p[5]), int(p[6]), 0)
        out.update({f"prepass_g{i}": gs, f"prepass_quads{i}": quads, f"prepass_depths{i}": depths})


def main():
    built = obuild.build_all()
    missing = [k for k in ("ref", "ref_ply", "ref_loader", "ref_prepass") if built[k] is None]
    if missing:
        raise SystemExit(f"oracle/_ref is not built ({', '.join(missing)}): the reference sources are not here")
    out = {}
    with tempfile.TemporaryDirectory() as d:
        gs_vectors(out)
        ply_vectors(out, d)
        loader_vectors(out, d)
        graph_vectors(out, d)
    prepass_vectors(out)
    np.savez_compressed(OUT, **out)
    print("wrote", OUT, os.path.getsize(OUT), "bytes;", len(out["graph_seeds"]), "scene graphs")


if __name__ == "__main__":
    main()
