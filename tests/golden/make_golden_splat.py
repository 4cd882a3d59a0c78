#!/usr/bin/env python3
"""Generates tests/golden/ref_splat_vectors.npz from the REFERENCE's own splatting shaders (SURVEY 8 f-6).

Runs only where the reference tree is present: oracle/build_render.py compiles src/shaders/rendering/gaussianSplattingVS.glsl and
gaussianSplattingPS.glsl (unmodified arithmetic, token-level GLSL -> C++ rewrites) against the reference's vendored GLM into
oracle/_ref/libm2s_refsplat.so.  The quads are those of the committed prepass golden cases (tests/golden/ref_prepass_vectors.npz,
at most 32 per case); for each quad the file stores the 4 corner positions and the five shader outputs, in render modes 0
and 4, at 16 fragment positions: 12 pixel centres inside the quad's box and 4 in the tails beyond it.  The committed .npz is
what travels.

    python tests/golden/make_golden_splat.py
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import build_render  # noqa: E402
from oracle import render as roracle  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
PER_CASE = 32
FRAGS_IN, FRAGS_TAIL = 12, 4


def fragment_positions(rng, quad, W, H):
    """Pixel centres inside the quad's window-space box and in the tails up to twice its half extent."""
    sx, sy = (quad[0] + 1) * 0.5 * W, (quad[1] + 1) * 0.5 * H
    ex = (abs(quad[4]) + abs(quad[6])) * 0.5 * W + 1.0
    ey = (abs(quad[5]) + abs(quad[7])) * 0.5 * H + 1.0
    u = rng.uniform(-1, 1, (FRAGS_IN, 2)) * [ex, ey]
    ang = rng.uniform(0, 2 * np.pi, FRAGS_TAIL)
    r = rng.uniform(1.0, 2.0, FRAGS_TAIL)
    t = np.stack([np.cos(ang) * r * ex, np.sin(ang) * r * ey], axis=1)
    p = np.concatenate([u, t]) + [sx, sy]
    return (np.floor(p) + 0.5).astype(np.float32)


def main():
    assert build_render.build_ref_splat() is not None, "needs the reference tree"
    pre = np.load(os.path.join(HERE, "ref_prepass_vectors.npz"))
    rng = np.random.default_rng(20261017)
    out = {}
    for i in range(int(pre["ncases"])):
        W, H = (float(v) for v in pre[f"params{i}"][:2])
        quads = pre[f"quads{i}"]
        quads = quads[np.isfinite(quads).all(axis=1)][:PER_CASE]
        frags = np.stack([fragment_positions(rng, q, W, H) for q in quads])
        corners = np.zeros((len(quads), 4, 4), np.float32)
        outs = np.zeros((2, len(quads), FRAGS_IN + FRAGS_TAIL, 5, 4), np.float32)
        for k, q in enumerate(quads):
            for m, mode in enumerate((0, 4)):
                c, o = roracle.ref_splat(q, W, H, mode, frags[k])
                corners[k] = c
                outs[m, k] = o
        out[f"quads{i}"] = quads; out[f"frags{i}"] = frags; out[f"corners{i}"] = corners
        out[f"out{i}"] = outs; out[f"size{i}"] = np.array([W, H], np.float32)
    out["ncases"] = np.array(int(pre["ncases"]))
    out["modes"] = np.array([0, 4])
    path = os.path.join(HERE, "ref_splat_vectors.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes;", [len(out[f"quads{i}"]) for i in range(int(pre["ncases"]))], "quads")


if __name__ == "__main__":
    main()
