"""Synthetic quads for the render tests (QuadNdcTransformation rows, 24 float32) and the G-buffer comparison."""
import numpy as np


def quad(cx, cy, ax, ay, bx, by, W, H, depth=-1.0, color=(0.8, 0.4, 0.2, 0.5), conic=(0.0, 0.0, 0.0), normal=(0.1, 0.2, 0.3, 0.25),
         ws=(1.0, 2.0, 3.0, 0.75)):
    """A quad centred at window position (cx, cy) with half axes (ax, ay) and (bx, by) in pixels; conic = 0 gives g = 1 exactly."""
    q = np.zeros(24, np.float32)
    q[0] = cx / (W * 0.5) - 1.0; q[1] = cy / (H * 0.5) - 1.0; q[2] = 0.5; q[3] = 1.0
    q[4] = ax / (W * 0.5); q[5] = ay / (H * 0.5); q[6] = bx / (W * 0.5); q[7] = by / (H * 0.5)
    q[8:12] = color
    q[12:15] = conic; q[15] = -depth
    q[16:20] = normal
    q[20:24] = ws
    return q


def synthetic_quads(W, H, seed, n=400, deep=0):
    """Conic-0 quads: random sizes from sub-pixel to 1024 px, rotated, straddling tiles and screen edges, equal depths, plus
    `deep` quads stacked over one pixel region."""
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n):
        cx, cy = rng.uniform(-0.1 * W, 1.1 * W), rng.uniform(-0.1 * H, 1.1 * H)
        kind = i % 5
        r = [0.3, 2.0, 9.0, 40.0, min(1024.0, 0.6 * max(W, H))][kind] * rng.uniform(0.5, 1.0)
        ang = rng.uniform(0, np.pi)
        e = rng.uniform(0.3, 1.0)
        ax, ay = r * np.cos(ang), r * np.sin(ang)
        bx, by = -e * r * np.sin(ang), e * r * np.cos(ang)
        col = rng.uniform(0, 1, 4).astype(np.float32)
        out.append(quad(cx, cy, ax, ay, bx, by, W, H, depth=-float(rng.integers(1, 4)), color=col,
                        normal=rng.uniform(-1, 1, 4), ws=rng.uniform(-5, 5, 4)))
    if n:
        out.append(quad(W * 0.5, H * 0.5, 1024.0, 0.0, 0.0, 3.0, W, H))   # at the prepass's 1024-pixel axis limit
    for k in range(deep):
        out.append(quad(W * 0.5 + 0.37 * (k % 7), H * 0.5 - 0.21 * (k % 5), 5.0 + k % 3, 1.0, -1.0, 4.0, W, H,
                        color=(0.3, 0.6, 0.9, 0.02 + 0.001 * (k % 10)), depth=-2.0))
    return np.stack(out).astype(np.float32) if out else np.zeros((0, 24), np.float32)


def assert_gbuffer_equal(got: dict, want: dict):
    for name in ("position", "normal", "albedo", "depth", "metallic_roughness"):
        g, w = np.asarray(got[name]), np.asarray(want[name])
        assert g.shape == w.shape, (name, g.shape, w.shape)
        gb = g.view(np.uint16) if g.dtype == np.float16 else g
        wb = w.view(np.uint16) if w.dtype == np.float16 else w
        bad = np.argwhere(gb != wb)
        assert len(bad) == 0, f"{name}: {len(bad)} components differ, first at {bad[:3].tolist()}: got {g[tuple(bad[0])]} want {w[tuple(bad[0])]}"
