"""Device time of the viewer's depth sort (m2s_sort_quads_enqueue) and splatting pass (m2s_splat) on the bench scene
(synth.helmet_standin(2048)) at R = 512 and R = 2048, both record layouts, 1920 x 1080, with the camera of
scripts/prepass_bench.py.  CUDA events on the context stream, L2 flushed between steps; for context, torch.sort(stable=True)
of the same keys.  Byte model (the least the passes move): sort = 4-byte keys and values read and written once per 8-bit
digit pass (4 passes) plus the 96-byte quads read and written by the gather; splat = the 96-byte quad, its 112-byte set-up
and the 8-byte pair read once per (tile, quad) pair, plus the G-buffer (24 B per pixel) written once."""
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import numpy as np  # noqa: E402
import torch  # noqa: E402
from make_golden_prepass import column_major, look_at, perspective  # noqa: E402

from mesh2splat_b200 import _abi, synth  # noqa: E402
from mesh2splat_b200._lib import check, lib  # noqa: E402
from mesh2splat_b200.api import Context, GBuffer  # noqa: E402


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        return r.stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name(0) + " (power limit not readable)"


def main(steps=10, warmup=3):
    print("GPU:", gpu_info())
    ctx = Context(0)
    scene = synth.helmet_standin(2048)
    ds = ctx.upload(scene)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    V = column_major(look_at(np.array([0.0, 0.5, 3.2]), np.zeros(3), np.array([0.0, 1.0, 0.0])).astype(np.float32))
    P = column_major(perspective(np.radians(45.0), 16 / 9, 0.01, 100.0))
    M = column_major(np.eye(4, dtype=np.float32))
    W, H = 1920, 1080
    rows = []
    for R in (512, 2048):
        for layout, name in ((_abi.LAYOUT_REF96, "ref96"), (_abi.LAYOUT_PACKED56, "packed56")):
            out = ctx.convert(ds, R, layout, flags=_abi.FLAG_UNCAPPED, capacity=6 * R * R)
            n = out.written
            std = 0.65 / R if layout == _abi.LAYOUT_REF96 else 1.0
            q, d = ctx.prepass(out.data, n, layout, V, P, M, (W, H), (0.01, 100.0), std, 0)
            m = len(q)
            quads, depths = torch.from_numpy(q).cuda(), torch.from_numpy(d).cuda()
            sorted_q = torch.empty((m, 24), dtype=torch.float32, device="cuda")
            gb = GBuffer.empty(W, H, 0, "cuda")
            g = gb.c_struct()
            sp = _abi.m2s_splat_params(W, H, 0, 0)
            ts_sort, ts_splat, ts_torch, pairs = [], [], [], 0
            for i in range(warmup + steps):
                flush.zero_(); torch.cuda.synchronize()
                ms = C.c_float(0)
                check(lib().m2s_sort_quads(ctx.handle, quads.data_ptr(), depths.data_ptr(), m, sorted_q.data_ptr(), None, C.byref(ms)))
                ts_sort.append(ms.value)
                flush.zero_(); torch.cuda.synchronize()
                pr, ms2 = C.c_uint64(0), C.c_float(0)
                check(lib().m2s_splat(ctx.handle, sorted_q.data_ptr(), m, None, C.byref(sp), C.byref(g), C.byref(pr), C.byref(ms2)))
                ts_splat.append(ms2.value); pairs = pr.value
                flush.zero_(); torch.cuda.synchronize()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                keys = depths.view(torch.int32).to(torch.int64) & 0xFFFFFFFF
                a.record()
                torch.sort(keys, stable=True)
                b.record(); torch.cuda.synchronize()
                ts_torch.append(a.elapsed_time(b))
            t_sort = float(np.median(ts_sort[warmup:])) * 1e-3
            t_splat = float(np.median(ts_splat[warmup:])) * 1e-3
            t_torch = float(np.median(ts_torch[warmup:])) * 1e-3
            sort_bytes = m * 8 * 2 * 4 + m * 96 * 2
            splat_bytes = pairs * (96 + 112 + 8) + W * H * 24
            row = dict(R=R, layout=name, gaussians=n, survivors=m, pairs=int(pairs), sort_us=t_sort * 1e6, splat_us=t_splat * 1e6,
                       torch_sort_stable_us=t_torch * 1e6, mgaussians_per_s=m / (t_sort + t_splat) / 1e6,
                       sort_gbs=sort_bytes / t_sort / 1e9, splat_gbs=splat_bytes / t_splat / 1e9)
            rows.append(row)
            print(f"render R={R:5d} {name:9s} gaussians {n:9d} survivors {m:9d} pairs {pairs:10d}  sort {t_sort * 1e6:9.1f} us "
                  f"(torch.sort stable int64 keys {t_torch * 1e6:9.1f} us)  splat {t_splat * 1e6:9.1f} us  "
                  f"{row['mgaussians_per_s']:8.1f} Mgaussians/s  byte model: sort {row['sort_gbs']:6.1f} GB/s, splat {row['splat_gbs']:6.1f} GB/s")
            del out, quads, depths, sorted_q
    print(json.dumps(rows))


if __name__ == "__main__":
    main()
