#!/usr/bin/env python3
"""Builds mesh2splat_b200/libm2s.so — the C-ABI shared library (CUDA kernels for sm_100a + C++ host).

In-tree build with plain nvcc so the .so travels with the repository snapshot to the GPU box
(a JIT cache would not).  `python -m mesh2splat_b200.build [--force] [--verbose]`.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libm2s.so")
SOURCES = ["m2s_kernels.cu", "m2s_prepass.cu", "m2s_render.cu", "m2s_api.cu", "m2s_host.cpp", "m2s_glb.cpp"]
HEADERS = ["m2s_device.cuh", "m2s_prepass.cuh", "m2s_render.cuh", "m2s_span.cuh", os.path.join("..", "..", "include", "m2s.h")]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]


def _nvcc() -> str:
    for c in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found")


def _stale() -> bool:
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [__file__]
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False, out: str | None = None, defs: list | None = None) -> str:
    """out/defs: build a tuning variant (e.g. defs=['M2S_WARPS_REF96=12','M2S_REGS_REF96=168']) to another file;
    select it at run time with the M2S_LIB environment variable."""
    if out is None and not defs and not force and not _stale():
        return OUT
    out = out or OUT
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    cmd = [_nvcc(), "-std=c++17", "-O3", "-lineinfo", *ARCH, "-shared", "-Xcompiler", "-fPIC,-fvisibility=hidden",
           "--cudart", "static", "-o", out, *[f"-D{d}" for d in (defs or [])], *srcs]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
        raise RuntimeError("nvcc failed")
    if verbose:
        sys.stderr.write(r.stdout + r.stderr)
    return out


if __name__ == "__main__":
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    out = None
    defs = []
    for a in sys.argv[1:]:
        if a.startswith("--out="):
            out = a[6:]
        if a.startswith("--def="):
            defs.append(a[6:])
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv, out=out, defs=defs))
