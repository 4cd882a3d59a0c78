#!/usr/bin/env python3
"""Build the checkers of the viewer passes after the prepass (TEST INFRASTRUCTURE — never linked into the product).

  libm2s_render_oracle.so     the plain-C restatement of the depth sort and the splatting pass (m2s_render_oracle.c),
                              always built (gcc, OpenMP)
  _ref/libm2s_refsplat.so     the REFERENCE's splatting shaders — gaussianSplattingVS.glsl and gaussianSplattingPS.glsl,
                              read where they lie under the reference tree and turned into C++ by the token rewrites
                              below — compiled against the reference's vendored GLM.  Only built where the reference
                              tree exists; elsewhere tests/golden/ref_splat_vectors.npz holds its outputs.  Nothing from
                              the reference is written into the repository (oracle/_ref/ is git-ignored).

The same conventions as oracle/build.py, whose helpers this module uses.
"""
from __future__ import annotations

import os
import re
import sys

from .build import CFLAGS, HERE, REF, REF_OUT, _FLOAT_LIT, _newer, _run


def build_render_oracle(force: bool = False) -> str:
    src = os.path.join(HERE, "m2s_render_oracle.c")
    out = os.path.join(HERE, "libm2s_render_oracle.so")
    if force or not _newer(out, src, __file__):
        _run(["gcc", "-std=c11", "-fopenmp", *CFLAGS, "-o", out, src, "-lm"])
    return out


def glsl_splat_to_cpp(src: str) -> str:
    """gaussianSplattingVS.glsl / gaussianSplattingPS.glsl -> a C++ include (token rewrites only): interface variables and
    uniforms become statics, float literals get their suffix, the rvalue swizzles become GLM swizzle functions."""
    src = re.sub(r"^\s*#version.*$", "", src, flags=re.M)
    src = _FLOAT_LIT.sub(lambda m: m.group(1) + "f", src)
    src = re.sub(r"layout\s*\(\s*location\s*=\s*\d+\s*\)\s*", "", src)
    src = re.sub(r"^\s*(?:in|out|uniform)\s+(\w+\s+\w+\s*;)", r"static \1", src, flags=re.M)
    src = re.sub(r"\.(xyz|xzy|xy|zw|rgb)\b(?!\s*\()", r".\1()", src)
    src = re.sub(r"\+\s*(\d+)\s*\)", r"+ \1.0f)", src)   # GLSL converts the int operand of vec + int
    return src


def build_ref_splat(force: bool = False) -> str | None:
    """The reference's splatting shaders (row f-6), compiled where they lie against the reference's GLM."""
    vs = os.path.join(REF, "src", "shaders", "rendering", "gaussianSplattingVS.glsl")
    ps = os.path.join(REF, "src", "shaders", "rendering", "gaussianSplattingPS.glsl")
    glm = os.path.join(REF, "thirdParty", "glm")
    out = os.path.join(REF_OUT, "libm2s_refsplat.so")
    if not (os.path.exists(vs) and os.path.exists(ps) and os.path.isdir(glm)):
        return out if os.path.exists(out) else None
    harness = os.path.join(HERE, "ref_splat_harness.cpp")
    if not force and _newer(out, vs, ps, harness, __file__):
        return out
    os.makedirs(REF_OUT, exist_ok=True)
    for src, name in ((vs, "splatVS.inc"), (ps, "splatPS.inc")):
        with open(src) as f:
            inc = glsl_splat_to_cpp(f.read())
        with open(os.path.join(REF_OUT, name), "w") as f:
            f.write(inc)
    _run(["g++", "-std=gnu++17", *CFLAGS, "-w", "-I", glm, "-I", REF_OUT, "-o", out, harness])
    return out


def build_all(force: bool = False) -> dict:
    return {"render_oracle": build_render_oracle(force), "ref_splat": build_ref_splat(force)}


if __name__ == "__main__":
    print(build_all(force="--force" in sys.argv))
