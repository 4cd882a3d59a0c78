"""The splatting kernel's triangle set-up (m2s_span.cuh, compiled for the host with g++) covers exactly the pixels the
oracle's rasteriser covers: each synthetic quad alone in overdraw mode, where a pixel's alpha counts its fragments."""
import os
import shutil
import subprocess

import numpy as np
import pytest

from oracle import render as roracle
from render_util import synthetic_quads

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("g++ not available")
    exe = str(tmp_path_factory.mktemp("span") / "render_span")
    subprocess.run([gxx, "-std=c++17", "-O2", "-ffp-contract=off", "-o", exe, os.path.join(HERE, "render_span_harness.cpp")], check=True)
    return exe


@pytest.mark.parametrize("W,H", [(97, 61), (16, 16), (1, 1), (300, 40)])
def test_kernel_setup_covers_what_the_oracle_covers(harness, W, H):
    q = synthetic_quads(W, H, seed=W + 1000 * H, n=150, deep=5)
    q = q[np.abs(q[:, 4:8]).max(axis=1) * max(W, H) < 400]   # keep the per-quad oracle renders small
    lines = [f"{W} {H} {len(q)}"] + [" ".join(repr(float(v)) for v in row[:2].tolist() + row[4:8].tolist()) for row in q]
    out = subprocess.run([harness], input="\n".join(lines) + "\n", capture_output=True, text=True, check=True).stdout.splitlines()
    assert len(out) == len(q)
    hit = 0
    for row, line in zip(q, out):
        v = [int(t) for t in line.split()]
        got = np.zeros(W * H, np.int64)
        np.add.at(got, np.array(v[2:], np.int64), 1)
        want = roracle.splat(row[None], W, H, 4)["albedo"][..., 3].reshape(-1).astype(np.int64) // 3
        assert np.array_equal(got, want)
        hit += v[0] + v[1]
    assert hit > 0
