"""CPU test of bench.py --dump-outputs: the files two runs or two builds are compared by must be finite, float32 or
float64, and independent of the order in which the kernels appended the records."""
import os

import numpy as np
import pytest

import bench
from mesh2splat_b200 import _abi


def _records(layout: int, n: int) -> np.ndarray:
    rng = np.random.default_rng(5)
    rec = np.zeros(n, _abi.record_dtype(layout))
    flat = rec.view(np.float32).reshape(n, -1)
    flat[:] = rng.normal(size=flat.shape).astype(np.float32)
    flat[::9, 0] = flat[1::9, 0]                                  # equal positions: the later columns decide
    flat[5] = flat[6]                                             # a duplicate record
    flat[7, 1], flat[8, 1] = np.float32(-0.0), np.float32(0.0)
    if layout == _abi.LAYOUT_PACKED56:
        rec["opacity"][: n // 2] = np.inf                         # logit(1): an opaque gaussian
        rec["opacity"][n // 2: n // 2 + 10] = -np.inf
    return rec


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


@pytest.mark.parametrize("layout", [_abi.LAYOUT_PACKED56, _abi.LAYOUT_REF96])
def test_dump_is_finite_and_independent_of_arrival_order(tmp_path, layout):
    rec = _records(layout, 3000)
    bench.dump_records(str(tmp_path / "a"), rec)
    bench.dump_records(str(tmp_path / "b"), rec[np.random.default_rng(1).permutation(len(rec))])
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    names = [n if n != "opacity" else "alpha" for n in rec.dtype.names]
    assert sorted(a) == sorted(names + ["total"])
    for k in a:
        assert a[k].dtype in (np.float32, np.float64), k
        assert np.isfinite(a[k]).all(), k
        assert a[k].tobytes() == b[k].tobytes(), k
    assert a["total"].tolist() == [3000.0]
    if layout == _abi.LAYOUT_PACKED56:
        alpha = np.sort(a["alpha"])
        assert alpha[0] == 0.0 and alpha[-1] == 1.0 and np.count_nonzero(alpha == 1.0) == 1500
        np.testing.assert_allclose(np.sort(1 / (1 + np.exp(-rec["opacity"][1510:].astype(np.float64)))), alpha[10:1500])


def test_dump_keeps_a_fixed_sample_within_the_byte_budget(tmp_path, monkeypatch):
    rec = _records(_abi.LAYOUT_PACKED56, 3000)
    monkeypatch.setattr(bench, "DUMP_BYTES", 100_000)
    bench.dump_records(str(tmp_path / "a"), rec)
    bench.dump_records(str(tmp_path / "b"), rec[::-1].copy())
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert sum(v.nbytes for v in a.values()) <= 100_000
    assert 0 < len(a["xyz"]) < 3000 and a["total"].tolist() == [3000.0]
    for k in a:
        assert len(a[k]) == len(a["xyz"]) or k == "total"
        assert a[k].tobytes() == b[k].tobytes(), k
