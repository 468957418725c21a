"""CPU checks of the nDSM evaluation: the numpy reference the GPU tests compare with (against brute-force sorted
lists), the argument checks of the t2h_residual_stats entry point, and every ValueError of residual_stats."""
import math
import os

import numpy as np
import pytest
import torch

from tomosar2height_b200 import _lib, residual_stats
from tomosar2height_b200.tests_support import numpy_residual_stats, residual_summary


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build_library()
    return _lib.load()


def brute_median(values):
    s = sorted(values)
    n = len(s)
    return s[n // 2] if n % 2 else (s[n // 2 - 1] + s[n // 2]) / 2


@pytest.mark.parametrize("n", [1, 2, 3, 4, 7, 10, 101, 1000])
def test_reference_against_sorted_lists(n):
    rng = np.random.default_rng(n)
    r = rng.standard_normal(n) * 10.0 ** rng.integers(-3, 4, n)
    got = residual_summary(r)
    vals = [float(v) for v in r]
    med = brute_median(vals)
    assert got["count"] == n
    assert got["median"] == med
    assert got["medae"] == brute_median([abs(v) for v in vals])
    assert got["nmad"] == 1.4826 * brute_median([abs(v - med) for v in vals])
    assert got["min"] == min(vals) and got["max"] == max(vals)
    assert math.isclose(got["mean"], math.fsum(vals) / n, rel_tol=1e-12, abs_tol=1e-300)
    assert math.isclose(got["rmse"], math.sqrt(math.fsum(v * v for v in vals) / n), rel_tol=1e-12)


def test_reference_even_median_is_the_mean_of_the_middle_pair():
    got = residual_summary(np.array([4.0, 1.0, 3.0, 2.0]))
    assert got["median"] == 2.5 and got["medae"] == 2.5
    assert got["nmad"] == 1.4826 * 1.0                       # |r - 2.5| = 1.5, 0.5, 0.5, 1.5
    assert residual_summary(np.array([1.0, 2.0]))["median"] == 1.5


def test_reference_empty_class_and_validity():
    got = residual_summary(np.array([], dtype=np.float64))
    assert got["count"] == 0 and all(math.isnan(got[k]) for k in got if k != "count")
    pred = np.array([[1.0, np.nan, 3.0], [np.inf, 5.0, 6.0]])
    gt = np.array([[0.0, 0.0, -9999.0], [0.0, np.nan, 1.0]])
    masks = {"left": np.array([[True, True, False], [True, True, False]]), "none": np.zeros((2, 3), bool)}
    ref = numpy_residual_stats(pred, gt, masks, nodata=-9999.0)
    assert ref["all"]["count"] == 2 and ref["all"]["median"] == 3.0       # r = 1 and 5
    assert ref["left"]["count"] == 1 and ref["left"]["max"] == 1.0
    assert ref["none"]["count"] == 0 and math.isnan(ref["none"]["median"])
    assert numpy_residual_stats(pred, gt)["all"]["count"] == 3           # without nodata -9999 is a value


def test_entry_point_refuses_bad_arguments_without_a_gpu(lib):
    small = lib.t2h_residual_stats_workspace_bytes(1000, 2)
    assert 0 < small < lib.t2h_residual_stats_workspace_bytes(1 << 20, 2)
    assert lib.t2h_residual_stats_workspace_bytes(1000, 9) == 0
    ws, out, cnt, p = 0x1000, 0x2000, 0x3000, 0x4000   # never dereferenced: the checks come before any launch
    # pred, gt, n_px, mask_bits, n_masks, use_nodata, nodata, ws, ws_bytes, out_stats, out_count, stream
    assert lib.t2h_residual_stats(None, p, 10, None, 0, 0, 0.0, ws, small, out, cnt, None) == 1
    assert lib.t2h_residual_stats(p, None, 10, None, 0, 0, 0.0, ws, small, out, cnt, None) == 1
    assert lib.t2h_residual_stats(p, p, 10, None, 2, 0, 0.0, ws, small, out, cnt, None) == 1      # masks without bits
    assert lib.t2h_residual_stats(p, p, 10, p, 9, 0, 0.0, ws, small, out, cnt, None) == 1        # > 8 masks
    assert lib.t2h_residual_stats(p, p, -1, None, 0, 0, 0.0, ws, small, out, cnt, None) == 1
    assert lib.t2h_residual_stats(p, p, 10, None, 0, 0, 0.0, None, small, out, cnt, None) == 1
    assert lib.t2h_residual_stats(p, p, 10, None, 0, 0, 0.0, ws, small, None, cnt, None) == 1
    assert lib.t2h_residual_stats(p, p, 10, None, 0, 0, 0.0, ws, small, out, None, None) == 1
    need = lib.t2h_residual_stats_workspace_bytes(1 << 20, 2)
    assert lib.t2h_residual_stats(p, p, 1 << 20, p, 2, 0, 0.0, ws, need - 1, out, cnt, None) == 4


@pytest.mark.parametrize("device", ["cpu", "meta"])
def test_residual_stats_value_errors(device):
    f = lambda *s, dt=torch.float64: torch.zeros(*s, dtype=dt, device=device)
    pred, gt = f(4, 5), f(4, 5, dt=torch.float32)
    with pytest.raises(ValueError, match="shape"):
        residual_stats(pred, f(5, 4))
    with pytest.raises(ValueError, match="at most 8"):
        residual_stats(pred, gt, masks={f"m{i}": f(4, 5, dt=torch.bool) for i in range(9)})
    with pytest.raises(ValueError, match='"all"'):
        residual_stats(pred, gt, masks={"all": f(4, 5, dt=torch.bool)})
    with pytest.raises(ValueError, match="boolean"):
        residual_stats(pred, gt, masks={"building": f(4, 5, dt=torch.uint8)})
    with pytest.raises(ValueError, match="shape"):
        residual_stats(pred, gt, masks={"building": f(5, 4, dt=torch.bool)})
    with pytest.raises(ValueError, match="floating"):
        residual_stats(f(4, 5, dt=torch.int32), gt)
    with pytest.raises(ValueError, match="floating"):
        residual_stats(pred, f(4, 5, dt=torch.int64))
    other = "meta" if device == "cpu" else "cpu"
    with pytest.raises(ValueError, match="devices"):
        residual_stats(pred, torch.zeros(4, 5, device=other))
    with pytest.raises(ValueError, match="devices"):
        residual_stats(pred, gt, masks={"building": torch.zeros(4, 5, dtype=torch.bool, device=other)})
    with pytest.raises(RuntimeError, match="CUDA"):
        residual_stats(pred, gt, masks={"building": f(4, 5, dt=torch.bool)}, nodata=-9999.0)
