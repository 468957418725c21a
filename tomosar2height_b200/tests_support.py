"""Small host-side helpers shared by tests and benchmarks (no oracle dependency)."""
import torch


def _compact1by1(v):
    v = v & 0x55555555
    v = (v | (v >> 1)) & 0x33333333
    v = (v | (v >> 2)) & 0x0F0F0F0F
    v = (v | (v >> 4)) & 0x00FF00FF
    v = (v | (v >> 8)) & 0x0000FFFF
    return v


def demorton(code: torch.Tensor):
    """Morton code (x in the even bits) -> (ix, iy), int64 tensors."""
    code = code.long()
    return _compact1by1(code), _compact1by1(code >> 1)


def numpy_residual_stats(pred, gt, masks=None, nodata=None):
    """fp64 numpy statement of ``evaluation.residual_stats`` (same validity rule, classes and fields): the host
    reference of the tests and of ``tools/bench_eval.py``.  Sums are numpy's pairwise sums."""
    import numpy as np
    p, g = np.asarray(pred, dtype=np.float64), np.asarray(gt, dtype=np.float64)
    valid = np.isfinite(p) & np.isfinite(g)
    if nodata is not None:
        valid &= g != nodata
    out = {}
    for name, m in [("all", None), *(masks or {}).items()]:
        sel = valid if m is None else valid & np.asarray(m, dtype=bool)
        out[name] = residual_summary(p[sel] - g[sel])
    return out


def residual_summary(r):
    """count, mean, mae, rmse, min, max, median, medae, nmad of a 1-D float64 residual array (NaN when empty)."""
    import numpy as np
    n = int(r.size)
    if n == 0:
        return {"count": 0, **{k: float("nan") for k in ("mean", "mae", "rmse", "min", "max", "median", "medae", "nmad")}}
    a = np.abs(r)
    med = np.median(r)
    return {"count": n, "mean": float(np.mean(r)), "mae": float(np.mean(a)), "rmse": float(np.sqrt(np.mean(r * r))),
            "min": float(r.min()), "max": float(r.max()), "median": float(med), "medae": float(np.median(a)),
            "nmad": float(1.4826 * np.median(np.abs(r - med)))}


def synthetic_eval_rasters(rows, cols, seed=0, device="cuda", border=64):
    """A seeded nDSM / ground-truth pair shaped like a scene evaluation: ``pred`` float64 heights with a NaN border of
    ``border`` pixels (as ``SceneGenerator.generate`` leaves uncovered pixels), ``gt`` float32 with -9999 no-data
    patches, and the masks ``building = gt > 2.5``, ``ground = ~building``.  Returns (pred, gt, masks, nodata)."""
    g = torch.Generator(device=device).manual_seed(seed)
    u = lambda *s: torch.rand(*s, generator=g, device=device, dtype=torch.float64)
    gt = (u(rows, cols) < 0.3) * (3.0 + 30.0 * u(rows, cols)) + 0.5 * u(rows, cols)
    pred = gt + torch.randn(rows, cols, generator=g, device=device, dtype=torch.float64) * (0.5 + 2.0 * (gt > 2.5))
    gt = gt.float()
    pred[:border], pred[-border:], pred[:, :border], pred[:, -border:] = (float("nan"),) * 4
    for _ in range(16):  # no-data patches
        r0, c0 = int(u(1) * (rows - rows // 20)), int(u(1) * (cols - cols // 20))
        gt[r0:r0 + rows // 20, c0:c0 + cols // 20] = -9999.0
    building = gt > 2.5
    return pred, gt, {"building": building, "ground": ~building}, -9999.0
