"""On-device evaluation of a scene nDSM against the ground-truth DSM (the evaluation step of the reference's inference
CLI, evaluator.py:53-99: residual statistics per mask class, evaluator.py:83-95).

``residual_stats`` makes one call of ``t2h_residual_stats`` (csrc/t2h_eval.cu) and one device-to-host read of the
results; everything in between stays on the stream.  count, min, max, median, medae and nmad equal numpy's fp64
results bit for bit; the sums come from a reduction tree fixed by the raster size (bitwise reproducible, independent of
which other masks are passed).
"""
import torch

from . import _lib

FIELDS = ("mean", "mae", "rmse", "min", "max", "median", "medae", "nmad")
MAX_MASKS = 8
# passes over the rasters made by t2h_residual_stats: statistics + first digit, 7 more digits of median(r) and
# median |r|, 8 digits of median |r - median(r)|
DATA_PASSES = 16


def residual_stats(pred, gt, masks=None, nodata=None):
    """Residual statistics of ``pred - gt`` per class.

    ``pred``, ``gt``: floating rasters of one shape on one CUDA device (e.g. the float64 output of
    ``SceneGenerator.generate``, NaN where no tile covers a pixel).  ``masks``: optional mapping of up to 8 names to
    boolean rasters of that shape (they may overlap).  ``nodata``: optional no-data value of ``gt``.

    A pixel is valid when ``pred`` and ``gt`` are finite and ``gt != nodata``; r = float64(pred) - float64(gt).  Returns
    ``{"all": stats, name: stats, ...}``, where "all" covers every valid pixel and each mask the valid pixels inside it,
    and ``stats`` holds ``count`` (int) and ``mean`` (bias), ``mae``, ``rmse``, ``min``, ``max``, ``median`` (numpy's
    rule: the mean of the two middle values for an even count), ``medae`` (median |r|) and
    ``nmad`` = 1.4826 * median |r - median(r)|.  An empty class has count 0 and NaN elsewhere.

    Raises ValueError for mismatched shapes or devices, a non-floating input, a non-boolean mask, more than 8 masks or a
    mask named "all"; RuntimeError for tensors that are not on a CUDA device (there is no CPU fallback)."""
    masks = dict(masks or {})
    for what, t in (("pred", pred), ("gt", gt)):
        if not isinstance(t, torch.Tensor) or not t.dtype.is_floating_point:
            raise ValueError(f"residual_stats: {what} must be a floating-point tensor, got "
                             f"{t.dtype if isinstance(t, torch.Tensor) else type(t).__name__}")
    if pred.shape != gt.shape:
        raise ValueError(f"residual_stats: pred {tuple(pred.shape)} and gt {tuple(gt.shape)} differ in shape")
    if len(masks) > MAX_MASKS:
        raise ValueError(f"residual_stats: at most {MAX_MASKS} masks, got {len(masks)}")
    if "all" in masks:
        raise ValueError('residual_stats: "all" is the class of every valid pixel and cannot name a mask')
    for name, m in masks.items():
        if not isinstance(m, torch.Tensor) or m.dtype != torch.bool:
            raise ValueError(f"residual_stats: mask {name!r} must be a boolean tensor")
        if m.shape != pred.shape:
            raise ValueError(f"residual_stats: mask {name!r} {tuple(m.shape)} differs in shape from pred {tuple(pred.shape)}")
    devices = {t.device for t in (pred, gt, *masks.values())}
    if len(devices) > 1:
        raise ValueError(f"residual_stats: inputs live on different devices {sorted(str(d) for d in devices)}")
    if not pred.is_cuda:
        raise RuntimeError("residual_stats: expected CUDA tensors (the B200 path has no CPU fallback)")

    p = pred.to(torch.float64).contiguous()
    g = gt.to(torch.float64).contiguous()
    bits = None
    if masks:
        bits = torch.zeros(p.shape, dtype=torch.uint8, device=p.device)
        for c, m in enumerate(masks.values()):
            bits.bitwise_or_(m.to(torch.uint8) << c)
    nc = 1 + len(masks)
    n_px = p.numel()
    lib = _lib.load()
    ws_bytes = lib.t2h_residual_stats_workspace_bytes(n_px, len(masks))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=p.device)
    # stats (nc x 8 float64) and counts (nc int64) in one buffer: one device-to-host copy at the end
    res = torch.empty(nc * 9 * 8, dtype=torch.uint8, device=p.device)
    stats, counts = res[:nc * 64].view(torch.float64), res[nc * 64:].view(torch.int64)
    _lib.call("t2h_residual_stats", _lib.ptr(p), _lib.ptr(g), n_px, _lib.ptr(bits), len(masks),
              int(nodata is not None), float(nodata) if nodata is not None else 0.0, _lib.ptr(ws), ws_bytes,
              _lib.ptr(stats), _lib.ptr(counts))
    host = res.cpu()
    stats, counts = host[:nc * 64].view(torch.float64).view(nc, 8).tolist(), host[nc * 64:].view(torch.int64).tolist()
    out = {}
    for c, name in enumerate(["all", *masks]):
        out[name] = {"count": counts[c], **dict(zip(FIELDS, stats[c]))}
    return out
