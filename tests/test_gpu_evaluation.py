"""residual_stats (t2h_residual_stats) on the device against the fp64 numpy reference: exact order statistics bit for
bit, sums within the fsum bound, adversarial inputs for the radix select, determinism, independence of the other
classes, a generated scene, the full Munich raster size and more than 2^31 pixels."""
import math
import struct

import numpy as np
import pytest
import torch

from tomosar2height_b200 import residual_stats
from tomosar2height_b200.tests_support import numpy_residual_stats, residual_summary, synthetic_eval_rasters

pytestmark = pytest.mark.gpu

EXACT = ("min", "max", "median", "medae", "nmad")


def same(a, b):
    return (math.isnan(a) and math.isnan(b)) or a == b


def check_exact(got, ref):
    assert list(got) == list(ref)
    for name in ref:
        assert got[name]["count"] == ref[name]["count"], name
        for k in EXACT:
            assert same(got[name][k], ref[name][k]), (name, k, got[name][k], ref[name][k])


def check_sums(stats, r):
    """|S - fsum(terms)| <= 1e-12 fsum(|terms|) for S = n mean, n mae, n rmse^2 (plus the rounding of the division
    and square root that turned S into the returned field)."""
    n = r.size
    for field, terms, total in (("mean", r, stats["mean"] * n), ("mae", np.abs(r), stats["mae"] * n),
                                ("rmse", r * r, stats["rmse"] ** 2 * n)):
        exact, mag = math.fsum(terms), math.fsum(np.abs(terms))
        assert abs(total - exact) <= 1e-12 * mag + 2.0 ** -48 * abs(exact), (field, total, exact)


def residuals(pred, gt, mask=None, nodata=None):
    p, g = pred.double().cpu().numpy(), gt.double().cpu().numpy()
    sel = np.isfinite(p) & np.isfinite(g)
    if nodata is not None:
        sel &= g != nodata
    if mask is not None:
        sel &= mask.cpu().numpy()
    return p[sel] - g[sel]


def host(masks):
    return {k: v.cpu().numpy() for k, v in masks.items()}


@pytest.mark.parametrize("parity", [0, 1])
def test_random_residuals_with_overlapping_masks(parity):
    g = torch.Generator(device="cuda").manual_seed(11 + parity)
    rows, cols = 300, 301
    gt = (torch.rand(rows, cols, generator=g, device="cuda") * 40.0).float()
    scale = 10.0 ** torch.randint(-3, 2, (rows, cols), generator=g, device="cuda").double()
    pred = gt.double() + torch.randn(rows, cols, generator=g, device="cuda", dtype=torch.float64) * scale
    pred[torch.rand(rows, cols, generator=g, device="cuda") < 0.05] = float("nan")
    n_valid = int(torch.isfinite(pred).sum())
    if n_valid % 2 != parity:
        pred.view(-1)[torch.isfinite(pred.view(-1)).nonzero()[0]] = float("nan")
    masks = {"high": gt > 20.0, "band": (gt > 10.0) & (gt < 30.0), "empty": torch.zeros_like(gt, dtype=torch.bool)}
    got = residual_stats(pred, gt, masks)
    ref = numpy_residual_stats(pred.cpu().numpy(), gt.cpu().numpy(), host(masks))
    assert got["all"]["count"] % 2 == parity and got["high"]["count"] and got["band"]["count"]
    assert got["empty"]["count"] == 0 and all(math.isnan(got["empty"][k]) for k in got["empty"] if k != "count")
    check_exact(got, ref)
    for name in ("all", "high", "band"):
        check_sums(got[name], residuals(pred, gt, masks.get(name)))


def adversarial(case, n, rng):
    if case == "equal":
        return np.full(n, 3.25)
    if case == "two_values":
        return rng.choice([-1.5, 2.0], n)
    if case == "ulp_apart":
        return 1.0 + rng.integers(0, 4, n) * np.spacing(1.0)
    if case == "signed_zeros":
        return rng.choice([-0.0, 0.0, -1e-3, 1e-3, -7.0, 0.0], n)
    if case == "subnormals":
        return rng.integers(-40, 41, n) * 5e-324
    if case == "huge":
        return rng.choice([-1.0, 1.0], n) * 1e300 * (1.0 + rng.integers(0, 8, n) * 2.0 ** -50)
    raise ValueError(case)


@pytest.mark.parametrize("shape", [(33, 31), (32, 32)])
@pytest.mark.parametrize("case", ["equal", "two_values", "ulp_apart", "signed_zeros", "subnormals", "huge"])
def test_adversarial_distributions(case, shape):
    rng = np.random.default_rng(sum(map(ord, case)))
    n = shape[0] * shape[1]
    r = adversarial(case, n, rng).reshape(shape)
    if case in ("equal", "two_values"):           # small integers: pred - gt gives r back exactly
        gt = rng.integers(-5, 6, shape).astype(np.float64)
        pred = r + gt
    else:                                           # gt = +0.0 keeps r bit for bit, -0.0 included
        gt = np.zeros(shape)
        pred = r.copy()
    assert np.array_equal((pred - gt).view(np.int64), r.view(np.int64))
    mask = rng.random(shape) < 0.5
    masks = {"half": torch.from_numpy(mask).cuda(), "all_px": torch.ones(shape, dtype=torch.bool, device="cuda")}
    got = residual_stats(torch.from_numpy(pred).cuda(), torch.from_numpy(gt).cuda(), masks)
    check_exact(got, numpy_residual_stats(pred, gt, host(masks)))
    assert got["all"]["count"] == n and got["all"]["median"] == np.median(r)
    if case not in ("huge", "subnormals"):         # squares overflow / underflow there; the exact fields still hold
        check_sums(got["all"], r.ravel())


def test_non_finite_inputs_and_nodata_are_excluded():
    rng = np.random.default_rng(5)
    shape = (40, 50)
    gt = rng.standard_normal(shape) * 5.0
    pred = gt + rng.standard_normal(shape)
    bad = rng.integers(0, 6, shape)
    pred[bad == 0] = np.inf
    pred[bad == 1] = -np.inf
    gt[bad == 2] = np.nan
    pred[bad == 3] = np.nan
    gt[bad == 4] = -9999.0
    gt[0, :7] = [np.inf, -np.inf, np.nan, -9999.0, -9999.0, 1.0, 2.0]
    pred[0, :7] = [1.0, 2.0, 3.0, np.nan, 4.0, np.inf, -np.inf]
    mask = rng.random(shape) < 0.3
    masks = {"m": torch.from_numpy(mask).cuda()}
    got = residual_stats(torch.from_numpy(pred).cuda(), torch.from_numpy(gt).cuda(), masks, nodata=-9999.0)
    ref = numpy_residual_stats(pred, gt, host(masks), nodata=-9999.0)
    assert ref["all"]["count"] == int((bad == 5).sum()) - int((bad[0, :7] == 5).sum())
    check_exact(got, ref)
    check_sums(got["all"], residuals(torch.from_numpy(pred), torch.from_numpy(gt), nodata=-9999.0))
    # without a nodata value -9999 is an ordinary (valid) ground-truth height
    check_exact(residual_stats(torch.from_numpy(pred).cuda(), torch.from_numpy(gt).cuda()),
                numpy_residual_stats(pred, gt))


def bitwise(stats):
    return {name: {k: (v if k == "count" else struct.pack("<d", v)) for k, v in s.items()} for name, s in stats.items()}


def test_deterministic_and_independent_of_the_other_masks():
    pred, gt, _, nodata = synthetic_eval_rasters(1000, 1200, seed=4, border=16)
    g = torch.Generator(device="cuda").manual_seed(8)
    masks = {f"m{i}": torch.rand(gt.shape, generator=g, device="cuda") < (i + 1) / 9 for i in range(8)}
    first = bitwise(residual_stats(pred, gt, masks, nodata))
    assert bitwise(residual_stats(pred, gt, masks, nodata)) == first
    assert bitwise(residual_stats(pred, gt, nodata=nodata))["all"] == first["all"]
    one = bitwise(residual_stats(pred, gt, {"m3": masks["m3"]}, nodata))
    assert one["all"] == first["all"] and one["m3"] == first["m3"]
    check_exact(residual_stats(pred, gt, masks, nodata), numpy_residual_stats(pred.cpu().numpy(), gt.cpu().numpy(),
                                                                               host(masks), nodata))


def test_generated_scene_against_numpy():
    import oracle
    import tomosar2height_b200 as t2h
    from cases import CASES, make_cfg
    from tomosar2height_b200.generator import SceneGenerator
    cfg = make_cfg(**CASES["berlin_small"]["cfg"])
    model = t2h.TomoSAR2Height(cfg)
    model.load_state_dict(oracle.synth_state_dict(oracle.reference_param_shapes(cfg), seed=3))
    model = model.cuda()
    g = torch.Generator().manual_seed(9)
    lo = torch.tensor([386000.0, 5820000.0], dtype=torch.float64)
    size = torch.tensor([300.0, 260.0], dtype=torch.float64)
    pts = torch.rand(60000, 3, generator=g, dtype=torch.float64)
    pts[:, :2] = lo + pts[:, :2] * size
    pts[:, 2] = 30.0 + pts[:, 2] * 40.0
    pts = pts[~((pts[:, 0] > lo[0] + 230) & (pts[:, 1] > lo[1] + 200))]
    gen = SceneGenerator(model, lo.tolist(), (lo + size).tolist(), cfg.dataset.normalize.z_bound,
                         patch_size=128.0, stride=64.0, pixel_size=1.0, tiles_per_batch=3)
    dsm, _ = gen.generate(pts.cuda())
    dsm[:8] = float("nan")                          # rows no tile covers, as a scene larger than its cloud leaves them
    gt = (dsm.nan_to_num(0.0) + torch.randn(dsm.shape, generator=g, dtype=torch.float64).cuda()).float()
    gt[100:120, 40:90] = -9999.0
    masks = {"building": gt > 2.5, "ground": gt <= 2.5}
    got = residual_stats(dsm, gt, masks, nodata=-9999.0)
    ref = numpy_residual_stats(dsm.cpu().numpy(), gt.cpu().numpy(), host(masks), nodata=-9999.0)
    check_exact(got, ref)
    for name, m in (("all", None), *masks.items()):
        check_sums(got[name], residuals(dsm, gt, m, nodata=-9999.0))


def test_munich_size_raster_against_numpy():
    pred, gt, masks, nodata = synthetic_eval_rasters(5730, 9050, seed=0)
    got = residual_stats(pred, gt, masks, nodata)
    ref = numpy_residual_stats(pred.cpu().numpy(), gt.cpu().numpy(), host(masks), nodata)
    check_exact(got, ref)
    for name in ref:
        # numpy's pairwise sums are within a few ulps of fsum at this size
        assert abs(got[name]["mean"] - ref[name]["mean"]) <= 2e-12 * ref[name]["mae"], name
        assert abs(got[name]["mae"] - ref[name]["mae"]) <= 2e-12 * ref[name]["mae"], name
        assert abs(got[name]["rmse"] ** 2 - ref[name]["rmse"] ** 2) <= 2e-12 * ref[name]["rmse"] ** 2, name


def test_more_than_2_31_pixels():
    m, k = 1001, 2145339
    assert m * k > 2 ** 31 and (m * k) % 2 == 1
    if torch.cuda.mem_get_info()[0] < 48 * 2 ** 30:
        pytest.skip("needs 48 GB of free device memory")
    pattern = np.random.default_rng(3).standard_normal(m) * 10.0
    pred = torch.from_numpy(pattern).cuda().repeat(k).view(k, m)
    gt = torch.zeros(k, m, dtype=torch.float64, device="cuda")
    got = residual_stats(pred, gt)["all"]
    del pred, gt
    own = residual_summary(pattern)
    assert got["count"] == m * k
    for f in EXACT:
        assert got[f] == own[f], f
    for field, terms, total in (("mean", pattern, got["mean"] * m * k), ("mae", np.abs(pattern), got["mae"] * m * k),
                                ("rmse", pattern ** 2, got["rmse"] ** 2 * m * k)):
        exact, mag = k * math.fsum(terms), k * math.fsum(np.abs(terms))
        assert abs(total - exact) <= 1e-12 * mag + 2.0 ** -48 * abs(exact), (field, total, exact)
