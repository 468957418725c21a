"""Scene generation with an orthophoto on the device: t2h_raster_windows against the torch expression, and whole-scene
generation of cloud + image and image-only models against a CPU restatement of the reference's per-tile path."""
import numpy as np
import pytest
import torch

import oracle
from oracle.generator import accumulate_scene, crop_normalize_tile, raster_col_row
from cases import CASES, make_cfg

pytestmark = pytest.mark.gpu


def torch_windows(raster, t_rows, l_cols, S, mean, std):
    """out[b, h, j, c] = (raster[c, t_row[b] + S-1-h, l_col[b] + j] - mean[c]) / std[c]"""
    wins = [raster[:, t:t + S, l:l + S].flip(1) for t, l in zip(t_rows, l_cols)]
    return torch.stack([((w - mean[:, None, None]) / std[:, None, None]).permute(1, 2, 0) for w in wins])


def run_windows(raster, t_rows, l_cols, S, mean, std):
    from tomosar2height_b200 import _lib
    C, H, W = raster.shape
    out = torch.empty(len(t_rows), S, S, C, device="cuda")
    # held in names until the kernel has run: a temporary's memory could be handed to the next allocation
    t_rows_d = torch.tensor(t_rows, dtype=torch.int32, device="cuda")
    l_cols_d = torch.tensor(l_cols, dtype=torch.int32, device="cuda")
    _lib.call("t2h_raster_windows", _lib.ptr(raster), C, H, W, _lib.ptr(t_rows_d), _lib.ptr(l_cols_d), len(t_rows), S,
              _lib.ptr(mean), _lib.ptr(std), _lib.ptr(out))
    torch.cuda.synchronize()
    return out


@pytest.mark.parametrize("C,S", [(1, 16), (3, 16), (3, 128), (1, 200)])
def test_raster_windows_bitwise(C, S):
    g = torch.Generator(device="cuda").manual_seed(C * 1000 + S)
    H, W = S + 37, S + 151
    raster = (torch.randn(C, H, W, generator=g, device="cuda") * 40.0 + 100.0).contiguous()
    mean = torch.randn(C, generator=g, device="cuda") * 50.0
    std = torch.rand(C, generator=g, device="cuda") * 30.0 + 0.3
    # the four corners (every raster edge touched), a repeated window, an interior one
    t_rows = [0, H - S, 0, H - S, 0, 17]
    l_cols = [0, W - S, W - S, 0, 0, 93]
    for B in (1, 4, 6):
        got = run_windows(raster, t_rows[:B], l_cols[:B], S, mean, std)
        ref = torch_windows(raster, t_rows[:B], l_cols[:B], S, mean, std)
        assert got.shape == (B, S, S, C)
        assert torch.equal(got, ref), (C, S, B)
    # the encoder's NCHW view of the channels-last windows
    assert torch.equal(got.permute(0, 3, 1, 2)[5, :, 0, :], ((raster[:, 17 + S - 1, 93:93 + S] - mean[:, None]) / std[:, None]))


def test_raster_windows_outside_pixels_are_nan():
    """An origin partly off the raster does not read outside it: those pixels come out as NaN, the rest as usual."""
    raster = torch.arange(2 * 20 * 30, dtype=torch.float32, device="cuda").reshape(2, 20, 30)
    mean, std = torch.tensor([1.0, 2.0], device="cuda"), torch.tensor([3.0, 4.0], device="cuda")
    got = run_windows(raster, [-3, 14], [25, -2], 8, mean, std)
    padded = torch.full((2, 20 + 6, 30 + 6), float("nan"), device="cuda")
    padded[:, 3:23, 3:33] = raster
    ref = torch_windows(padded, [0, 17], [28, 1], 8, mean, std)
    assert torch.equal(torch.isnan(got), torch.isnan(ref)) and bool(torch.isnan(got).any())
    assert torch.equal(got[~torch.isnan(got)], ref[~torch.isnan(ref)])


def oracle_generate_dsm_image(P, cfg, points, scene_min, scene_max, image, left, top, mean, std, patch, stride, px):
    """oracle.generator.oracle_generate_dsm with the orthophoto input: per tile, the window at RasterData.query_col_row
    of the tile's corner pixels in the image, flipped (row 0 = southern edge), normalised per channel, and handed to
    oracle_forward with the tile's points (or alone for an image-only cfg).  Tiles without points are skipped."""
    pts = points.double().cpu()
    l, b = float(scene_min[0]), float(scene_min[1])
    r, t = float(scene_max[0]), float(scene_max[1])
    z_bound = cfg["dataset"]["normalize"]["z_bound"]
    S = int(round(patch / px))
    xs = np.concatenate([np.arange(l, r - patch, stride), [r - patch]])
    ys = np.concatenate([np.arange(b, t - patch, stride), [t - patch]])
    tiles, anchors = [], []
    for y0 in ys:
        for x0 in xs:
            x0, y0 = float(x0), float(y0)
            _, norm = crop_normalize_tile(pts, x0, y0, patch, z_bound[1] - z_bound[0])
            anchors.append((x0, y0))
            if norm is None or norm.shape[0] == 0:
                tiles.append(None)
                continue
            l_col, _ = raster_col_row(x0 + px / 2.0, y0 + px / 2.0, left, top, px)
            _, t_row = raster_col_row(x0 + patch - px / 2.0, y0 + patch - px / 2.0, left, top, px)
            window = image[:, t_row:t_row + S, l_col:l_col + S].flip(1)
            window = (window - mean[:, None, None]) / std[:, None, None]
            with torch.no_grad():
                cloud = norm[None] if cfg["use_cloud"] else None
                tiles.append(oracle.oracle_forward(P, cfg, cloud, window[None])[0][0])
    dsm, weight = accumulate_scene(tiles, anchors, scene_min, scene_max, patch, px)
    return torch.maximum(dsm / weight, torch.tensor(0., dtype=torch.float64)), weight


def scene_points():
    """the scene of test_gpu_generator.py (300 m x 260 m, one empty corner, points on an anchor line), Munich heights"""
    g = torch.Generator().manual_seed(9)
    lo = torch.tensor([386000.0, 5820000.0], dtype=torch.float64)
    size = torch.tensor([300.0, 260.0], dtype=torch.float64)
    pts = torch.rand(60000, 3, generator=g, dtype=torch.float64)
    pts[:, :2] = lo + pts[:, :2] * size
    pts[:, 2] = 470.0 + pts[:, 2] * 60.0
    pts = pts[~((pts[:, 0] > lo[0] + 230) & (pts[:, 1] > lo[1] + 200))]
    pts[:50, 0] = lo[0] + 64.0
    return pts, lo.tolist(), (lo + size).tolist()


@pytest.mark.parametrize("use_cloud", [True, False], ids=["cloud+image", "image-only"])
def test_scene_generation_with_image_matches_oracle(use_cloud):
    import tomosar2height_b200 as t2h
    from tomosar2height_b200.generator import OrthoImage, SceneGenerator
    from tomosar2height_b200.parallel import shard_tiles
    torch.backends.cudnn.allow_tf32 = False
    cfg = make_cfg(**CASES["munich_small"]["cfg"])  # cloud + image + footprint head, 128 m tiles at 1 m pixels
    cfg["use_cloud"] = use_cloud
    params = oracle.synth_state_dict(oracle.reference_param_shapes(cfg), seed=5)
    model = t2h.TomoSAR2Height(cfg)
    model.load_state_dict(params)
    model = model.cuda()
    pts, lo, hi = scene_points()
    # an orthophoto reaching past the scene, its corner 7.25 / 5.5 pixels off the scene's
    g = torch.Generator().manual_seed(21)
    image = torch.randn(3, 280, 320, generator=g) * 60.0 + 120.0
    left, top = lo[0] - 7.25, hi[1] + 5.5
    mean, std = torch.tensor([118.0, 121.5, 125.0]), torch.tensor([55.0, 61.0, 58.5])
    ortho = OrthoImage(image, left, top, 1.0, mean, std)
    gen = SceneGenerator(model, lo, hi, cfg.dataset.normalize.z_bound, patch_size=128.0, stride=64.0, pixel_size=1.0,
                         tiles_per_batch=3)
    dsm, weight = gen.generate(pts.cuda(), image=ortho)
    ref, ref_w = oracle_generate_dsm_image(params, cfg, pts, lo, hi, image, left, top, mean, std, 128.0, 64.0, 1.0)
    assert dsm.shape == ref.shape == (260, 300)
    assert torch.allclose(weight.cpu(), ref_w, rtol=1e-12, atol=0)      # same live tiles, same windows
    covered = ref_w > 0
    scale = ref[covered].abs().max()
    assert scale > 0
    assert (dsm.cpu()[covered] - ref[covered]).abs().max() <= 1e-4 * scale
    # tile sharding: partial rasters of 2 ranks (equal blocks) and of 3 ranks (blocks balanced by points) add up
    for parts in ([gen.generate(pts.cuda(), image=ortho, tile_range=shard_tiles(len(gen.anchors), rk, 2)) for rk in range(2)],
                  [gen.generate(pts.cuda(), image=ortho, rank=rk, world=3) for rk in range(3)]):
        w_sum = sum(p[1] for p in parts)
        assert torch.allclose(w_sum.cpu(), ref_w, rtol=1e-12, atol=0)
        merged = gen.finalize(sum(p[0] for p in parts), w_sum)
        assert (merged[covered.cuda()] - dsm[covered.cuda()]).abs().max().item() <= 1e-5 * scale.item()
