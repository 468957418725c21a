"""Pin the CPU oracle against fixtures produced by the real reference (tests/golden/make_golden.py)."""
import json
import os

import numpy as np
import pytest
import torch

import oracle
from cases import CASES, make_cfg, grad_probe_positions

CASE_NAMES = list(CASES)


def _load(golden_dir, name):
    return np.load(os.path.join(golden_dir, name + ".npz"))


def test_op_vectors(golden_dir):
    v = _load(golden_dir, "op_vectors")
    # G-1 (pointnet.py:114-123): index and plane of the reference's printed self-check
    xy = torch.from_numpy(v["g1_xy"])
    idx = oracle.cell_index(xy, 2)
    assert idx.dtype == torch.int64 and idx.tolist() == [[[0, 2, 1, 3, 0]]]
    assert np.array_equal(idx.numpy(), v["g1_index"])
    plane = oracle.segment_mean(xy.permute(0, 2, 1), idx, 4).reshape(1, 2, 2, 2)
    np.testing.assert_allclose(plane.numpy(), v["g1_plane"], rtol=1e-6)
    np.testing.assert_allclose(plane.numpy(), [[[[0.05, 0.9], [0.3, 0.9]], [[0.1, 0.3], [0.9, 0.9]]]], rtol=1e-6)
    # G-2 ties / empty
    out, arg = oracle.segment_max(torch.from_numpy(v["g2_src"]), torch.from_numpy(v["g2_index"]), 5)
    assert out.flatten().tolist() == [1, 3, 0, -2, 0] and arg.flatten().tolist() == [0, 1, 4, 3, 4]
    assert np.array_equal(out.numpy(), v["g2_out"]) and np.array_equal(arg.numpy(), v["g2_arg"])
    # G-3 border points
    edge = torch.from_numpy(v["g3_xy"])
    for r in (256, 100):
        assert np.array_equal(oracle.cell_index(edge, r).numpy(), v[f"g3_index_{r}"])
    assert oracle.cell_index(edge, 256)[0, 0, 0].item() == 255
    # G-4 grid_sample through the reference call
    got = oracle.bilinear_sample_points(torch.from_numpy(v["g4_plane"]), torch.from_numpy(v["g4_p"])[..., :2])
    np.testing.assert_allclose(got.numpy(), v["g4_out"], rtol=1e-6, atol=1e-6)
    assert abs(got[0, 0, 0].item() - 3.9) < 1e-5
    # G-5 interpolate
    t = torch.from_numpy(v["g5_in"])
    assert np.array_equal(oracle.upsample_bilinear_align(t, 6).numpy(), v["g5_same"])
    np.testing.assert_allclose(oracle.upsample_bilinear_align(t, 12).numpy(), v["g5_up"], rtol=1e-6, atol=1e-7)


@pytest.mark.parametrize("name", CASE_NAMES + ["berlin_full", "berlin_image_full", "munich_full", "munich_image_full"])
def test_param_shapes_match_reference(golden_dir, name):
    with open(os.path.join(golden_dir, f"state_dict_{name}.json")) as fh:
        ref = {k: tuple(v) for k, v in json.load(fh).items()}
    if name in CASES:
        cfg = make_cfg(**CASES[name]["cfg"])
    else:
        from tomosar2height_b200.config import berlin_config, munich_config
        cfg = (berlin_config if name.startswith("berlin") else munich_config)(use_image="image" in name)
    assert oracle.reference_param_shapes(cfg) == ref


@pytest.mark.parametrize("aten", [True, False])
@pytest.mark.parametrize("name", CASE_NAMES)
def test_forward_backward_matches_reference(golden_dir, name, aten):
    g = _load(golden_dir, name)
    spec = CASES[name]
    cfg = make_cfg(**spec["cfg"])
    shapes = oracle.reference_param_shapes(cfg)
    P = {k: v.requires_grad_(True) for k, v in oracle.synth_state_dict(shapes, seed=spec["seed"]).items()}
    cloud = torch.from_numpy(g["cloud"])
    image = torch.from_numpy(g["image"]) if "image" in g.files else None
    dsm = torch.from_numpy(g["dsm"])
    trace = {}
    pa, pb = oracle.oracle_forward(P, cfg, cloud, image, aten=aten, trace=trace)
    assert np.array_equal(trace["index"].numpy(), g["index"])  # bit-exact cell ids
    scale = np.abs(g["pa_f32"]).max()
    np.testing.assert_allclose(pa.detach().numpy(), g["pa_f32"], rtol=0, atol=2e-5 * scale)
    if pb is not None:
        np.testing.assert_allclose(pb.detach().numpy(), g["pb_f32"], rtol=0, atol=2e-5 * np.abs(g["pb_f32"]).max())
    loss = oracle.oracle_loss(pa, pb, dsm, cfg.use_footprint)
    assert abs(loss.item() - float(g["loss_f32"])) <= 1e-5 * abs(float(g["loss_f32"]))
    loss.backward()
    names = [str(n) for n in g["param_names"]]
    for k, pname in enumerate(names):
        ref_norm = float(g["grad_norm_f32"][k])
        grad = P[pname].grad
        if ref_norm < 0:  # reference parameter never received a gradient (unused last-UpConv branches)
            assert grad is None or float(grad.abs().max()) == 0.0, pname
            continue
        flat = grad.double().flatten()
        assert abs(flat.norm().item() - ref_norm) <= 2e-4 * max(ref_norm, 1e-6), pname
        pos = grad_probe_positions(flat.numel())
        got = np.asarray([flat[i].item() for i in pos])
        ref = g["grad_probe_f32"][k][: len(pos)]
        np.testing.assert_allclose(got, ref, rtol=0, atol=2e-4 * max(ref_norm / np.sqrt(flat.numel()), 1e-7) * 50, err_msg=pname)


def test_explicit_bilinear_matches_aten():
    """The explicit restatements vs ATen's kernels (the reference's actual dependency)."""
    import torch.nn.functional as F
    g = torch.Generator().manual_seed(3)
    plane = torch.randn(2, 5, 16, 16, generator=g, dtype=torch.float64)
    xy = torch.rand(2, 400, 2, generator=g, dtype=torch.float64)
    xy[0, :4] = torch.tensor([[0.0, 0.0], [1.0, 1.0], [1.0, 0.0], [0.5, 1.0]])
    want = F.grid_sample(plane, (2 * xy - 1)[:, :, None], padding_mode="border", align_corners=True).squeeze(-1)
    torch.testing.assert_close(oracle.bilinear_sample_points(plane, xy), want, rtol=1e-12, atol=1e-12)
    for size in (16, 31, 32, 50):
        want = F.interpolate(plane, size=size, mode="bilinear", align_corners=True)
        torch.testing.assert_close(oracle.upsample_bilinear_align(plane, size), want, rtol=1e-12, atol=1e-12)


def test_scene_pieces_match_reference(golden_dir):
    """oracle/generator.py against outputs of the REAL reference functions (tests/golden/make_golden_scene.py):
    blend windows, strict crop + normalisation, raster index arithmetic, flip / window / accumulate / clamp."""
    import math
    from oracle.generator import blend_window, crop_normalize_tile, raster_col_row, accumulate_scene
    v = np.load(os.path.join(golden_dir, "scene_vectors.npz"))
    ref_windows = {tag: v["window_" + tag] for tag in ("w128", "w9x7", "w16")}
    ref_windows["w512"] = np.outer(v["window_w512_wy"], v["window_w512_wx"])  # stored as its two ramps: same bits
    for tag, shape, hb in (("w128", (128, 128), (0.5, 0.5)), ("w512", (512, 512), (0.5, 0.5)), ("w9x7", (9, 7), (0.3, 0.5)),
                           ("w16", (16, 16), (0.0, 0.25))):
        assert np.array_equal(blend_window(*shape, hb).numpy(), ref_windows[tag]), tag
    pts = torch.from_numpy(v["crop_points"])
    for k in range(2):
        x0, y0 = v[f"crop_anchor_{k}"]
        idx, norm = crop_normalize_tile(pts, float(x0), float(y0), 128.0, 156.5 - (-33.7))
        assert np.array_equal(idx.numpy(), v[f"crop_index_{k}"])       # strict inequalities, both crops
        assert np.array_equal(norm.numpy(), v[f"crop_norm_{k}"])       # same matrix path -> bit-exact float32
    for (x, y), (col, row) in zip(v["raster_query_xy"], v["raster_query_colrow"]):
        assert raster_col_row(float(x), float(y), 386000.0, 5820260.0, 1.0) == (int(col), int(row))
    assert tuple(v["raster_shape"]) == (math.floor(260.0 / 1.0), math.floor(300.0 / 1.0))
    tiles = [torch.from_numpy(t) for t in v["scene_tiles"]]
    dsm, weight = accumulate_scene(tiles, [tuple(a) for a in v["scene_anchors"]], (386000.0, 5820000.0),
                                   (386300.0, 5820260.0), 128.0, 1.0)
    got = torch.maximum(dsm / weight, torch.tensor(0., dtype=torch.float64)).numpy()
    ref = v["scene_dsm"]
    assert np.array_equal(np.isnan(got), np.isnan(ref))                # uncovered pixels stay NaN
    assert np.array_equal(got[~np.isnan(ref)], ref[~np.isnan(ref)])    # same additions in the same order
