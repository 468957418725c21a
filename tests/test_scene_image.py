"""Scene generation with an orthophoto, host side: OrthoImage and SceneGenerator.generate reject bad inputs before
anything is launched, the image windows follow RasterData.query_col_row on the image's own corner, and
t2h_raster_windows refuses bad arguments without a launch.  No GPU needed."""
import os

import numpy as np
import pytest
import torch

import tomosar2height_b200 as t2h
from tomosar2height_b200 import _lib
from tomosar2height_b200.generator import OrthoImage, SceneGenerator
from oracle.generator import raster_col_row
from cases import CASES, make_cfg

LO, HI = [386000.0, 5820000.0], [386300.0, 5820260.0]


def ortho(C=3, left=LO[0] - 7.25, top=HI[1] + 5.5, rows=280, cols=320, px=1.0):
    """an image covering the scene with a margin, its corner a non-integral number of pixels off the scene's"""
    bands = np.random.default_rng(0).standard_normal((C, rows, cols)).astype(np.float32)
    return OrthoImage(bands, left, top, px, [0.1] * C, [2.0] * C, device="cpu")


def model(use_image=True, use_cloud=True):
    cfg = make_cfg(**{**CASES["munich_small"]["cfg"], "use_image": use_image})
    cfg["use_cloud"] = use_cloud
    return t2h.TomoSAR2Height(cfg)


def scene(m, **kw):
    return SceneGenerator(m, LO, HI, (465.5, 599.5), patch_size=128.0, stride=64.0, pixel_size=1.0, **kw)


POINTS = torch.tensor([[LO[0] + 10.0, LO[1] + 10.0, 470.0]], dtype=torch.float64)


def test_ortho_image_rejects_bad_bands_and_normalisation():
    good = np.zeros((3, 8, 8), np.float32)
    with pytest.raises(ValueError, match="float32"):
        OrthoImage(good.astype(np.float64), 0.0, 8.0, 1.0, [0.0] * 3, [1.0] * 3, device="cpu")
    with pytest.raises(ValueError, match="float32"):
        OrthoImage(torch.zeros(3, 8, 8, dtype=torch.float16), 0.0, 8.0, 1.0, [0.0] * 3, [1.0] * 3, device="cpu")
    with pytest.raises(ValueError, match=r"\(C, H, W\)"):
        OrthoImage(good[0], 0.0, 8.0, 1.0, [0.0], [1.0], device="cpu")
    with pytest.raises(ValueError, match="mean and std"):
        OrthoImage(good, 0.0, 8.0, 1.0, [0.0] * 2, [1.0] * 3, device="cpu")
    with pytest.raises(ValueError, match="mean and std"):
        OrthoImage(good, 0.0, 8.0, 1.0, [0.0] * 3, [1.0] * 4, device="cpu")
    with pytest.raises(ValueError, match="std"):
        OrthoImage(good, 0.0, 8.0, 1.0, [0.0] * 3, [1.0, 0.0, 1.0], device="cpu")
    img = OrthoImage(torch.ones(3, 8, 8), 0.0, 8.0, 1.0, [0.0] * 3, [1.0] * 3, device="cpu")
    assert img.bands.dtype == torch.float32 and img.mean.dtype == img.std.dtype == torch.float32


def test_ortho_image_from_raster(tmp_path):
    bands = [np.full((6, 9), i, np.float32) for i in range(3)]
    path = str(tmp_path / "ortho")
    t2h.write_raster(path, bands, (686167.25, 5331627.0), (686176.25, 5331633.5), 0.5, 25832)
    img = OrthoImage.from_raster(path, [1.0, 2.0, 3.0], [4.0, 5.0, 6.0], device="cpu")
    assert (img.left, img.top, img.pixel_size) == (686167.25, 5331633.5, 0.5)
    assert img.bands.shape == (3, 6, 9) and float(img.bands[2, 0, 0]) == 2.0
    assert img.mean.tolist() == [1.0, 2.0, 3.0] and img.std.tolist() == [4.0, 5.0, 6.0]
    t2h.write_raster(path, bands, (0.0, 0.0), (9.0, 6.0), (1.0, 2.0), 25832)   # rectangular pixels
    with pytest.raises(ValueError, match="non-square"):
        OrthoImage.from_raster(path, [0.0] * 3, [1.0] * 3, device="cpu")


def test_generate_rejects_modality_mismatch():
    with pytest.raises(ValueError, match="image branch"):
        scene(model(use_image=True)).generate(POINTS)                     # cloud + image model, no image
    with pytest.raises(ValueError, match="image branch"):
        scene(model(use_image=True, use_cloud=False)).generate(POINTS)    # image-only model, no image
    with pytest.raises(ValueError, match="no image branch"):
        scene(model(use_image=False)).generate(POINTS, image=ortho())     # cloud-only model, an image


def test_generate_rejects_image_that_does_not_fit():
    gen = scene(model())
    with pytest.raises(ValueError, match="pixel size"):
        gen.generate(POINTS, image=ortho(px=0.5))
    with pytest.raises(ValueError, match="bands"):
        gen.generate(POINTS, image=ortho(C=1))
    # one pixel short on every side in turn: the anchors on that edge are not covered
    for kw in (dict(left=LO[0] + 1.0), dict(top=HI[1] - 1.0), dict(cols=306), dict(rows=265)):
        with pytest.raises(ValueError, match="does not cover"):
            gen.generate(POINTS, image=ortho(**kw))


def test_image_windows_follow_query_col_row():
    """The window origin of every tile in the image: RasterData.query_col_row (pinned by the oracle) on the image's
    own corner, which sits 7.25 / 5.5 pixels off the scene's."""
    gen = scene(None)
    img = ortho()
    S = 128
    assert len(gen.anchors) == 16
    for x0, y0 in gen.anchors:
        t_row, l_col = gen.raster_window(x0, y0, img.left, img.top)
        ref_col, _ = raster_col_row(x0 + 0.5, y0 + 0.5, img.left, img.top, 1.0)
        _, ref_row = raster_col_row(x0 + S - 0.5, y0 + S - 0.5, img.left, img.top, 1.0)
        assert (t_row, l_col) == (ref_row, ref_col)
        # against the scene's own raster (tile corners on whole metres): floor(0.5 + 5.5) rows, floor(0.5 + 7.25) columns
        assert (t_row, l_col) == tuple(a + b for a, b in zip(gen.raster_window(x0, y0), (6, 7)))


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build_library()
    return _lib.load()


def test_raster_windows_argument_validation_without_gpu(lib):
    # raster, C, rows, cols, t_row, l_col, n_tiles, S, mean, std, out, stream
    dummy = 16  # any non-null address: nothing is read, the call returns before a launch
    ok = [dummy, 3, 64, 64, dummy, dummy, 2, 16, dummy, dummy, dummy]
    for i in (0, 4, 5, 8, 9, 10):                     # every pointer argument NULL in turn
        args = list(ok)
        args[i] = None
        assert lib.t2h_raster_windows(*args, None) == 1, i
    for i, bad in ((7, 0), (7, -1), (1, 0), (1, -3), (2, 0), (3, 0), (6, -1)):   # S, C, rows, cols, n_tiles
        args = list(ok)
        args[i] = bad
        assert lib.t2h_raster_windows(*args, None) == 1, (i, bad)
    assert lib.t2h_raster_windows(None, 3, 64, 64, None, None, 0, 16, None, None, None, None) == 0   # no tiles
