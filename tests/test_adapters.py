"""Config / IO adapters (f4): the Hydra-free loader against a replica of the structure of the reference's conf/
tree, the chunk reader and the raster container."""
import numpy as np
import pytest
import yaml

import tomosar2height_b200 as t2h
from tomosar2height_b200.adapters import ChunkCloud, load_config, read_raster, write_raster


def _replica(tmp_path):
    """Same composition features as the reference tree: defaults list with _self_ first, _global_ group files, a group
    option with its own defaults, interpolation."""
    conf = tmp_path / "conf"
    (conf / "model").mkdir(parents=True)
    (conf / "dataset").mkdir()
    (conf / "config.yaml").write_text(
        "defaults:\n  - _self_\n  - model: tomosar2height\n  - dataset: munich\n  - override hydra/job_logging: custom\n"
        "use_cloud: true\nuse_image: false\ngpu_id: 0\nhydra:\n  verbose: false\n")
    (conf / "model" / "tomosar2height.yaml").write_text(
        "# @package _global_\nmodel:\n  encoder: pointnet_local_pool\n  encoder_kwargs:\n    hidden_dim: 32\n    feature_dim: 32\n"
        "    plane_resolution: 256\n    scatter_type: max\n    unet_type: alto\n    unet_kwargs: {depth: 5, merge_mode: concat, start_filts: 32}\n"
        "  encoder2: unet\n  encoder2_kwargs: {num_classes: 32, in_channels: 3, depth: 6, merge_mode: concat, start_filts: 32}\n"
        "  decoder_pixel_kwargs:\n    mode: conv\n    use_footprint: ${use_footprint}\n    hidden_dim: 32\n    out_dim: 1\n"
        "    sample_mode: bilinear\n    leaky: false\n  data_dim: 3\ntest:\n  threshold: 0.5\n  check_point: ./outputs/${test.run_name}/model_best.pt\n")
    (conf / "dataset" / "base.yaml").write_text(
        "# @package _global_\ndataset:\n  normalize: {x_range: [0., 1.], y_range: [0., 1.], z_shift: local_min}\n  patch_size: [512, 512]\n")
    (conf / "dataset" / "berlin.yaml").write_text(
        "# @package _global_\ndefaults:\n  - base\nuse_footprint: false\ntest: {run_name: T-berlin}\ndataset:\n  name: berlin\n  normalize:\n    z_bound: [-33.7, 156.5]\n")
    (conf / "dataset" / "munich.yaml").write_text(
        "# @package _global_\ndefaults:\n  - base\nuse_footprint: true\nmodel:\n  encoder_kwargs:\n    unet_kwargs:\n      depth: 6\n"
        "test: {run_name: T-munich}\ndataset:\n  name: munich\n  normalize:\n    z_bound: [465.5, 599.5]\n")
    return str(conf)


@pytest.mark.parametrize("source", ["replica"])
def test_load_config_composes_like_hydra(tmp_path, source):
    conf = _replica(tmp_path)
    cfg = load_config(conf)  # defaults: model tomosar2height, dataset munich
    assert cfg.dataset.name == "munich" and cfg.use_footprint is True
    assert cfg.model.encoder_kwargs.unet_kwargs.depth == 6                      # munich.yaml overrides the model group
    assert cfg.model.decoder_pixel_kwargs.use_footprint is True                 # ${use_footprint}, typed
    assert cfg["dataset"]["normalize"]["z_bound"] == [465.5, 599.5] and cfg.dataset.normalize.z_shift == "local_min"
    assert "hydra" not in cfg and cfg.use_cloud is True and cfg.use_image is False
    assert cfg.test.check_point.endswith("/model_best.pt") and "${" not in cfg.test.check_point
    b = load_config(conf, ["dataset=berlin", "use_image=true", "model.encoder_kwargs.unet_kwargs.depth=4"])
    assert b.dataset.name == "berlin" and b.use_image is True and b.use_footprint is False
    assert b.model.encoder_kwargs.unet_kwargs.depth == 4 and b.model.decoder_pixel_kwargs.use_footprint is False
    # the composed tree equals the hard-coded mirrors the benchmarks use, on every key the model reads
    for got, want in ((load_config(conf, ["dataset=berlin"]), t2h.berlin_config()), (cfg, t2h.munich_config())):
        assert {k: got.model[k] for k in want.model if k != "name"} == {k: want.model[k] for k in want.model if k != "name"}
        assert got.dataset.normalize.z_bound == want.dataset.normalize.z_bound
        assert (got.use_cloud, got.use_image, got.use_footprint) == (want.use_cloud, want.use_image, want.use_footprint)
        model = t2h.TomoSAR2Height(got)    # the model constructs from the loaded tree
        assert model.z_scale == want.dataset.normalize.z_bound[1] - want.dataset.normalize.z_bound[0]


def test_chunk_cloud_and_raster_container(tmp_path):
    root = tmp_path / "generated"
    info = {}
    rng = np.random.default_rng(0)
    for idx, (x0, y0) in enumerate([(686167.0, 5331627.0), (688430.0, 5331627.0)]):
        name = f"chunk_{idx:02d}"
        (root / name).mkdir(parents=True)
        pts = rng.random((100, 3)) * [2263.0, 1910.0, 60.0] + [x0, y0, 465.5]
        np.savez(root / name / "input_point_cloud.npz", pts=pts.astype(np.float32 if idx else np.float64))
        info[idx] = {"name": name, "min_bound": [x0, y0, 465.5], "max_bound": [x0 + 2263.0, y0 + 1910.0, 525.5]}
    with open(root / "chunk_info.yaml", "w") as fh:
        yaml.safe_dump(info, fh)
    cc = ChunkCloud(str(root))
    lo, hi = cc.bounds()
    assert lo == [686167.0, 5331627.0] and hi == [688430.0 + 2263.0, 5331627.0 + 1910.0]
    assert cc.all_points().shape == (200, 3) and cc.all_points().dtype == np.float64
    assert ChunkCloud(str(root), [1]).all_points().shape == (100, 3)
    dsm = rng.random((5, 7))
    meta = write_raster(str(tmp_path / "ndsm"), dsm, lo, hi, [1.0, 1.0], 25832)
    arr, meta2 = read_raster(str(tmp_path / "ndsm"))
    assert meta == meta2 and arr.shape == (1, 5, 7) and arr.dtype == np.float32
    assert meta["transform"] == [1.0, 0.0, lo[0], 0.0, -1.0, hi[1]] and meta["crs_epsg"] == 25832
    np.testing.assert_allclose(arr[0], dsm.astype(np.float32))
