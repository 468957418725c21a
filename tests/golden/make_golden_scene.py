#!/usr/bin/env python
"""Golden vectors for the scene-inference pieces either side of the model (SURVEY §8f-f2), produced by the REAL
reference code in the build container (needs /root/reference):

    python tests/golden/make_golden_scene.py      ->  tests/golden/scene_vectors.npz

What is executed from the reference, unmodified:
  * utils/crop_cloud.py   crop_pc_2d                     (strict 2-D crop)
  * utils/coordinate.py   apply_transform, invert_transform
  * dataset.py            the normalisation recipe of __getitem__ (:243-278), replayed here line by line with the
                          module's own scale_mat / shift_norm construction (:185-196) -- the class itself needs
                          chunk files on disk
  * utils/io_raster.py    RasterData.set_transform / query_col_row, RasterWriter.cal_dsm_shape
  * generator.py          DSMGenerator._linear_blend_patch_weight and DSMGenerator.generate_dsm (built with
                          object.__new__, a list as data loader and a table-lookup model, so that flip, window,
                          accumulation, division and clamp are the reference's own statements)
Stubs: open3d / laspy / rasterio are IO-only; ``rasterio.transform.Affine`` gets a minimal stand-in for the
axis-aligned case (a, 0, c, 0, e, f) with ``~`` and ``*`` -- the affine package is third-party and absent;
``transformations`` gets identity matrices (no augmentation on the test split: dataset.py:252-262 picks key 0 / -1).
"""
import math
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
REFERENCE = os.environ.get("T2H_REFERENCE", "/root/reference")


class Affine:
    """x' = a*x + c, y' = e*y + f (b = d = 0): the only form io_raster.py:56-62 builds."""

    def __init__(self, a, b, c, d, e, f):
        assert b == 0.0 and d == 0.0
        self.a, self.c, self.e, self.f = float(a), float(c), float(e), float(f)

    def __invert__(self):
        return Affine(1.0 / self.a, 0.0, -self.c / self.a, 0.0, 1.0 / self.e, -self.f / self.e)

    def __mul__(self, xy):
        x, y = xy
        return x * self.a + self.c, y * self.e + self.f


def import_reference():
    class _Anything(types.ModuleType):
        def __getattr__(self, attr):
            if attr.startswith("__"):
                raise AttributeError(attr)
            return _Anything(self.__name__ + "." + attr)

    for name in ("open3d", "rasterio", "rasterio.crs", "rasterio.io", "laspy", "torch_scatter"):
        sys.modules.setdefault(name, _Anything(name))
    rt = types.ModuleType("rasterio.transform")
    rt.Affine = Affine
    sys.modules["rasterio.transform"] = rt
    sys.modules["rasterio"].crs = types.SimpleNamespace(CRS=types.SimpleNamespace(from_epsg=lambda e: e))
    tf = types.ModuleType("transformations")
    tf.rotation_matrix = lambda angle, axis: np.eye(4)
    tf.reflection_matrix = lambda origin, axis: np.eye(4)
    sys.modules["transformations"] = tf
    sys.path.insert(0, REFERENCE)
    from utils.crop_cloud import crop_pc_2d
    from utils.coordinate import apply_transform, invert_transform
    from utils.io_raster import RasterData, RasterWriter
    import generator as ref_generator
    return crop_pc_2d, apply_transform, invert_transform, RasterData, RasterWriter, ref_generator


def main():
    crop_pc_2d, apply_transform, invert_transform, RasterData, RasterWriter, ref_generator = import_reference()
    DSMGenerator = ref_generator.DSMGenerator
    out = {}
    # ---- blend windows (generator.py:85-113) ---------------------------------------------------------------
    for tag, shape, hb in (("w128", (128, 128), [0.5, 0.5]), ("w512", (512, 512), [0.5, 0.5]), ("w9x7", (9, 7), [0.3, 0.5]),
                           ("w16", (16, 16), [0.0, 0.25])):
        out["window_" + tag] = DSMGenerator._linear_blend_patch_weight(shape, hb).numpy()
    # the 512 x 512 window is kept as its two ramps (row and column 255, where the other ramp is 1): their outer product
    # is the window bit for bit, and the file stays small
    w = out.pop("window_w512")
    out["window_w512_wy"], out["window_w512_wx"] = w[:, 255].copy(), w[255].copy()
    assert np.array_equal(np.outer(out["window_w512_wy"], out["window_w512_wx"]), w)
    # ---- crop + normalise (crop_cloud.py:21-29, dataset.py:185-196,243-278) ----------------------------------
    g = torch.Generator().manual_seed(21)
    lo = torch.tensor([386000.0, 5820000.0], dtype=torch.float64)
    pts = torch.rand(4000, 3, generator=g, dtype=torch.float64)
    pts[:, :2] = lo + pts[:, :2] * torch.tensor([300.0, 260.0], dtype=torch.float64)
    pts[:, 2] = 30.0 + pts[:, 2] * 40.0
    pts[:25, 0] = lo[0] + 64.0            # exactly on a tile's lower edge -> excluded by the strict crop
    pts[25:50, 1] = lo[1] + 64.0 + 128.0  # exactly on its upper edge
    patch = torch.tensor([128.0, 128.0, 0.0], dtype=torch.float64)  # TomoSARDataset.patch_size (z unused here)
    z_bound = [-33.7, 156.5]
    x_range = y_range = [0.0, 1.0]
    scale_mat = torch.diag(torch.tensor([patch[0] / (x_range[1] - x_range[0]), patch[1] / (y_range[1] - y_range[0]),
                                         z_bound[1] - z_bound[0], 1], dtype=torch.float64))
    shift_norm = torch.cat([torch.eye(4, 3, dtype=torch.float64),
                            torch.tensor([(x_range[1] - x_range[0]) / 2., (y_range[1] - y_range[0]) / 2., 0, 1]).reshape(-1, 1)], 1)
    out["crop_points"] = pts.numpy()
    for k, anchor in enumerate([[lo[0] + 64.0, lo[1] + 64.0], [lo[0] + 172.0, lo[1] + 132.0]]):
        min_bound = torch.tensor(anchor, dtype=torch.float64)
        max_bound = min_bound + patch[:2]
        inputs, index = crop_pc_2d(pts, min_bound, max_bound)
        z_shift = torch.min(inputs[:, 2]).double().reshape(1)
        transform_mat = scale_mat.clone()
        transform_mat[0:3, 3] = torch.cat([(min_bound + max_bound) / 2., z_shift], 0)
        normalize_mat = shift_norm.double() @ torch.eye(4, dtype=torch.float64) @ torch.eye(4, dtype=torch.float64) \
            @ invert_transform(transform_mat).double()
        inputs_norm = apply_transform(inputs, normalize_mat).float()
        inputs_norm, index2 = crop_pc_2d(inputs_norm, [x_range[0], y_range[0]], [x_range[1], y_range[1]])
        out[f"crop_anchor_{k}"] = min_bound.numpy()
        out[f"crop_index_{k}"] = index.numpy()[index2.numpy()]
        out[f"crop_norm_{k}"] = inputs_norm.numpy()
    # ---- raster index arithmetic (io_raster.py:56-62,78-95,123-131) -------------------------------------------
    bl, tr, px = [386000.0, 5820000.0], [386300.0, 5820260.0], [1.0, 1.0]
    rd = RasterData()
    rd.set_transform(bl_bound=bl, tr_bound=tr, pixel_size=px, crs_epsg=25832)
    q = np.array([[386000.5, 5820000.5], [386063.5, 5820191.5], [386299.5, 5820259.5], [386064.5, 5820064.5]])
    out["raster_query_xy"] = q
    out["raster_query_colrow"] = np.array([rd.query_col_row(x, y) for x, y in q])
    out["raster_shape"] = np.array(RasterWriter.cal_dsm_shape(bl, tr, np.array(px)))
    # ---- generate_dsm (generator.py:115-165) with a table-lookup model -----------------------------------------
    S = 128
    anchors = [(386000.0, 5820000.0), (386064.0, 5820000.0), (386172.0, 5820000.0), (386000.0, 5820064.0),
               (386064.0, 5820064.0), (386172.0, 5820132.0)]
    g = torch.Generator().manual_seed(5)
    tiles = torch.randn(len(anchors), S, S, 1, generator=g) * 20.0   # heights incl. negatives (clamped at 0 afterwards)
    loader = [{"is_valid": [True], "min_bound": torch.tensor([a], dtype=torch.float64),
               "max_bound": torch.tensor([a], dtype=torch.float64) + 128.0, "inputs": torch.tensor([[float(k)]])}
              for k, a in enumerate(anchors)]
    loader.insert(2, {"is_valid": [False]})

    class Lookup(torch.nn.Module):
        def forward(self, input_cloud=None, input_image=None):
            return tiles[int(input_cloud.flatten()[0].item())][None], None

    gen = object.__new__(DSMGenerator)
    gen.model, gen.device, gen.data_loader = Lookup(), "cpu", loader
    gen.pixel_size = torch.tensor(px, dtype=torch.float64)
    gen.crs_epsg, gen.use_cloud, gen.use_image = 25832, True, False
    gen.l_bound, gen.b_bound, gen.r_bound, gen.t_bound = bl[0], bl[1], tr[0], tr[1]
    gen.dsm_shape = RasterWriter.cal_dsm_shape(bl, tr, gen.pixel_size)
    gen.patch_weight = DSMGenerator._linear_blend_patch_weight((S, S), [0.5, 0.5])
    ref_generator.RasterWriter = lambda data: types.SimpleNamespace(write_to_file=lambda path: None, data=data)
    writer = gen.generate_dsm("unused.tif")
    out["scene_anchors"] = np.array(anchors)
    out["scene_tiles"] = tiles.numpy()
    out["scene_dsm"] = writer.data.get_data(1)
    np.savez_compressed(os.path.join(HERE, "scene_vectors.npz"), **out)
    print({k: v.shape for k, v in out.items()})


if __name__ == "__main__":
    main()
