"""Whole-scene nDSM generation on the device (SURVEY §8f rank f2).

Restates the inference pipeline of the reference -- regular tile anchors (dataset.py:160-181), strict 2-D
crop (utils/crop_cloud.py:21-29), per-tile normalisation with the local z minimum (dataset.py:243-278,
conf/dataset/base.yaml:18-22), model forward, vertical flip, separable linear blend window and
weighted accumulation into float64 scene rasters (generator.py:85-113,127-157) -- with the points
resident in HBM: the scene cloud is binned once by stride-sized cells (one sort), every tile gathers its
candidates from <= 9 contiguous cell ranges instead of scanning the whole chunk on the CPU
(dataset.py:234), and tiles with different point counts are batched as a ``RaggedCloud``.
No collective is needed: with several GPUs every rank generates a block of the tile list into its own
partial rasters (``tile_range``), which are summed afterwards.
Models with the image branch get, per batch, the normalised orthophoto windows of the tiles, cut on the device
from an ``OrthoImage`` that stays resident (t2h_raster_windows).
"""
import math

import numpy as np
import torch

from .topology import RaggedCloud


class OrthoImage:
    """An orthophoto on the device, the image input of scene generation.

    ``bands`` (C, H, W) float32, row 0 = northern edge (the layout of ``read_raster`` / ``write_raster``); ``left``,
    ``top`` the world coordinates of its upper-left corner and ``pixel_size`` its (square) pixel edge; ``mean`` /
    ``std`` the per-channel normalisation of the training images (dataset.py:111-113): a window is fed to the model as
    (band - mean) / std."""

    def __init__(self, bands, left, top, pixel_size, mean, std, device="cuda"):
        if not isinstance(bands, torch.Tensor):
            bands = np.asarray(bands)
            if bands.dtype != np.float32:
                raise ValueError(f"OrthoImage: bands must be float32, got {bands.dtype}")
            bands = torch.from_numpy(bands)
        elif bands.dtype != torch.float32:
            raise ValueError(f"OrthoImage: bands must be float32, got {bands.dtype}")
        if bands.dim() != 3:
            raise ValueError(f"OrthoImage: bands must be (C, H, W), got shape {tuple(bands.shape)}")
        C = bands.shape[0]
        mean = torch.as_tensor(mean, dtype=torch.float32).flatten()
        std = torch.as_tensor(std, dtype=torch.float32).flatten()
        if mean.numel() != C or std.numel() != C:
            raise ValueError(f"OrthoImage: mean and std need {C} values (one per band), got {mean.numel()} and {std.numel()}")
        if bool((std == 0).any()):
            raise ValueError("OrthoImage: std must not be 0")
        self.bands = bands.to(device).contiguous()
        self.left, self.top, self.pixel_size = float(left), float(top), float(pixel_size)
        self.mean, self.std = mean.to(device), std.to(device)

    @classmethod
    def from_raster(cls, path, mean, std, device="cuda"):
        """Read a ``write_raster`` container (``path.npy`` + ``path.json``): corner and pixel size from its affine
        (px, 0, left, 0, -px, top)."""
        from .adapters import read_raster
        bands, meta = read_raster(path)
        a, b, left, d, e, top = meta["transform"]
        if b != 0.0 or d != 0.0 or a != -e:
            raise ValueError(f"OrthoImage.from_raster: {path} is rotated or has non-square pixels ({meta['transform']})")
        return cls(bands, left, top, a, mean, std, device)


def regular_anchors(lo, hi, patch, stride):
    """dataset.py:165-170: arange(lo, hi - patch, stride) plus the last anchor hi - patch."""
    out, v = [], lo
    while v < hi - patch:
        out.append(v)
        v += stride
    out.append(hi - patch)
    return out


def linear_blend_weight(n_rows, n_cols, half_blend=(0.5, 0.5), min_weight=1e-3, device="cpu"):
    """generator.py:85-113: separable ramp min_weight -> 1 -> min_weight, float64 (n_rows, n_cols)."""
    wx = torch.ones(n_rows, n_cols, dtype=torch.float64, device=device)
    wy = torch.ones(n_rows, n_cols, dtype=torch.float64, device=device)
    ix, iy = math.floor(n_rows * half_blend[0]), math.floor(n_cols * half_blend[1])
    if ix > 0:
        wx[:, :ix] = torch.linspace(min_weight, 1, ix, dtype=torch.float64, device=device)
        wx[:, -ix:] = torch.linspace(1, min_weight, ix, dtype=torch.float64, device=device)
    if iy > 0:
        wy[:iy, :] = torch.linspace(min_weight, 1, iy, dtype=torch.float64, device=device)[:, None]
        wy[-iy:, :] = torch.linspace(1, min_weight, iy, dtype=torch.float64, device=device)[:, None]
    return wx * wy


def blend_vectors(n_rows, n_cols, half_blend=(0.5, 0.5), min_weight=1e-3, device="cpu"):
    """The two 1-D ramps of generator.py:85-113: (wx over the columns, wy over the rows); the window is wy[:, None] * wx."""
    wx = torch.ones(n_cols, dtype=torch.float64, device=device)
    wy = torch.ones(n_rows, dtype=torch.float64, device=device)
    ix, iy = math.floor(n_rows * half_blend[0]), math.floor(n_cols * half_blend[1])
    if ix > 0:
        wx[:ix] = torch.linspace(min_weight, 1, ix, dtype=torch.float64, device=device)
        wx[-ix:] = torch.linspace(1, min_weight, ix, dtype=torch.float64, device=device)
    if iy > 0:
        wy[:iy] = torch.linspace(min_weight, 1, iy, dtype=torch.float64, device=device)
        wy[-iy:] = torch.linspace(1, min_weight, iy, dtype=torch.float64, device=device)
    return wx, wy


class SceneGenerator:
    """DSMGenerator.generate_dsm (generator.py:115-165) with the scene resident in HBM.

    One sort bins the cloud by stride-sized cells; ONE pair of kernels crops and normalises the points of every
    tile of the scene (t2h_tile_count / t2h_tile_write) with a single host read of the per-tile counts; the tiles
    then run through the model in ragged batches (views of that one buffer, no per-tile host work) and every batch
    is flipped, windowed and accumulated into the float64 rasters by t2h_blend_accumulate."""

    def __init__(self, model, scene_min, scene_max, z_bound, patch_size=512.0, stride=256.0, pixel_size=1.0,
                 half_blend=(0.5, 0.5), tiles_per_batch=4):
        self.model = model
        self.l, self.b = float(scene_min[0]), float(scene_min[1])
        self.r, self.t = float(scene_max[0]), float(scene_max[1])
        self.patch, self.stride, self.px = float(patch_size), float(stride), float(pixel_size)
        self.z_scale = float(z_bound[1] - z_bound[0])
        self.tiles_per_batch = tiles_per_batch
        # RasterWriter.cal_dsm_shape (utils/io_raster.py:78-95)
        self.n_rows = math.floor((self.t - self.b) / self.px)
        self.n_cols = math.floor((self.r - self.l) / self.px)
        xs = regular_anchors(self.l, self.r, self.patch, self.stride)
        ys = regular_anchors(self.b, self.t, self.patch, self.stride)
        self.anchors = [(x, y) for y in ys for x in xs]  # meshgrid order of dataset.py:171-172
        self.half_blend = half_blend

    # -- binning: one sort of the scene cloud by stride-sized cell --------------------------------------
    def _grid(self):
        nx = max(int(math.ceil((self.r - self.l) / self.stride)), 1)
        ny = max(int(math.ceil((self.t - self.b) / self.stride)), 1)
        return nx, ny

    def _tile_cells(self, x0, y0, nx, ny):
        """bin cells (cx0..cx1, cy0..cy1) a tile overlaps"""
        x1, y1 = x0 + self.patch, y0 + self.patch
        cx0 = min(max(int(math.floor((x0 - self.l) / self.stride)), 0), nx - 1)
        cx1 = min(max(int(math.floor((x1 - self.l) / self.stride)), 0), nx - 1)
        cy0 = min(max(int(math.floor((y0 - self.b) / self.stride)), 0), ny - 1)
        cy1 = min(max(int(math.floor((y1 - self.b) / self.stride)), 0), ny - 1)
        return cx0, cx1, cy0, cy1

    def _bin(self, pts64, rank=None, world=None):
        """Histogram of the cloud over the stride cells (one pass), then a stable sort by cell of the points this rank
        needs: with ``world`` ranks the tile list is split into contiguous blocks balanced by candidate points (from the
        histogram: identical on every rank, no communication) and only the cell rows this rank's tiles overlap are sorted.
        Returns ((binned points, bin starts (host list), nx, ny), tile_range or None)."""
        from .parallel import shard_tiles_weighted
        nx, ny = self._grid()
        cx = ((pts64[:, 0] - self.l) / self.stride).floor().clamp(0, nx - 1).long()
        cy = ((pts64[:, 1] - self.b) / self.stride).floor().clamp(0, ny - 1).long()
        cell = cy * nx + cx
        counts = torch.bincount(cell, minlength=nx * ny)
        tile_range = None
        if world is not None:
            acc = [0] + counts.cumsum(0).tolist()
            tile_range = shard_tiles_weighted(self.tile_weights(acc, nx, ny), rank, world)
            rows = [self._tile_cells(*self.anchors[i], nx, ny) for i in tile_range]
            cy_lo = min((r[2] for r in rows), default=0)
            cy_hi = max((r[3] for r in rows), default=-1)
            keep = (cy >= cy_lo) & (cy <= cy_hi)
            pts64, cell = pts64[keep], cell[keep]
            inside = torch.zeros(ny, dtype=torch.bool, device=counts.device)
            inside[cy_lo:cy_hi + 1] = True
            counts = counts * inside.repeat_interleave(nx)
        order = torch.argsort(cell, stable=True)
        starts = [0] + counts.cumsum(0).tolist()
        return (pts64[order].contiguous(), starts, nx, ny), tile_range

    def _work_items(self, todo, starts, nx, ny):
        """Candidate row ranges of every tile (the bin cells it overlaps), cut into <= 1024-row work items."""
        items = []
        for t, (x0, y0) in enumerate(todo):
            cx0, cx1, cy0, cy1 = self._tile_cells(x0, y0, nx, ny)
            for cy in range(cy0, cy1 + 1):
                first, last = starts[cy * nx + cx0], starts[cy * nx + cx1 + 1]
                for f in range(first, last, 1024):
                    items.append((t, min(1024, last - f), f & 0xFFFFFFFF, f >> 32))
        return items

    def tile_weights(self, starts, nx, ny):
        """candidate points of every tile of the scene (from the bin table): the work estimate for sharding"""
        w = []
        for (x0, y0) in self.anchors:
            cx0, cx1, cy0, cy1 = self._tile_cells(x0, y0, nx, ny)
            w.append(sum(starts[cy * nx + cx1 + 1] - starts[cy * nx + cx0] for cy in range(cy0, cy1 + 1)))
        return w

    def crop_tiles(self, points, todo, binned=None):
        """Strict crop + normalisation of every tile in ``todo`` (a list of anchors) in two launches.
        Returns (flat (P, 4) fp32 rows (x, y, z, 0), per-tile counts as a python list)."""
        from . import _lib
        dev = points.device
        binned, starts, nx, ny = self._bin(points.double())[0] if binned is None else binned
        items = self._work_items(todo, starts, nx, ny)
        n_items, n_tiles = len(items), len(todo)
        if n_items == 0:
            return torch.empty(0, 4, device=dev), [0] * n_tiles
        items_h = torch.tensor(items, dtype=torch.int64)
        items_d = items_h.to(torch.int32).to(dev).contiguous()  # {tile, count, first_lo, first_hi}: 16 bytes per item
        tile_xy = torch.tensor(todo, dtype=torch.float64, device=dev).contiguous()
        item_count = torch.empty(n_items, dtype=torch.int32, device=dev)
        zmin = torch.full((n_tiles,), -1, dtype=torch.int64, device=dev)
        _lib.call("t2h_tile_count", _lib.ptr(binned), _lib.ptr(items_d), n_items, _lib.ptr(tile_xy), self.patch,
                  _lib.ptr(item_count), _lib.ptr(zmin))
        counts64 = item_count.long()
        item_offset = (counts64.cumsum(0) - counts64).contiguous()
        per_tile = torch.zeros(n_tiles, dtype=torch.int64, device=dev).index_add_(0, items_h[:, 0].to(dev), counts64)
        counts = per_tile.tolist()  # the one host read of the scene
        out = torch.empty(sum(counts), 4, dtype=torch.float32, device=dev)
        _lib.call("t2h_tile_write", _lib.ptr(binned), _lib.ptr(items_d), n_items, _lib.ptr(tile_xy), self.patch, self.z_scale,
                  _lib.ptr(item_offset), _lib.ptr(zmin), _lib.ptr(out))
        return out, counts

    def raster_window(self, x0, y0, left=None, top=None):
        """generator.py:139-154 with RasterData.query_col_row (io_raster.py:123-131): (t_row, l_col) of a tile in the
        output raster, or in a raster of the same pixel size whose upper-left corner is (left, top)."""
        left = self.l if left is None else left
        top = self.t if top is None else top
        l_col = math.floor((x0 + self.px / 2 - left) / self.px)
        t_row = math.floor((top - (y0 + self.patch - self.px / 2)) / self.px)
        return t_row, l_col

    def _check_inputs(self, points, image):
        """Host-side checks of the modalities and the orthophoto, before anything is launched."""
        use_image = bool(getattr(self.model, "use_image", False))
        if use_image and image is None:
            raise ValueError("generate: the model has the image branch (use_image); pass image=OrthoImage(...)")
        if image is None:
            return
        if not use_image:
            raise ValueError("generate: an image was passed but the model has no image branch (use_image is false)")
        if image.pixel_size != self.px:
            raise ValueError(f"generate: image pixel size {image.pixel_size} != output pixel size {self.px}")
        C, H, W = image.bands.shape
        if C != self.model.image_encoder.in_channels:
            raise ValueError(f"generate: image has {C} bands, the image encoder takes {self.model.image_encoder.in_channels}")
        if image.bands.device != points.device:
            raise ValueError(f"generate: image on {image.bands.device}, points on {points.device}")
        S = int(round(self.patch / self.px))
        for x0, y0 in self.anchors:
            t_row, l_col = self.raster_window(x0, y0, image.left, image.top)
            if t_row < 0 or l_col < 0 or t_row + S > H or l_col + S > W:
                raise ValueError(f"generate: the image ({H} x {W} pixels from ({image.left}, {image.top})) does not cover "
                                 f"the tile at ({x0}, {y0}): window rows {t_row}..{t_row + S - 1}, columns {l_col}..{l_col + S - 1}")

    @torch.no_grad()
    def generate(self, points, image=None, tile_range=None, rank=None, world=None):
        """points (P, 3) world coordinates on the device (float64 recommended for geo-coordinates); ``image`` an
        ``OrthoImage`` on the same device, required by models with the image branch (tiles without points are skipped
        whatever the modality, as the dataset marks them invalid: dataset.py:235-241).
        Returns (dsm (n_rows, n_cols) float64, weight float64); with ``tile_range`` (or ``rank`` / ``world``: a
        contiguous block of the tile list balanced by candidate points, identical on every rank without
        communication) the un-normalised partial sums of that block of tiles -- sum the partials of all ranks, then
        ``finalize``."""
        from . import _lib
        self._check_inputs(points, image)
        dev = points.device
        if tile_range is None and world is not None:
            binned, tile_range = self._bin(points.double(), rank, world)
            self.last_tile_range = tile_range
        else:
            binned, _ = self._bin(points.double())
        todo = list(self.anchors if tile_range is None else [self.anchors[i] for i in tile_range])
        flat, counts = self.crop_tiles(points, todo, binned)
        dsm = torch.zeros(self.n_rows, self.n_cols, dtype=torch.float64, device=dev)
        weight = torch.zeros_like(dsm)
        S = int(round(self.patch / self.px))
        wx, wy = blend_vectors(S, S, self.half_blend, device=dev)
        # non-empty tiles in anchor order (empty tiles are skipped: generator.py:133), their point ranges, windows
        live = [t for t, c in enumerate(counts) if c > 0]
        starts, acc = [], 0
        for c in counts:
            starts.append(acc)
            acc += c
        win = [self.raster_window(*todo[t]) for t in live]
        t_rows = torch.tensor([w[0] for w in win], dtype=torch.int32, device=dev)
        l_cols = torch.tensor([w[1] for w in win], dtype=torch.int32, device=dev)
        bounds = torch.tensor([starts[t] for t in live] + [0], dtype=torch.int64, device=dev)
        if image is not None:
            # the tiles' orthophoto windows: the same arithmetic on the image's own corner
            img_win = [self.raster_window(*todo[t], image.left, image.top) for t in live]
            img_rows = torch.tensor([w[0] for w in img_win], dtype=torch.int32, device=dev)
            img_cols = torch.tensor([w[1] for w in img_win], dtype=torch.int32, device=dev)
            C, H, W = image.bands.shape
            windows = torch.empty(self.tiles_per_batch, S, S, C, dtype=torch.float32, device=dev)
        use_cloud = bool(getattr(self.model, "use_cloud", True))
        self.model.eval()
        for k in range(0, len(live), self.tiles_per_batch):
            tiles = live[k:k + self.tiles_per_batch]
            nb = len(tiles)
            p0, p1 = starts[tiles[0]], starts[tiles[-1]] + counts[tiles[-1]]
            # live tiles are contiguous in the flat buffer (empty ones hold no rows); offsets relative to the batch
            offsets = torch.cat([bounds[k:k + nb] - p0, bounds.new_tensor([p1 - p0])])
            cloud = RaggedCloud(flat[p0:p1], offsets) if use_cloud else None
            img = None
            if image is not None:
                _lib.call("t2h_raster_windows", _lib.ptr(image.bands), C, H, W, _lib.ptr(img_rows[k:k + nb]),
                          _lib.ptr(img_cols[k:k + nb]), nb, S, _lib.ptr(image.mean), _lib.ptr(image.std), _lib.ptr(windows))
                img = windows[:nb].permute(0, 3, 1, 2)  # channels-last memory, the NCHW view the image encoder takes
            heights = self.model(input_cloud=cloud, input_image=img)[0]  # (B, S, S, 1)
            rows = [w[0] for w in win[k:k + nb]]
            cols = [w[1] for w in win[k:k + nb]]
            r0, c0 = min(rows), min(cols)
            _lib.call("t2h_blend_accumulate", _lib.ptr(heights.contiguous()), nb, S, _lib.ptr(t_rows[k:k + nb]),
                      _lib.ptr(l_cols[k:k + nb]), _lib.ptr(wx), _lib.ptr(wy), r0, c0, max(rows) + S - r0, max(cols) + S - c0,
                      self.n_rows, self.n_cols, _lib.ptr(dsm), _lib.ptr(weight))
        if tile_range is not None:
            return dsm, weight
        return self.finalize(dsm, weight), weight

    @staticmethod
    def finalize(dsm_sum, weight_sum):
        """generator.py:156-157: divide by the accumulated weight, clamp at 0 (uncovered pixels stay NaN)."""
        return torch.maximum(dsm_sum / weight_sum, torch.zeros((), dtype=dsm_sum.dtype, device=dsm_sum.device))
