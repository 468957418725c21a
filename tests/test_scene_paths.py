"""Host planning of scene generation (generator.py) and numpy restatements of the scene kernels (t2h_scene.cu).

The restatements below are the references of tests/test_gpu_scene_paths.py.  They repeat the kernels' own
arithmetic one rounded operation at a time, so every comparison there is bit for bit:

- crop: first crop in fp64 with strict inequalities; per tile z_shift = the minimum, by the order-preserving 64-bit
  code, of the z of the first-crop survivors (-0.0 below +0.0, NaN of either sign below everything); then
  fp32((x - x0) / patch), fp32((y - y0) / patch), fp32((z - z_shift) / z_scale) and the second crop on the fp32
  values.  A tile whose z_shift is NaN has no survivors: the reference's normalisation matrix (torch.inverse of a
  transform with a NaN translation) is NaN in every entry, so its re-crop drops every point.
- blend: in tile order, acc = acc + fl(h * fl(wx[j] * wy[i])) with the product and the sum rounded separately.
"""
import math

import numpy as np
import pytest
import torch

import oracle.generator as ogen
from tomosar2height_b200.generator import SceneGenerator, blend_vectors, linear_blend_weight

SIGN = np.uint64(1 << 63)
NO_SURVIVOR = np.uint64(0xFFFFFFFFFFFFFFFF)   # tile_zmin fill: no first-crop survivor
ITEM = np.dtype([("tile", "<i4"), ("count", "<i4"), ("first", "<i8")])   # CropItem, 16 bytes


# =====================================================================================================
# references
# =====================================================================================================
def encode_f64(z):
    """order-preserving uint64 code of fp64 values (t2h_common.cuh); NaN of either sign -> 0"""
    z = np.ascontiguousarray(z, dtype=np.float64)
    b = z.view(np.uint64)
    code = np.where((b & SIGN) != 0, ~b, b | SIGN)
    return np.where(np.isnan(z), np.uint64(0), code)


def decode_f64(code):
    code = np.atleast_1d(np.asarray(code, dtype=np.uint64))
    return np.where((code & SIGN) != 0, code & ~SIGN, ~code).view(np.float64)


def first_crop(x, y, x0, y0, patch):
    x0, y0, patch = np.float64(x0), np.float64(y0), np.float64(patch)
    return (x > x0) & (x < x0 + patch) & (y > y0) & (y < y0 + patch)


def second_crop(nx, ny):
    return (nx > 0) & (nx < 1) & (ny > 0) & (ny < 1)


def pack_items(items):
    """(tile, count, first) triples -> the int32 (n, 4) words {tile, count, first_lo, first_hi} crop_tiles builds"""
    return torch.tensor([(t, c, f & 0xFFFFFFFF, f >> 32) for t, c, f in items], dtype=torch.int64).to(torch.int32)


def normalise(q, x0, y0, z_shift, patch, z_scale):
    """(k, 4) float32 rows fp32((x - x0) / patch), fp32((y - y0) / patch), fp32((z - z_shift) / z_scale), +0.0"""
    v = np.zeros((len(q), 4), dtype=np.float32)
    with np.errstate(invalid="ignore", over="ignore"):
        v[:, 0] = ((q[:, 0] - np.float64(x0)) / np.float64(patch)).astype(np.float32)
        v[:, 1] = ((q[:, 1] - np.float64(y0)) / np.float64(patch)).astype(np.float32)
        v[:, 2] = ((q[:, 2] - np.float64(z_shift)) / np.float64(z_scale)).astype(np.float32)
    return v


def crop_reference(pts, items, tile_xy, patch, z_scale, base=0):
    """t2h_tile_count + t2h_tile_write for work items (tile, count, first); ``pts`` holds rows base.. of the cloud.
    Returns (item_count (n_items,) int64, tile_zmin (n_tiles,) uint64 codes, rows: per item the (k, 4) float32 rows it
    writes, in candidate order).  item_count counts the survivors of both crops whatever z_shift is; the items of a
    tile whose z_shift is NaN (code 0) write nothing."""
    zmin = np.full(len(tile_xy), NO_SURVIVOR)
    kept = []
    for t, c, f in items:
        p = pts[f - base:f - base + c]
        m = first_crop(p[:, 0], p[:, 1], *tile_xy[t], patch)
        if m.any():
            zmin[t] = min(zmin[t], encode_f64(p[m, 2]).min())
        kept.append(p[m])
    z_shift = decode_f64(zmin)
    counts, rows = [], []
    for (t, _, _), q in zip(items, kept):
        v = normalise(q, *tile_xy[t], z_shift[t], patch, z_scale)
        keep = second_crop(v[:, 0], v[:, 1])
        counts.append(int(keep.sum()))
        rows.append(v[:0] if zmin[t] == 0 else v[keep])
    return np.array(counts, dtype=np.int64), zmin, rows


def bin_order(pts, l, b, stride, nx, ny):
    """the binned order of SceneGenerator._bin: a stable sort of the points by stride cell (clamped to the grid)"""
    cx = np.clip(np.floor((pts[:, 0] - l) / stride), 0, nx - 1).astype(np.int64)
    cy = np.clip(np.floor((pts[:, 1] - b) / stride), 0, ny - 1).astype(np.int64)
    return np.argsort(cy * nx + cx, kind="stable")


def scene_crop_reference(pts, order, anchors, patch, z_scale):
    """crop_tiles of a whole scene: per tile, the survivors of the binned cloud ``pts[order]`` in binned order.
    Returns (per-tile float32 (k, 4) rows, per-tile indices into ``pts``)."""
    binned = pts[order]
    out, idx = [], []
    for x0, y0 in anchors:
        m = np.nonzero(first_crop(binned[:, 0], binned[:, 1], x0, y0, patch))[0]
        zmin = encode_f64(binned[m, 2]).min(initial=NO_SURVIVOR)
        if zmin == 0 or len(m) == 0:
            out.append(np.zeros((0, 4), np.float32))
            idx.append(np.zeros(0, np.int64))
            continue
        v = normalise(binned[m], x0, y0, decode_f64(zmin)[0], patch, z_scale)
        keep = second_crop(v[:, 0], v[:, 1])
        out.append(v[keep])
        idx.append(order[m[keep]])
    return out, idx


def blend_reference(dsm, weight, heights, t_row, l_col, wx, wy, r0, c0, box_rows, box_cols):
    """t2h_blend_accumulate: for the raster pixels of the box, in tile order, dsm += fl(h[S-1-i, j] * fl(wx[j] * wy[i]))
    and weight += fl(wx[j] * wy[i]), each product and sum rounded on its own (numpy does not contract)."""
    dsm, weight = dsm.copy(), weight.copy()
    n_rows, n_cols = dsm.shape
    S = heights.shape[1]
    w = wy[:, None] * wx[None, :]
    for k in range(len(t_row)):
        h = heights[k, ::-1, :].astype(np.float64)
        t, c = int(t_row[k]), int(l_col[k])
        ra, rb = max(t, r0, 0), min(t + S, r0 + box_rows, n_rows)
        ca, cb = max(c, c0, 0), min(c + S, c0 + box_cols, n_cols)
        if ra >= rb or ca >= cb:
            continue
        i, j = slice(ra - t, rb - t), slice(ca - c, cb - c)
        dsm[ra:rb, ca:cb] = dsm[ra:rb, ca:cb] + h[i, j] * w[i, j]
        weight[ra:rb, ca:cb] = weight[ra:rb, ca:cb] + w[i, j]
    return dsm, weight


def blend_hits(shape, t_row, l_col, S, r0, c0, box_rows, box_cols):
    """pixels of the raster that some tile of the batch writes"""
    hit = np.zeros(shape, dtype=bool)
    inbox = np.zeros(shape, dtype=bool)
    inbox[max(r0, 0):max(r0 + box_rows, 0), max(c0, 0):max(c0 + box_cols, 0)] = True
    for t, c in zip(t_row, l_col):
        hit[max(t, 0):max(t + S, 0), max(c, 0):max(c + S, 0)] = True
    return hit & inbox


# =====================================================================================================
# self-tests of the references
# =====================================================================================================
def test_encode_orders_doubles_and_sends_nan_to_zero():
    vals = np.array([-np.inf, -1e300, -1.0, -5e-324, -0.0, 0.0, 5e-324, 1.0, 1e300, np.inf])
    codes = encode_f64(vals)
    assert np.all(codes[1:] > codes[:-1]) and codes[0] > 0
    assert np.array_equal(decode_f64(codes).view(np.uint64), vals.view(np.uint64))
    nans = np.array([0x7FF8000000000000, 0xFFF8000000000000, 0x7FF0000000000001, 0xFFFFFFFFFFFFFFFF],
                    dtype=np.uint64).view(np.float64)
    assert np.all(encode_f64(nans) == 0) and np.isnan(decode_f64(0)[0])
    # the fill of tile_zmin is no code of a non-NaN double
    assert NO_SURVIVOR > encode_f64(np.array([np.inf]))[0]


def test_crop_reference_matches_oracle_at_power_of_two_patches():
    """The restatement against the pinned reference crop (oracle.crop_normalize_tile): for patch sizes 128, 256 and
    512 the (p - min) / patch of the kernels equals the reference's 4x4 matrix product bit for bit, ulp-edge points
    included; this is what makes the GPU comparison with the oracle exact."""
    g = np.random.default_rng(4)
    for patch in (128.0, 256.0, 512.0):
        x0, y0 = 386000.0 + patch, 5820000.0 + 2 * patch
        pts = np.column_stack([x0 - 3 + g.random(4000) * (patch + 6), y0 - 3 + g.random(4000) * (patch + 6),
                               30.0 + g.random(4000) * 40.0])
        pts[:8, 0] = [x0, x0 + patch, np.nextafter(x0, np.inf), np.nextafter(x0 + patch, -np.inf)] * 2
        pts[8:16, 1] = [y0, y0 + patch, np.nextafter(y0, np.inf), np.nextafter(y0 + patch, -np.inf)] * 2
        _, _, rows = crop_reference(pts, [(0, len(pts), 0)], [(x0, y0)], patch, 190.2)
        idx, norm = ogen.crop_normalize_tile(torch.from_numpy(pts), x0, y0, patch, 190.2)
        assert np.array_equal(rows[0][:, :3].view(np.uint32), norm.numpy().view(np.uint32)), patch


def test_oracle_drops_every_point_of_a_tile_with_nan_z():
    """The reference's behaviour the kernels follow: one NaN z among the first-crop survivors, of either sign, makes
    the normalisation matrix NaN and the tile empty."""
    g = np.random.default_rng(5)
    pts = np.column_stack([g.random(500) * 128.0, g.random(500) * 128.0, g.random(500)])
    for bits in (0x7FF8000000000000, 0xFFF8000000000000):
        p = pts.copy()
        p[7, 2] = np.array([bits], dtype=np.uint64).view(np.float64)[0]
        idx, norm = ogen.crop_normalize_tile(torch.from_numpy(p), 0.0, 0.0, 128.0, 10.0)
        assert len(idx) == 0 and norm.shape[0] == 0
        counts, zmin, rows = crop_reference(p, [(0, 500, 0)], [(0.0, 0.0)], 128.0, 10.0)
        assert zmin[0] == 0 and counts[0] > 0 and len(rows[0]) == 0


def test_blend_reference_matches_oracle_accumulation():
    """blend_reference with the product window is oracle.accumulate_scene's slice-add for in-raster windows"""
    g = np.random.default_rng(6)
    S = 8
    wx, wy = (v.numpy() for v in blend_vectors(S, S))
    heights = g.standard_normal((3, S, S)).astype(np.float32)
    dsm, weight = np.zeros((20, 30)), np.zeros((20, 30))
    rows, cols = [0, 4, 12], [0, 22, 5]
    got, got_w = blend_reference(dsm, weight, heights, rows, cols, wx, wy, 0, 0, 20, 30)
    ref, ref_w = np.zeros((20, 30)), np.zeros((20, 30))
    win = ogen.blend_window(S, S).numpy()
    for k in range(3):
        ref[rows[k]:rows[k] + S, cols[k]:cols[k] + S] += torch.from_numpy(heights[k])[None].flip(1).squeeze().double().numpy() * win
        ref_w[rows[k]:rows[k] + S, cols[k]:cols[k] + S] += win
    assert np.array_equal(got, ref) and np.array_equal(got_w, ref_w)


# =====================================================================================================
# blend vectors
# =====================================================================================================
@pytest.mark.parametrize("shape", [(1, 1), (2, 2), (3, 3), (7, 7), (8, 8), (128, 128), (129, 129), (7, 9), (12, 5)])
@pytest.mark.parametrize("half_blend", [(0.5, 0.5), (0.25, 0.4), (0.3, 0.7), (0.0, 0.5), (1.0, 1.0)])
def test_blend_vectors_match_window(shape, half_blend):
    n_rows, n_cols = shape
    if math.floor(n_rows * half_blend[0]) > n_cols or math.floor(n_cols * half_blend[1]) > n_rows:
        pytest.skip("the reference cannot build this window (ramp longer than the axis)")
    wx, wy = blend_vectors(n_rows, n_cols, half_blend)
    assert wx.shape == (n_cols,) and wy.shape == (n_rows,)
    prod = (wy[:, None] * wx[None, :]).numpy()
    for ref in (linear_blend_weight(n_rows, n_cols, half_blend), ogen.blend_window(n_rows, n_cols, half_blend)):
        assert np.array_equal(prod.view(np.uint64), ref.numpy().view(np.uint64))


# =====================================================================================================
# host planning: binning, tile cells, work items
# =====================================================================================================
LO = (386000.25, 5820000.5)

# (extent x, extent y, patch, stride, pixel size): patch / stride 1, 2, 3 and 1.5, extents that are no multiple of the
# stride or the pixel size (last anchor off the bin grid), a scene smaller than one patch
SCENES = [
    (300.0, 260.0, 64.0, 64.0, 1.0),
    (300.3, 260.7, 128.0, 64.0, 0.5),
    (333.3, 250.1, 96.0, 32.0, 0.3),
    (401.7, 199.9, 96.0, 64.0, 0.7),
    (50.5, 40.25, 64.0, 32.0, 0.25),
]


def scene_points(ex, ey, patch, seed, n=40000):
    """points over the scene plus a margin of half a patch on every side (they fall into the clamped border bins),
    points on every anchor line and one fp64 ulp either side of it"""
    g = np.random.default_rng(seed)
    m = patch / 2
    pts = np.column_stack([LO[0] - m + g.random(n) * (ex + 2 * m), LO[1] - m + g.random(n) * (ey + 2 * m),
                           30.0 + g.random(n) * 40.0])
    return pts


def add_anchor_edges(pts, gen, seed):
    """points exactly on the anchor lines and tile ends of ``gen`` and one ulp either side"""
    g = np.random.default_rng(seed)
    xs = sorted({a[0] for a in gen.anchors} | {a[0] + gen.patch for a in gen.anchors})
    ys = sorted({a[1] for a in gen.anchors} | {a[1] + gen.patch for a in gen.anchors})
    rows = []
    for v in xs:
        for e in (np.nextafter(v, -np.inf), v, np.nextafter(v, np.inf)):
            rows.append((e, gen.b + g.random() * (gen.t - gen.b), 30.0 + 40.0 * g.random()))
    for v in ys:
        for e in (np.nextafter(v, -np.inf), v, np.nextafter(v, np.inf)):
            rows.append((gen.l + g.random() * (gen.r - gen.l), e, 30.0 + 40.0 * g.random()))
    return np.concatenate([pts, np.array(rows)])


def make_scene(k, n=40000):
    ex, ey, patch, stride, px = SCENES[k]
    gen = SceneGenerator(None, LO, (LO[0] + ex, LO[1] + ey), (-33.7, 156.5), patch_size=patch, stride=stride,
                         pixel_size=px)
    return gen, add_anchor_edges(scene_points(ex, ey, patch, 10 + k, n), gen, 20 + k)


@pytest.mark.parametrize("k", range(len(SCENES)))
def test_work_items_cover_every_first_crop_survivor_once(k):
    gen, pts = make_scene(k)
    (binned, starts, nx, ny), _ = gen._bin(torch.from_numpy(pts))
    binned = binned.numpy()
    assert nx * ny + 1 == len(starts) and starts[-1] == len(pts)
    items = gen._work_items(gen.anchors, starts, nx, ny)
    assert all(1 <= c <= 1024 for _, c, _, _ in items)
    if SCENES[k][0] < SCENES[k][2]:
        assert len(gen.anchors) == 1 and gen.anchors[0][0] < gen.l   # the single tile reaches past the scene
    for t, (x0, y0) in enumerate(gen.anchors):
        mine = [(c, lo + (hi << 32)) for tt, c, lo, hi in items if tt == t]
        # the tile's cell ranges, one per bin row, each cut into consecutive items of 1024 rows (the last shorter)
        cx0, cx1, cy0, cy1 = gen._tile_cells(x0, y0, nx, ny)
        want = []
        for cy in range(cy0, cy1 + 1):
            a, b = starts[cy * nx + cx0], starts[cy * nx + cx1 + 1]
            want += [(min(1024, b - f), f) for f in range(a, b, 1024)]
        assert mine == want, (t, x0, y0)
        covered = np.zeros(len(binned), dtype=np.int64)
        for c, f in mine:
            covered[f:f + c] += 1
        assert covered.max(initial=0) <= 1   # no candidate row twice: it would be written twice
        inside = first_crop(binned[:, 0], binned[:, 1], x0, y0, gen.patch)
        assert inside.any() and np.all(covered[inside] == 1), (t, x0, y0, int((covered[inside] == 0).sum()))


def test_work_items_pack_offsets_beyond_32_bits():
    """first = 2^31 - 1, 2^31 and 2^32 + 5 survive _work_items -> int32 words -> the 16-byte CropItem"""
    gen = SceneGenerator(None, (0.0, 0.0), (40.0, 40.0), (0.0, 1.0), patch_size=10.0, stride=10.0)
    nx, ny = gen._grid()
    assert (nx, ny) == (4, 4)
    counts = [0] * 16
    counts[0:4] = [1, 2, 3, 2 ** 31 - 7]   # starts[4] = 2^31 - 1
    counts[4:7] = [1, 1030, 2]             # starts[5] = 2^31
    counts[7] = 2 ** 32 + 5 - (2 ** 31 + 1032)   # starts[10] = 2^32 + 5
    counts[10], counts[14], counts[15] = 5, 1, 1
    starts = [0] + np.cumsum(counts).tolist()
    todo = [(0.0, 0.0), (10.0, 0.0), (20.0, 20.0)]
    items = gen._work_items(todo, starts, nx, ny)
    want = [(0, 3, 0), (0, 1024, 2 ** 31 - 1), (0, 7, 2 ** 31 + 1023),
            (1, 5, 1), (1, 1024, 2 ** 31), (1, 8, 2 ** 31 + 1024),
            (2, 5, 2 ** 32 + 5), (2, 2, 2 ** 32 + 10)]
    assert [(t, c, lo + (hi << 32)) for t, c, lo, hi in items] == want
    words = torch.tensor(items, dtype=torch.int64).to(torch.int32).contiguous()   # as crop_tiles uploads them
    assert torch.equal(words, pack_items(want))
    rec = words.numpy().view(ITEM).reshape(-1)
    assert rec.itemsize == 16 and rec.shape == (len(want),)
    assert [(int(r["tile"]), int(r["count"]), int(r["first"])) for r in rec] == want
    assert int(words[4, 2]) < 0   # the low word of 2^31 is negative as an int32
