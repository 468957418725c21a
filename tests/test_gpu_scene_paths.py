"""The scene crop, normalisation and blend kernels (t2h_scene.cu) against exact references at every edge.

t2h_tile_count / t2h_tile_write (strict crop, local z minimum, normalisation, re-crop) and t2h_blend_accumulate
(flip, blend window, fp64 accumulation) produce every pixel of a generated nDSM.  They are compared bit for bit
with the numpy restatements of tests/test_scene_paths.py, called directly through the C ABI on hand-built work
items (item lengths around the 256-thread rounds and the 1024-row chunk, tiles spread over interleaved items,
points on and one ulp inside the tile edges, NaN / inf coordinates, z of every sign class, offsets beyond 2^31)
and through SceneGenerator on the host-planned scenes.  Outputs of direct calls are pre-filled with NaN (the
item counts with 0x7fc0dead, the rasters with a NaN payload), so that a value a kernel writes where it must not,
or fails to write, changes the comparison; the comparison is also what shows that the kernel ran.  The profiler
is only asked whether calls without work launched nothing: it keeps a GPU record only if the record's timestamp,
converted to the host clock, falls inside its window, and once the process has left the device idle that conversion
can be off by more than 0.2 s, so a kernel that did run can be missing from the list (Kineto counts it as
'Out-of-range'), while a kernel that did not run is never in it.

The agreement with the reference crop itself (oracle.crop_normalize_tile, pinned to the real reference code)
is exact for power-of-two patch sizes; for other sizes the kernels' (p - min) / patch and the reference's 4x4
matrix product differ by at most 2^-24 in absolute terms.
"""
from fractions import Fraction

import numpy as np
import pytest
import torch

import oracle.generator as ogen
from test_scene_paths import (LO, NO_SURVIVOR, SCENES, add_anchor_edges, bin_order, blend_hits, blend_reference,
                              crop_reference, decode_f64, make_scene, pack_items, scene_crop_reference,
                              scene_points)
from tomosar2height_b200 import _lib
from tomosar2height_b200.generator import SceneGenerator

pytestmark = pytest.mark.gpu

Z_SCALE = 156.5 + 33.7
SENTINEL_I32 = 0x7FC0DEAD
NAN_PAYLOAD = 0x7FF8DEADBEEF0001
U24 = 2.0 ** -24
SCENE_KERNELS = ("tile_count_kernel", "tile_write_kernel", "blend_accumulate_kernel")


# =====================================================================================================
# helpers
# =====================================================================================================
def launched(fn):
    """run fn under the profiler; the set of kernel names it reported (spaces removed): a subset of the kernels fn
    launched, see the module docstring"""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name.replace(" ", "") for e in prof.events()}


def same_f32(a, b):
    """bit for bit, except that any NaN equals any NaN (inf - inf is the canonical NaN on the device, the host's
    default NaN carries the sign bit)"""
    a, b = np.asarray(a, dtype=np.float32), np.asarray(b, dtype=np.float32)
    return a.shape == b.shape and bool(np.all((a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))))


def f64(bits):
    return np.array([bits], dtype=np.uint64).view(np.float64)[0]


def run_crop(pts_d, items, tile_xy, patch, z_scale=Z_SCALE):
    """t2h_tile_count then t2h_tile_write on hand-built items; the scan between them is crop_tiles' (the items of a tile
    with code 0 counted as 0).  Returns (item_count, tile_zmin codes, out with one NaN sentinel row past the end)."""
    words = pack_items(items).cuda()
    txy = torch.tensor(tile_xy, dtype=torch.float64, device="cuda")
    n = len(items)
    item_count = torch.full((n,), SENTINEL_I32, dtype=torch.int32, device="cuda")
    zmin = torch.full((len(tile_xy),), -1, dtype=torch.int64, device="cuda")
    _lib.call("t2h_tile_count", _lib.ptr(pts_d), _lib.ptr(words), n, _lib.ptr(txy), patch, _lib.ptr(item_count),
              _lib.ptr(zmin))
    counts = item_count.long().masked_fill(zmin[words[:, 0].long()] == 0, 0)
    offset = (counts.cumsum(0) - counts).contiguous()
    out = torch.full((int(counts.sum()) + 1, 4), float("nan"), dtype=torch.float32, device="cuda")
    _lib.call("t2h_tile_write", _lib.ptr(pts_d), _lib.ptr(words), n, _lib.ptr(txy), patch, z_scale, _lib.ptr(offset),
              _lib.ptr(zmin), _lib.ptr(out))
    return item_count.cpu().numpy(), zmin.cpu().numpy().view(np.uint64), out.cpu().numpy()


def check_crop(pts, items, tile_xy, patch, z_scale=Z_SCALE, pts_d=None, base=0):
    """run_crop against crop_reference: item counts, tile_zmin codes and every output row in item order, bit for bit"""
    if pts_d is None:
        pts_d = torch.from_numpy(pts).cuda()
    got_count, got_zmin, out = run_crop(pts_d, items, tile_xy, patch, z_scale)
    ref_count, ref_zmin, rows = crop_reference(pts, items, tile_xy, patch, z_scale, base)
    assert np.array_equal(got_count, ref_count), (got_count, ref_count)   # every 0x7fc0dead slot was written
    assert np.array_equal(got_zmin, ref_zmin), (got_zmin, ref_zmin)
    want = np.concatenate(rows)
    assert out.shape[0] == len(want) + 1
    assert same_f32(out[:-1], want)
    assert np.all(out[:-1, 3].view(np.uint32) == 0)    # column 3 is +0.0
    assert np.all(np.isnan(out[-1]))                   # nothing written past the end
    return ref_count, ref_zmin, rows


class Cloud:
    """a cloud built from runs of points; returns the first row of every run"""

    def __init__(self, seed):
        self.g = np.random.default_rng(seed)
        self.parts, self.n = [], 0

    def add(self, rows):
        first = self.n
        self.parts.append(np.asarray(rows, dtype=np.float64).reshape(-1, 3))
        self.n += len(self.parts[-1])
        return first

    def run(self, x0, y0, patch, mask, z=None):
        """len(mask) points: inside the tile where mask, left of it elsewhere"""
        c = len(mask)
        u = 0.001 + 0.998 * self.g.random((c, 2))
        x = np.where(mask, x0 + u[:, 0] * patch, x0 - 1.0 - 5.0 * u[:, 0])
        y = y0 + u[:, 1] * patch
        z = 30.0 + 40.0 * self.g.random(c) if z is None else z
        return self.add(np.column_stack([x, y, z]))

    def array(self):
        return np.concatenate(self.parts)


PATTERNS = {
    "all": lambda i, c: np.ones(c, bool),
    "none": lambda i, c: np.zeros(c, bool),
    "alternate": lambda i, c: i % 2 == 0,
    "single": lambda i, c: i == min(17, c - 1),
    "last_round": lambda i, c: i >= ((c - 1) // 256) * 256,   # survivors only in the last 256-row round
}


# =====================================================================================================
# 1. crop and normalise through the C ABI
# =====================================================================================================
def test_crop_item_lengths_and_survivor_patterns():
    """items of 1 .. 1024 candidates with every survivor pattern, each tile spread over several items listed out of
    order and interleaved with the other tiles, one candidate range shared by two tiles"""
    cloud = Cloud(1)
    tiles = [(386000.0 + 64.0 * k, 5820000.0 + 32.0 * k) for k in range(5)]   # overlapping tiles
    patch = 128.0
    items = []
    for b, c in enumerate((1, 31, 32, 255, 256, 257, 1023, 1024)):
        for p, pat in enumerate(PATTERNS.values()):
            t = (p + b) % len(tiles)
            items.append((t, c, cloud.run(*tiles[t], patch, pat(np.arange(c), c))))
    t, c, f = items[-1]
    items.append(((t + 1) % len(tiles), c, f))   # the same rows, cropped by an overlapping tile
    items = [items[i] for i in np.random.default_rng(2).permutation(len(items))]
    pts = cloud.array()
    counts, zmin, _ = check_crop(pts, items, tiles, patch)
    assert all(zmin[t] not in (0, NO_SURVIVOR) for t in range(len(tiles)))
    assert sum(counts) > 5000


@pytest.mark.parametrize("patch", [100.0, 128.0])
def test_crop_tile_edges(patch):
    """points on the four edges (excluded), one fp64 ulp inside (kept by the first crop; at the upper edges the
    normalised value rounds to 1.0f and the second crop drops it, while its z still sets z_shift), NaN and +-inf x / y"""
    x0, y0 = 386000.0, 5820000.0
    x1, y1 = x0 + patch, y0 + patch
    xm, ym = x0 + 0.37 * patch, y0 + 0.61 * patch
    edge = [(x0, ym), (x1, ym), (xm, y0), (xm, y1),
            (np.nextafter(x0, np.inf), ym), (np.nextafter(x1, -np.inf), ym),
            (xm, np.nextafter(y0, np.inf)), (xm, np.nextafter(y1, -np.inf)),
            (np.nan, ym), (np.inf, ym), (-np.inf, ym), (xm, np.nan), (xm, np.inf), (xm, -np.inf),
            (f64(0xFFF8000000000000), ym)]
    cloud = Cloud(3)
    g = np.random.default_rng(4)
    z = 30.0 + 40.0 * g.random(len(edge))
    z[5] = 1.5   # the lowest z of the tile, on a point that only the second crop drops
    z[0] = 1.0   # lower still, exactly on x0: outside the strict first crop, so it must not become z_shift
    f_edge = cloud.add(np.column_stack([np.array(edge), z]))
    f_bulk = cloud.run(x0, y0, patch, np.ones(300, bool))
    items = [(0, 300, f_bulk), (0, len(edge), f_edge)]
    counts, zmin, rows = check_crop(cloud.array(), items, [(x0, y0)], patch)
    assert decode_f64(zmin[0])[0] == 1.5
    assert counts[1] == 2   # the two lower-edge ulp points
    kept = rows[1]
    assert np.all(kept[:, :2] > 0) and np.all(kept[:, :2] < 1) and kept[:, :2].min() < 1e-10


Z_CASES = {
    "negative": lambda g, n: -50.0 + 40.0 * g.random(n),
    "mixed": lambda g, n: -40.0 + 80.0 * g.random(n),
    "signed_zeros": lambda g, n: np.where(np.arange(n) % 3 == 0, -0.0, np.where(np.arange(n) % 3 == 1, 0.0, g.random(n))),
    "plus_zero": lambda g, n: np.where(np.arange(n) % 2 == 0, 0.0, g.random(n)),
    "huge": lambda g, n: np.array([1e300, -1e300, 9.9e299, -9.9e299, -1.7e308])[np.arange(n) % 5],
    "plus_inf": lambda g, n: np.where(np.arange(n) % 4 == 0, np.inf, g.random(n)),
    "all_plus_inf": lambda g, n: np.full(n, np.inf),
    "minus_inf": lambda g, n: np.where(np.arange(n) % 4 == 0, -np.inf, g.random(n)),
    "nan_positive": lambda g, n: np.where(np.arange(n) == n - 3, f64(0x7FF8000000000000), g.random(n)),
    "nan_negative": lambda g, n: np.where(np.arange(n) == n - 3, f64(0xFFF8000000000000), g.random(n)),
    "no_first_crop_survivor": lambda g, n: g.random(n),
}


def test_crop_z_classes():
    """z_shift over negative, mixed, signed-zero, huge, infinite and NaN z, every tile split over two items that are
    interleaved with the other tiles' (the minimum of one tile comes from either item)"""
    cloud = Cloud(5)
    g = np.random.default_rng(6)
    names = list(Z_CASES)
    tiles = [(386000.0 + 130.0 * k, 5820000.0) for k in range(len(names))]
    first, second = [], []
    for t, name in enumerate(names):
        n = 300
        z = Z_CASES[name](g, n)
        mask = np.ones(n, bool) if name != "no_first_crop_survivor" else np.zeros(n, bool)
        f = cloud.run(*tiles[t], 128.0, mask, z)
        first.append((t, 140, f))
        second.append((t, n - 140, f + 140))
    items = first + second[::-1]
    counts, zmin, rows = check_crop(cloud.array(), items, tiles, 128.0)
    zs = dict(zip(names, decode_f64(zmin)))
    assert zs["signed_zeros"].view(np.uint64) == f64(0x8000000000000000).view(np.uint64)   # -0.0, not +0.0
    assert zs["plus_zero"].view(np.uint64) == 0 and zs["huge"] == -1.7e308
    assert zs["all_plus_inf"] == np.inf and zs["minus_inf"] == -np.inf
    for name in ("nan_positive", "nan_negative"):
        t = names.index(name)
        assert zmin[t] == 0 and counts[t] + counts[len(names) + len(names) - 1 - t] == 300   # counted, then dropped
    assert zmin[names.index("no_first_crop_survivor")] == NO_SURVIVOR
    # the z of a -0.0 point shifted by -0.0 is +0.0; by a wrong +0.0 shift it would be -0.0
    t = names.index("signed_zeros")
    z_out = np.concatenate([rows[t], rows[len(names) + len(names) - 1 - t]])[:, 2]
    assert np.sum(z_out == 0) == 200 and np.all(z_out[z_out == 0].view(np.uint32) == 0)


# =====================================================================================================
# 2. host planning on the device: crop_tiles and sharding
# =====================================================================================================
@pytest.mark.parametrize("k", range(len(SCENES)))
def test_crop_tiles_matches_reference(k):
    gen, pts = make_scene(k)
    nx, ny = gen._grid()
    flat, counts = gen.crop_tiles(torch.from_numpy(pts).cuda(), gen.anchors)
    ref, _ = scene_crop_reference(pts, bin_order(pts, gen.l, gen.b, gen.stride, nx, ny), gen.anchors, gen.patch,
                                  gen.z_scale)
    assert counts == [len(r) for r in ref]
    assert sum(counts) > 0 and same_f32(flat.cpu().numpy(), np.concatenate(ref))


@pytest.mark.parametrize("world", [2, 3, 5])
def test_sharded_bins_give_the_same_tiles(world):
    """the binned subset of _bin(rank, world) gives every tile of the rank's range the rows of the unsharded bin"""
    gen, pts = make_scene(2)
    P = torch.from_numpy(pts).cuda()
    flat, counts = gen.crop_tiles(P, gen.anchors)
    starts = np.cumsum([0] + counts)
    owned = []
    for rank in range(world):
        binned, tr = gen._bin(P.double(), rank, world)
        f, c = gen.crop_tiles(P, [gen.anchors[i] for i in tr], binned)
        assert binned[0].shape[0] < P.shape[0] or world == 1
        assert c == counts[tr.start:tr.stop]
        assert torch.equal(f.view(torch.int32), flat[starts[tr.start]:starts[tr.stop]].view(torch.int32))
        owned += list(tr)
    assert owned == list(range(len(gen.anchors)))


# =====================================================================================================
# 4. agreement with the reference crop
# =====================================================================================================
@pytest.mark.parametrize("patch,stride", [(128.0, 64.0), (256.0, 128.0), (512.0, 256.0), (100.0, 50.0), (153.6, 76.8)])
def test_crop_agrees_with_reference_crop(patch, stride):
    """Power-of-two patches: the same survivors with bit-identical coordinates as oracle.crop_normalize_tile.
    Other patches: the same survivors, every coordinate within 2^-24 absolute (near 0 that is millions of ulps)."""
    ex, ey = 2.5 * patch + 0.3, 2.2 * patch + 0.7
    gen = SceneGenerator(None, LO, (LO[0] + ex, LO[1] + ey), (-33.7, 156.5), patch_size=patch, stride=stride)
    pts = add_anchor_edges(scene_points(ex, ey, patch, 30, n=30000), gen, 31)
    nx, ny = gen._grid()
    flat, counts = gen.crop_tiles(torch.from_numpy(pts).cuda(), gen.anchors)
    ref_rows, ref_idx = scene_crop_reference(pts, bin_order(pts, gen.l, gen.b, stride, nx, ny), gen.anchors, patch,
                                             Z_SCALE)
    assert same_f32(flat.cpu().numpy(), np.concatenate(ref_rows))   # so ref_idx are the points of the kernel's rows
    P = torch.from_numpy(pts)
    exact = patch in (128.0, 256.0, 512.0)
    worst = 0.0
    for t, (x0, y0) in enumerate(gen.anchors):
        idx, norm = ogen.crop_normalize_tile(P, x0, y0, patch, Z_SCALE)
        assert norm is not None and counts[t] == len(idx) > 0, (t, counts[t], len(idx))
        order = np.argsort(ref_idx[t])
        assert np.array_equal(ref_idx[t][order], idx.numpy()), t   # the same survivors
        got, want = ref_rows[t][order, :3], norm.numpy()
        if exact:
            assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), t
        worst = max(worst, float(np.abs(got.astype(np.float64) - want).max()))
    assert worst <= U24 and (exact or worst > 0)


def test_nan_z_drops_the_tile_like_the_reference():
    """One NaN z of either sign empties every tile whose first crop holds it, as in the reference (its normalisation
    matrix is NaN); the other tiles are unchanged.  Before NaN was mapped to code 0 a positive NaN was ignored."""
    gen, pts = make_scene(0, n=20000)
    P = torch.from_numpy(pts).cuda()
    _, base_counts = gen.crop_tiles(P, gen.anchors)
    bad = pts.copy()
    a = gen.anchors
    hit = []
    for k, bits in ((0, 0x7FF8000000000000), (len(a) - 1, 0xFFF8000000000000)):
        x0, y0 = a[k]
        i = int(np.nonzero((bad[:, 0] > x0 + 5) & (bad[:, 0] < x0 + 20) & (bad[:, 1] > y0 + 5) & (bad[:, 1] < y0 + 20))[0][0])
        bad[i, 2] = f64(bits)
        hit.append(i)
    flat, counts = gen.crop_tiles(torch.from_numpy(bad).cuda(), gen.anchors)
    Q = torch.from_numpy(bad)
    emptied = 0
    for t, (x0, y0) in enumerate(a):
        idx, norm = ogen.crop_normalize_tile(Q, x0, y0, gen.patch, gen.z_scale)
        holds = any(x0 < bad[i, 0] < x0 + gen.patch and y0 < bad[i, 1] < y0 + gen.patch for i in hit)
        assert counts[t] == len(idx) == (0 if holds else base_counts[t]), t
        emptied += holds
    assert emptied >= 2 and not np.isnan(flat.cpu().numpy()).any()
    nx, ny = gen._grid()
    ref, _ = scene_crop_reference(bad, bin_order(bad, gen.l, gen.b, gen.stride, nx, ny), a, gen.patch, gen.z_scale)
    assert same_f32(flat.cpu().numpy(), np.concatenate(ref))


# =====================================================================================================
# 3. blend
# =====================================================================================================
def fma_differs(h, w, acc):
    """some (h, w, acc) whose fused multiply-add rounds differently from fl(acc + fl(h * w))"""
    for a, b, c in zip(h, w, acc):
        exact = float(Fraction(float(a)) * Fraction(float(b)) + Fraction(float(c)))
        if exact != float(c) + float(a) * float(b):
            return True
    return False


def blend_case(S, shape, origins, box, seed):
    """(dsm0, weight0, heights, wx, wy): hit pixels random finite, all others a NaN payload; wx != wy.  The first term
    added to the raster is made one whose fused multiply-add rounds differently from the separate product and sum."""
    g = np.random.default_rng(seed)
    t_row, l_col = [o[0] for o in origins], [o[1] for o in origins]
    hit = blend_hits(shape, t_row, l_col, S, *box)
    nan = np.full(shape, NAN_PAYLOAD, dtype=np.uint64).view(np.float64)
    dsm0 = np.where(hit, g.standard_normal(shape) * 10.0, nan)
    w0 = np.where(hit, g.random(shape), nan)
    heights = (g.standard_normal((len(origins), S, S)) * 30.0 + 5.0).astype(np.float32)
    wx, wy = g.uniform(1e-3, 1.0, S), g.uniform(1e-3, 1.0, S)
    for k, (t, c) in enumerate(origins):   # the first tile that hits the box, at its first hit pixel
        win = hit[max(t, 0):max(t + S, 0), max(c, 0):max(c + S, 0)]
        if win.any():
            r, q = np.argwhere(win)[0] + (max(t, 0), max(c, 0))
            i, j = r - t, q - c
            h, w = heights[k, S - 1 - i, j], wx[j] * wy[i]
            for _ in range(1000):   # an accumulator of the product's size: about one try in eight differs
                dsm0[r, q] = 0.7 * float(h) * w
                if fma_differs([h], [w], [dsm0[r, q]]):
                    break
                h = np.nextafter(h, np.float32(np.inf), dtype=np.float32)
            heights[k, S - 1 - i, j] = h
            break
    return dsm0, w0, heights, wx, wy


def run_blend(dsm0, w0, heights, t_row, l_col, wx, wy, batches):
    """t2h_blend_accumulate over consecutive batches [(start, end, r0, c0, box_rows, box_cols), ...]"""
    dsm, weight = torch.from_numpy(dsm0).cuda(), torch.from_numpy(w0).cuda()
    h = torch.from_numpy(heights).cuda()
    tr = torch.tensor(t_row, dtype=torch.int32, device="cuda")
    lc = torch.tensor(l_col, dtype=torch.int32, device="cuda")
    wxd, wyd = torch.from_numpy(wx).cuda(), torch.from_numpy(wy).cuda()
    S = heights.shape[1]
    for a, b, r0, c0, br, bc in batches:
        _lib.call("t2h_blend_accumulate", _lib.ptr(h[a:b].contiguous()), b - a, S, _lib.ptr(tr[a:b]), _lib.ptr(lc[a:b]),
                  _lib.ptr(wxd), _lib.ptr(wyd), r0, c0, br, bc, dsm.shape[0], dsm.shape[1], _lib.ptr(dsm), _lib.ptr(weight))
    return dsm.cpu().numpy(), weight.cpu().numpy()


def union_box(t_row, l_col, S):
    r0, c0 = min(t_row), min(l_col)
    return r0, c0, max(t_row) + S - r0, max(l_col) + S - c0


def blend_origins(S, n_rows, n_cols):
    """windows over every edge and corner, the centre three times, one window outside the raster: 12 tiles"""
    o = max(S // 2, 1)
    rows = (-o, (n_rows - S) // 2, n_rows - S + o)
    cols = (-o, (n_cols - S) // 2, n_cols - S + o)
    out = [(r, c) for r in rows for c in cols]
    centre = out[4]
    return out[:5] + [centre, centre] + out[5:] + [(n_rows + 2, -S - 3)]


BLEND_CASES = [(S, shape) for S, shape in
               [(1, (5, 8)), (2, (9, 6)), (3, (11, 14)), (7, (20, 33)), (128, (300, 211)), (129, (211, 300)),
                (1, (1, 1)), (3, (1, 1))]]


@pytest.mark.parametrize("S,shape", BLEND_CASES)
def test_blend_matches_reference(S, shape):
    n_rows, n_cols = shape
    if shape == (1, 1):
        origins = [(0, 0), (1 - S, 1 - S), (0, 1 - S), (0, 0), (-S, 0)][:5 if S > 1 else 2] + [(0, 0)]
    else:
        origins = blend_origins(S, n_rows, n_cols)
    t_row, l_col = [o[0] for o in origins], [o[1] for o in origins]
    r0, c0, br, bc = union_box(t_row, l_col, S)
    box = (r0 - 2, c0 - 3, br + 5, bc + 4)   # negative corner, larger than the union of the windows
    assert box[0] < 0 and box[1] < 0
    dsm0, w0, heights, wx, wy = blend_case(S, shape, origins, box, seed=S * 1000 + n_rows)
    ref, ref_w = blend_reference(dsm0, w0, heights, t_row, l_col, wx, wy, *box)
    n = len(origins)
    m = n // 2
    splits = [[(0, n, *box)],
              [(k, k + 1, *union_box(t_row[k:k + 1], l_col[k:k + 1], S)) for k in range(n)],
              [(0, m, *union_box(t_row[:m], l_col[:m], S)), (m, n, *union_box(t_row[m:], l_col[m:], S))]]
    for batches in splits:
        got, got_w = run_blend(dsm0, w0, heights, t_row, l_col, wx, wy, batches)
        assert np.array_equal(got.view(np.uint64), ref.view(np.uint64)), len(batches)
        assert np.array_equal(got_w.view(np.uint64), ref_w.view(np.uint64)), len(batches)
    hit = blend_hits(shape, t_row, l_col, S, *box)
    assert hit.any() and np.all(ref[~hit].view(np.uint64) == NAN_PAYLOAD)
    assert np.all(ref_w[hit] > w0[hit])   # every hit pixel changes: the match above needs the kernel to have run
    # the data can tell a fused multiply-add from the separately rounded product and sum
    r, c = np.nonzero(hit)
    k = next(k for k in range(n) if np.any((r >= t_row[k]) & (r < t_row[k] + S) & (c >= l_col[k]) & (c < l_col[k] + S)))
    sel = (r >= t_row[k]) & (r < t_row[k] + S) & (c >= l_col[k]) & (c < l_col[k] + S)
    i, j = r[sel] - t_row[k], c[sel] - l_col[k]
    assert fma_differs(heights[k, S - 1 - i, j], wx[j] * wy[i], dsm0[r[sel], c[sel]])


def test_blend_batch_sizes_1_to_12():
    S, shape = 7, (20, 33)
    origins = blend_origins(S, *shape)
    t_row, l_col = [o[0] for o in origins], [o[1] for o in origins]
    for n in range(1, 13):
        box = union_box(t_row[:n], l_col[:n], S)
        dsm0, w0, heights, wx, wy = blend_case(S, shape, origins[:n], box, seed=n)
        ref, ref_w = blend_reference(dsm0, w0, heights, t_row[:n], l_col[:n], wx, wy, *box)
        got, got_w = run_blend(dsm0, w0, heights, t_row[:n], l_col[:n], wx, wy, [(0, n, *box)])
        assert np.array_equal(got.view(np.uint64), ref.view(np.uint64)), n
        assert np.array_equal(got_w.view(np.uint64), ref_w.view(np.uint64)), n


# =====================================================================================================
# 6. launches
# =====================================================================================================
def test_empty_work_launches_nothing():
    d = torch.full((4, 4), 7.0, dtype=torch.float64, device="cuda")
    w = torch.full((4, 4), 1.0, dtype=torch.float64, device="cuda")
    h = torch.ones(1, 2, 2, device="cuda")
    i32 = torch.zeros(1, dtype=torch.int32, device="cuda")
    v = torch.ones(2, dtype=torch.float64, device="cuda")

    def calls():
        _lib.call("t2h_tile_count", None, None, 0, None, 128.0, None, None)
        _lib.call("t2h_tile_write", None, None, 0, None, 128.0, 1.0, None, None, None)
        _lib.call("t2h_blend_accumulate", None, 0, 2, None, None, None, None, 0, 0, 4, 4, 4, 4, None, None)
        for br, bc in ((0, 4), (4, 0)):
            _lib.call("t2h_blend_accumulate", _lib.ptr(h), 1, 2, _lib.ptr(i32), _lib.ptr(i32), _lib.ptr(v), _lib.ptr(v),
                      0, 0, br, bc, 4, 4, _lib.ptr(d), _lib.ptr(w))
    names = launched(calls)
    assert not [n for n in names if any(k in n for k in SCENE_KERNELS)], sorted(names)
    assert bool((d == 7.0).all()) and bool((w == 1.0).all())
    gen, pts = make_scene(0, n=1000)
    flat, counts = gen.crop_tiles(torch.from_numpy(pts).cuda(), [])
    assert flat.shape == (0, 4) and counts == []


# =====================================================================================================
# 5. offsets beyond 32 bits
# =====================================================================================================
def _free_bytes():
    free, _ = torch.cuda.mem_get_info()
    return free


def test_crop_offsets_beyond_2_31():
    """a 2^31 + 4096-row cloud (51.5 GB) with items starting just below and above row 2^31: the low word of `first` is
    negative as an int32; only the rows the items read are filled"""
    if _free_bytes() < 56e9:
        pytest.skip(f"needs ~56 GB of free device memory, {_free_bytes() / 1e9:.1f} GB free")
    base = 2 ** 31 - 2048
    tiles = [(386000.0, 5820000.0), (386500.0, 5820000.0)]
    cloud = Cloud(7)
    g = np.random.default_rng(8)
    f0 = cloud.run(*tiles[0], 128.0, g.random(3072) < 0.7)
    f1 = cloud.run(*tiles[1], 128.0, g.random(3072) < 0.4)
    host = cloud.array()
    items = [(0, 1024, base + f0 + 1548), (0, 1, 2 ** 31 - 1), (1, 1024, base + f1 + 5), (0, 1024, base + f0),
             (1, 72, base + f1 + 3000), (0, 1000, 2 ** 31 - 1), (0, 500, 2 ** 31)]
    assert base + f0 + 1548 < 2 ** 31 < base + f0 + 1548 + 1024 and base + f1 > 2 ** 31
    assert base + len(host) == 2 ** 31 + 4096
    assert (pack_items(items)[:, 2] < 0).sum() == 3
    try:
        pts_d = torch.empty(2 ** 31 + 4096, 3, dtype=torch.float64, device="cuda")
        pts_d[base:base + len(host)] = torch.from_numpy(host).cuda()
        counts, _, _ = check_crop(host, items, tiles, 128.0, pts_d=pts_d, base=base)
        assert counts.sum() > 1000
    finally:
        pts_d = None
        torch.cuda.empty_cache()


def test_blend_raster_beyond_2_31_pixels():
    """two 46 341 x 46 341 fp64 rasters (more than 2^31 pixels each, 34 GB), tiles at the far corner"""
    if _free_bytes() < 48e9:
        pytest.skip(f"needs ~48 GB of free device memory, {_free_bytes() / 1e9:.1f} GB free")
    N, S, M = 46341, 129, 400
    assert N * N > 2 ** 31
    origins = [(N - S, N - S), (N - 100, N - 60), (N - 300, N - S + 9), (N - S, N - S)]
    t_row, l_col = [o[0] for o in origins], [o[1] for o in origins]
    box = union_box(t_row, l_col, S)
    # the M x M corner of the raster, in local coordinates
    lt, ll = [t - (N - M) for t in t_row], [c - (N - M) for c in l_col]
    lbox = (box[0] - (N - M), box[1] - (N - M), box[2], box[3])
    dsm0, w0, heights, wx, wy = blend_case(S, (M, M), list(zip(lt, ll)), lbox, seed=9)
    ref, ref_w = blend_reference(dsm0, w0, heights, lt, ll, wx, wy, *lbox)
    try:
        dsm = torch.empty(N, N, dtype=torch.float64, device="cuda")
        weight = torch.empty(N, N, dtype=torch.float64, device="cuda")
        dsm[N - M:, N - M:] = torch.from_numpy(dsm0).cuda()
        weight[N - M:, N - M:] = torch.from_numpy(w0).cuda()
        h = torch.from_numpy(heights).cuda()
        tr = torch.tensor(t_row, dtype=torch.int32, device="cuda")
        lc = torch.tensor(l_col, dtype=torch.int32, device="cuda")
        wxd, wyd = torch.from_numpy(wx).cuda(), torch.from_numpy(wy).cuda()
        _lib.call("t2h_blend_accumulate", _lib.ptr(h), len(origins), S, _lib.ptr(tr), _lib.ptr(lc), _lib.ptr(wxd),
                  _lib.ptr(wyd), *box, N, N, _lib.ptr(dsm), _lib.ptr(weight))
        got = dsm[N - M:, N - M:].cpu().numpy()
        got_w = weight[N - M:, N - M:].cpu().numpy()
    finally:
        dsm = weight = None
        torch.cuda.empty_cache()
    assert np.array_equal(got.view(np.uint64), ref.view(np.uint64))
    assert np.array_equal(got_w.view(np.uint64), ref_w.view(np.uint64))
