"""Every dispatch path of the point / plane kernels against exact and fp64 references.

The segment reductions (t2h_segment.cu), the bilinear point sampling with its atomic-free backward and the plane
up-sampling (t2h_sample.cu) pick among several kernels and template instances from C, the Morton flag, the level
shift and the point density.  Each case below reaches one such choice through its natural trigger, asserts by the
profiler's kernel names that it did, and compares the result with a reference that detects a single missing term:

- Segment ops get integer features in [-8, 8]: every fp32 sum the kernels form is then exact in any order, so
  sums, maxima, argmaxima and gradients must equal the fp64 reference bit for bit, means must equal
  fp32(S) * fp32(1 / n) (the kernels' one division), and the fused broadcast-add may differ by its FMA contraction.
- Sampling and up-sampling are checked per element: the tap weights are recomputed in fp32 with the kernels'
  step-by-step arithmetic, products and sums in fp64, and |got - ref| <= (n + 2) 2^-24 sum|w_i g_i| for the n terms
  of that element.  That holds for any summation order and fails on a missing or doubled term in any element with
  fewer than about 4 000 comparable terms.
- Dyadic coordinates j / 2^m with integer planes and gradients make sampling exact too, as long as every element's
  sum|terms| * 2^(2m) < 2^24; the builders assert that budget, and then the kernels must match bit for bit, including
  a cell that 20 000 points share.

Outputs of direct C-ABI calls are pre-filled with NaN (int32 outputs with 0x7fc0dead) and workspaces with NaN bytes,
so that an element a kernel never writes, or a scratch slot it reads without writing, fails the comparison.
"""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as Fnn

import oracle
from cases import synthetic_cloud
from tomosar2height_b200.functional import SUPPORTED_C

U = 2.0 ** -24
LO, HI = 2.0 ** -24, 1.0 - 2.0 ** -24
SENTINEL_I32 = 0x7FC0DEAD
# row counts that sit on the chunk borders: kChunk (32), kRowChunk and Rows9 (128, 256), kLongList * kChunk (512)
COUNTS = (31, 32, 33, 127, 128, 129, 255, 256, 257, 511, 512, 513)

_SEEN = set()   # every kernel name the profiler reported in this session


# =====================================================================================================
# references (CPU)
# =====================================================================================================
def cells_of(xy, tile, r):
    """plane row b*r*r + iy*r + ix of every point: trunc(p * r) in fp32 (coordinate2index)"""
    c = (xy.float() * r).long()
    return tile * (r * r) + c[:, 1] * r + c[:, 0]


def taps_f32(xy, r):
    """The kernels' make_taps: four tap cells (x0/x0+1, y0/y0+1) and their fp32 weights, one rounded op at a time.
    Returns (ix (n, 4), iy (n, 4), w (n, 4) fp32); a tap beyond the last row / column carries weight 0."""
    def axis(p):
        g = p * 2.0 - 1.0
        i = ((g + 1.0) * 0.5) * float(r - 1)
        i = i.clamp(0.0, float(r - 1))
        f = i.floor()
        return f.long(), (f + 1.0) - i, i - f
    x0, wx0, wx1 = axis(xy[:, 0].float())
    y0, wy0, wy1 = axis(xy[:, 1].float())
    wx1 = torch.where(x0 + 1 < r, wx1, torch.zeros_like(wx1))
    wy1 = torch.where(y0 + 1 < r, wy1, torch.zeros_like(wy1))
    ix = torch.stack([x0, x0 + 1, x0, x0 + 1], 1).clamp(max=r - 1)
    iy = torch.stack([y0, y0, y0 + 1, y0 + 1], 1).clamp(max=r - 1)
    w = torch.stack([wx0 * wy0, wx1 * wy0, wx0 * wy1, wx1 * wy1], 1)  # fp32 products, each rounded once
    return ix, iy, w


def sample_taps(xy, tile, r):
    """(plane row of every tap (n, 4), fp32 weight (n, 4))"""
    ix, iy, w = taps_f32(xy, r)
    return tile[:, None] * (r * r) + iy * r + ix, w


def sample_fwd_ref(plane, idx, w):
    """plane (n_cells, C) -> (ref fp64 (n, C), A = sum|w v|, n_terms = 4)"""
    ref = torch.zeros(idx.shape[0], plane.shape[1], dtype=torch.float64)
    A = torch.zeros_like(ref)
    p64 = plane.double()
    for t in range(4):
        term = w[:, t, None].double() * p64[idx[:, t]]
        ref += term
        A += term.abs()
    return ref, A, 4


def sample_bwd_ref(g, idx, w, n_cells):
    """g (n, C) -> (ref fp64 (n_cells, C), A, number of non-zero terms per cell (n_cells, 1))"""
    C = g.shape[1]
    ref = torch.zeros(n_cells, C, dtype=torch.float64)
    A = torch.zeros_like(ref)
    g64 = g.double()
    for t in range(4):
        term = w[:, t, None].double() * g64
        ref.index_add_(0, idx[:, t], term)
        A.index_add_(0, idx[:, t], term.abs())
    nz = w != 0
    n = torch.bincount(idx[nz], minlength=n_cells)[:, None].double()
    return ref, A, n


def upsample_axis_f32(n_in, n_out):
    """The kernels' make_axis for every output index: (i0, i1, l0, l1), scale = fp32(n_in - 1) / fp32(n_out - 1)"""
    scale = np.float32(n_in - 1) / np.float32(n_out - 1) if n_out > 1 else np.float32(0.0)
    src = (scale * np.arange(n_out, dtype=np.float32)).astype(np.float32)
    i0 = np.minimum(src.astype(np.int64), n_in - 1)
    i1 = i0 + (i0 < n_in - 1)
    l1 = (src - i0.astype(np.float32)).astype(np.float32)
    l0 = (np.float32(1.0) - l1).astype(np.float32)
    return i0, i1, l0, l1


def upsample_fwd_ref(x, oh, ow):
    """x (B, h, w, C) -> (ref fp64 (B, oh, ow, C), A, 4)"""
    B, h, w, C = x.shape
    ay, ax = upsample_axis_f32(h, oh), upsample_axis_f32(w, ow)
    x64 = x.double()
    ref = torch.zeros(B, oh, ow, C, dtype=torch.float64)
    A = torch.zeros_like(ref)
    for iy, ly in ((ay[0], ay[2]), (ay[1], ay[3])):
        for ix, lx in ((ax[0], ax[2]), (ax[1], ax[3])):
            wgt = torch.from_numpy(ly.astype(np.float64))[:, None] * torch.from_numpy(lx.astype(np.float64))[None, :]
            term = wgt[None, :, :, None] * x64[:, torch.from_numpy(iy)][:, :, torch.from_numpy(ix)]
            ref += term
            A += term.abs()
    return ref, A, 4


def _axis_pairs(n_in, n_out):
    """(output index, input index, fp32 weight) with the backward's per-axis weight
    fp32((i0 == y ? l0 : 0) + (i1 == y ? l1 : 0)), non-zero entries only"""
    i0, i1, l0, l1 = upsample_axis_f32(n_in, n_out)
    out, inp, wt = [], [], []
    for o in range(n_out):
        for y in sorted({int(i0[o]), int(i1[o])}):
            v = np.float32((l0[o] if i0[o] == y else np.float32(0)) + (l1[o] if i1[o] == y else np.float32(0)))
            if v != 0:
                out.append(o); inp.append(y); wt.append(v)
    return np.array(out), np.array(inp), np.array(wt, dtype=np.float32)


def upsample_bwd_ref(g, h, w):
    """g (B, oh, ow, C) -> (ref fp64 (B, h, w, C), A, terms per input pixel (h, w, 1))"""
    B, oh, ow, C = g.shape
    oy, y, wy = _axis_pairs(h, oh)
    ox, x, wx = _axis_pairs(w, ow)
    wgt = torch.from_numpy((wy[:, None] * wx[None, :]).astype(np.float32)).double()  # fp32(wy * wx), as the kernel
    src = (torch.from_numpy(oy)[:, None] * ow + torch.from_numpy(ox)[None, :]).reshape(-1)
    dst = (torch.from_numpy(y)[:, None] * w + torch.from_numpy(x)[None, :]).reshape(-1)
    term = wgt.reshape(1, -1, 1) * g.double().reshape(B, oh * ow, C)[:, src]
    ref = torch.zeros(B, h * w, C, dtype=torch.float64).index_add_(1, dst, term)
    A = torch.zeros(B, h * w, C, dtype=torch.float64).index_add_(1, dst, term.abs())
    n = torch.bincount(dst, minlength=h * w).double()
    return ref.view(B, h, w, C), A.view(B, h, w, C), n.view(h, w, 1)


def seg_refs(feat, cell, n_seg):
    """Exact per-cell sum (fp64), count, max and argmax (smallest point index among ties; -1 when empty)."""
    n, C = feat.shape
    S = torch.zeros(n_seg, C, dtype=torch.float64).index_add_(0, cell, feat.double())
    cnt = torch.bincount(cell, minlength=n_seg)
    ce = cell[:, None].expand(n, C)
    vmax = torch.full((n_seg, C), -math.inf).scatter_reduce(0, ce, feat, "amax", include_self=True)
    cand = torch.where(feat == vmax[cell], torch.arange(n)[:, None], torch.full((1, 1), n))
    arg = torch.full((n_seg, C), n).scatter_reduce(0, ce, cand, "amin", include_self=True)
    empty = (cnt == 0)[:, None]
    return S, cnt, torch.where(empty, torch.zeros(()), vmax), torch.where(empty, torch.full((), -1), arg)


def mean_ref(S, cnt):
    """fp32(S) * fp32(1 / n): the kernels take one IEEE division per cell; empty cells are 0"""
    inv = 1.0 / cnt.float().clamp(min=1)
    return torch.where((cnt > 0)[:, None], S.float() * inv[:, None], torch.zeros(()))


def assert_bound(got, ref, A, n, what):
    """|got - ref| <= (n + 2) 2^-24 A per element (plus the fp64 reference's own rounding); NaN / inf fail"""
    got = got.detach().double().cpu().reshape(ref.shape)
    assert bool(torch.isfinite(got).all()), f"{what}: {int((~torch.isfinite(got)).sum())} elements unwritten or non-finite"
    tol = (n + 2) * U * A + (n + 2) * 2.0 ** -50 * A
    err = (got - ref).abs()
    bad = err > tol
    if bool(bad.any()):
        i = int(torch.argmax((err - tol).reshape(-1)))
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} elements outside the bound; worst at flat {i}: "
                             f"got {got.reshape(-1)[i].item()!r} ref {ref.reshape(-1)[i].item()!r} "
                             f"tol {tol.expand_as(ref).reshape(-1)[i].item():.3e}")


def assert_bitwise(got, want, what):
    got = got.detach().cpu()
    want = want.to(got.dtype).reshape(got.shape)
    if not torch.equal(got, want):
        same = (got == want) | (torch.isnan(got) & torch.isnan(want)) if got.is_floating_point() else got == want
        bad = (~same).nonzero()
        raise AssertionError(f"{what}: {bad.shape[0]} of {got.numel()} elements differ; first at {bad[0].tolist()}: "
                             f"got {got[tuple(bad[0])].item()!r} want {want[tuple(bad[0])].item()!r}")


# =====================================================================================================
# inputs
# =====================================================================================================
def _dyadic_m(xy):
    """smallest m with p * 2^m integral for both coordinates of every point (24 when none <= 24)"""
    p = xy.double()
    m = torch.full((xy.shape[0],), 24, dtype=torch.long)
    for k in range(24, -1, -1):
        ok = ((p * 2.0 ** k) == (p * 2.0 ** k).floor()).all(1)
        m = torch.where(ok, torch.full_like(m, k), m)
    return m


def _edge_points(R):
    """cell edges k / r of the finest and coarser levels, the extreme coordinates 2^-24 and 1 - 2^-24, duplicates"""
    pts = [(LO, LO), (LO, HI), (HI, LO), (HI, HI), (0.5, HI), (HI, 0.5), (LO, 0.5), (0.5, LO)]
    levels = [R] + ([R // 4, R // 16, 2] if R & (R - 1) == 0 else [])
    for r in levels:
        ks = sorted({1, r // 2, r - 1} - {0})
        for a in ks:
            for b in ks:
                pts.append((a / r, b / r))
            pts.append((a / r, 0.37))
            pts.append((0.61, a / r))
    pts += pts[:6]  # exact duplicates
    return torch.tensor(pts, dtype=torch.float32)


def _count_cells(R):
    return [((7 + 5 * i) % R, (11 + 7 * i) % R) for i in range(len(COUNTS))]


def _fill_tile(xy, R, g, heavy=0, counts=True):
    """tile xy (N, 2) in place: edge points, a `heavy`-row cell, cells of exactly COUNTS rows; shuffled"""
    N = xy.shape[0]
    e = _edge_points(R)
    k = e.shape[0]
    xy[:k] = e
    hc = torch.tensor([19.0, 38.0]) if R >= 64 else torch.tensor([1.0, 2.0])
    if heavy:
        xy[k:k + heavy] = (hc + 0.1 + 0.8 * torch.rand(heavy, 2, generator=g)) / R
        k += heavy
    designated = _count_cells(R) if counts else []
    if counts:
        for (cx, cy), c in zip(designated, COUNTS):
            xy[k:k + c] = (torch.tensor([cx, cy], dtype=torch.float32) + 0.05 + 0.9 * torch.rand(c, 2, generator=g)) / R
            k += c
        assert k <= N
        # nothing else may land in a designated cell: move such points into the heavy cell (or onto a corner)
        cell = (xy * R).long()
        for cx, cy in designated:
            hit = (cell[:, 0] == cx) & (cell[:, 1] == cy)
            hit[:k] = False
            xy[hit] = ((hc + 0.5) / R) if heavy else torch.tensor([LO, LO])
    xy.copy_(xy[torch.randperm(N, generator=g)])


class Cloud:
    """Points (n, 2) fp32 in flat order, their tile, and (lazily, on the GPU) the Topology that sorts them."""

    def __init__(self, xy, tile, R, B, N=None, offsets=None):
        self.xy, self.tile, self.R, self.B, self.N, self.offsets = xy, tile, R, B, N, offsets
        self._topo = None

    @property
    def n(self):
        return self.xy.shape[0]

    def topo(self):
        from tomosar2height_b200.topology import Topology
        if self._topo is None:
            if self.offsets is None:
                t = Topology(self.xy.view(self.B, self.N, 2).cuda(), self.R)
            else:
                t = Topology(self.xy.cuda(), self.R, offsets=self.offsets.cuda())
            self.perm = t.perm.long().cpu()
            self.inv = torch.empty_like(self.perm)
            self.inv[self.perm] = torch.arange(self.n)
            self._topo = t
        return self._topo

    def level(self, r):
        """(n_seg, shift, morton) of plane level r"""
        t = self.topo()
        shift = 0 if r == self.R else 2 * ((self.R // r).bit_length() - 1)
        assert r == self.R or (t.morton and self.R % r == 0 and r << (shift // 2) == self.R)
        return self.B * r * r, shift, int(t.morton)


def _dense(B, N, R, seed, heavy=0, counts=True):
    g = torch.Generator().manual_seed(seed)
    xy = synthetic_cloud(B, N, seed)[..., :2].contiguous()
    _fill_tile(xy[0], R, g, heavy=heavy, counts=counts)
    return Cloud(xy.reshape(-1, 2).contiguous(), torch.arange(B).repeat_interleave(N), R, B, N=N)


def _ragged(tiles, R):
    sizes = torch.tensor([0] + [t.shape[0] for t in tiles])
    offsets = sizes.cumsum(0)
    tile = torch.repeat_interleave(torch.arange(len(tiles)), sizes[1:])
    return Cloud(torch.cat(tiles).contiguous(), tile, R, len(tiles), offsets=offsets)


def _ragged_tiles(R, seed, dyadic):
    """an empty tile first, in the middle and last; a one-point tile; a tile whose points share one cell"""
    g = torch.Generator().manual_seed(seed)
    if dyadic:
        pt = lambda n: torch.randint(1, 1024, (n, 2), generator=g).float() / 1024
        one_cell = (torch.tensor([9.0, 4.0]) + torch.randint(0, 16, (500, 2), generator=g).float() / 16) / R
        big = pt(3000)
    else:
        one_cell = (torch.tensor([9.0, 4.0]) + 0.05 + 0.9 * torch.rand(500, 2, generator=g)) / R
        big = synthetic_cloud(1, 3200, seed)[0, :, :2].contiguous()
        _fill_tile(big, R, g)
        pt = lambda n: synthetic_cloud(1, n, seed + n)[0, :, :2].contiguous()
    empty = torch.zeros(0, 2)
    return [empty, pt(1), one_cell, big, empty, pt(700), empty]


def _dyadic_dense(B, N, seed, m=10):
    g = torch.Generator().manual_seed(seed)
    xy = torch.randint(1, 2 ** m, (B * N, 2), generator=g).float() / 2 ** m
    e = torch.tensor([[k / 64, l / 64] for k in (1, 16, 32, 63) for l in (1, 32, 63)] + [[0.5, 0.5]] * 3)
    xy[:e.shape[0]] = e  # cell edges of every level, duplicates
    return Cloud(xy, torch.arange(B).repeat_interleave(N), 64, B, N=N)


HEAVY_AT = (5 / 8, 3 / 8)  # m = 3; on a cell edge of every level


def _dyadic_heavy(N=26000, heavy=20000, seed=5):
    """20 000 points at one dyadic coordinate; the others (m = 6, so that a few of them may share a cell within the
    budget) stay out of its tap neighbourhood at r >= 16"""
    g = torch.Generator().manual_seed(seed)
    xy = torch.randint(1, 64, (N, 2), generator=g).float() / 64
    xy[:heavy] = torch.tensor(HEAVY_AT)
    near = ((xy - torch.tensor(HEAVY_AT)).abs() < 0.15).all(1)
    near[:heavy] = False
    xy[near, 0] = xy[near, 0] - 5 / 16  # stays dyadic, moves >= 0.16 away
    xy.copy_(xy[torch.randperm(N, generator=g)])
    return Cloud(xy, torch.zeros(N, dtype=torch.long), 64, 1, N=N)


_CLOUDS = {}
_BUILDERS = {
    "A": lambda: _dense(2, 6000, 64, seed=11),                        # fine levels, chunk-border cells
    "H": lambda: _dense(1, 32768, 64, seed=12, heavy=20000),          # a 20 000-row cell
    "M": lambda: _dense(2, 4000, 100, seed=13),                       # row-major keys (R not a power of two)
    "M10": lambda: Cloud(cloud("M").xy, cloud("M").tile, 10, 2, N=4000),  # row-major, many rows per cell
    "G": lambda: _ragged(_ragged_tiles(64, 21, dyadic=False), 64),
    "D": lambda: _dyadic_dense(2, 5000, seed=31),
    "DG": lambda: _ragged(_ragged_tiles(64, 22, dyadic=True), 64),
    "E": lambda: _dyadic_heavy(),
}


def cloud(name):
    if name not in _CLOUDS:
        _CLOUDS[name] = _BUILDERS[name]()
    return _CLOUDS[name]


def int_tensor(shape, seed):
    """integers in [-8, 8] as fp32"""
    return torch.randint(-8, 9, shape, generator=torch.Generator().manual_seed(seed)).float()


def assert_exact_budget(A, m_elem, what):
    """sum|terms| * 2^(2m) < 2^24 for every element: then every partial sum is a representable fp32 value"""
    over = A * torch.exp2(2.0 * m_elem.double()) >= 2.0 ** 24
    assert not bool(over.any()), f"{what}: {int(over.sum())} elements exceed the exactness budget"


def sample_m_bwd(c, idx, w, n_cells):
    m = _dyadic_m(c.xy)
    out = torch.zeros(n_cells, dtype=torch.long)
    for t in range(4):
        nz = w[:, t] != 0
        out.scatter_reduce_(0, idx[nz, t], m[nz], "amax")
    return out[:, None]


# =====================================================================================================
# GPU plumbing: direct C-ABI calls with sentinel outputs, and the kernels they launched
# =====================================================================================================
def _lib():
    from tomosar2height_b200 import _lib as L
    return L.load()


def _call(name, *args):
    from tomosar2height_b200 import _lib
    _lib.call(name, *args)


def _p(t):
    from tomosar2height_b200._lib import ptr
    return ptr(t)


def nan_f32(*shape):
    return torch.full(shape, float("nan"), dtype=torch.float32, device="cuda")


def sentinel_i32(*shape):
    return torch.full(shape, SENTINEL_I32, dtype=torch.int32, device="cuda")


def nan_workspace(nbytes):
    return torch.full((max(int(nbytes), 1),), 0xFF, dtype=torch.uint8, device="cuda")


def launched(fn):
    """run fn under the profiler; the set of kernel names it launched (spaces removed)"""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = {e.name.replace(" ", "") for e in prof.events()}
    _SEEN.update(names)
    return names


def expect(names, *kernels, only=None):
    """every kernel in `kernels` ran; with only=prefix, no other kernel whose name contains the prefix ran"""
    for k in kernels:
        k = k.replace(" ", "")
        assert any(k in n for n in names), f"kernel {k} did not run; launched: {sorted(names)}"
    if only is not None:
        extra = {n for n in names if only in n and not any(k.replace(' ', '') in n for k in kernels)}
        assert not extra, f"unexpected {only} kernels {sorted(extra)} (expected {kernels})"


def RS(C):
    lpr = min(C // 4, 32)
    return f"t2h::RowShape<{lpr},{C // (4 * lpr)}>"


# =====================================================================================================
# 5. CPU self-tests of the references
# =====================================================================================================
def test_sample_reference_matches_oracle_and_grid_sample():
    g = torch.Generator().manual_seed(1)
    for r in (1, 2, 7, 64, 100):
        B, N, C = 2, 700, 3
        xy = torch.rand(B * N, 2, generator=g)
        xy[:8] = _edge_points(64)[:8]
        tile = torch.arange(B).repeat_interleave(N)
        plane = torch.randn(B, C, r, r, generator=g, dtype=torch.float64)
        idx, w = sample_taps(xy, tile, r)
        ref, A, _ = sample_fwd_ref(plane.permute(0, 2, 3, 1).reshape(-1, C), idx, w)
        want = oracle.bilinear_sample_points(plane, xy.double().view(B, N, 2)).permute(0, 2, 1).reshape(-1, C)
        aten = Fnn.grid_sample(plane, (2 * xy.double().view(B, N, 1, 2) - 1), padding_mode="border",
                               align_corners=True).squeeze(-1).permute(0, 2, 1).reshape(-1, C)
        tol = 16 * U * max(r, 1) * plane.abs().max()  # fp32 weights against fp64 ones
        assert float((ref - want).abs().max()) <= tol and float((ref - aten).abs().max()) <= tol, r
        # the backward reference is the adjoint of the forward one
        gr = torch.randn(B * N, C, generator=g, dtype=torch.float64)
        gp, _, _ = sample_bwd_ref(gr, idx, w, B * r * r)
        lhs, rhs = (ref * gr).sum(), (gp * plane.permute(0, 2, 3, 1).reshape(-1, C)).sum()
        assert abs(float(lhs - rhs)) <= 1e-9 * float((ref.abs() * gr.abs()).sum()), r


def test_upsample_reference_matches_interpolate():
    g = torch.Generator().manual_seed(2)
    for h, w, oh, ow in [(1, 1, 1, 1), (1, 5, 3, 1), (4, 4, 9, 9), (7, 5, 12, 3), (33, 17, 20, 9), (40, 40, 80, 79),
                         (2, 40, 1, 80), (13, 1, 26, 5)]:
        x = torch.randn(2, h, w, 3, generator=g, dtype=torch.float64)
        ref, A, _ = upsample_fwd_ref(x, oh, ow)
        want = Fnn.interpolate(x.permute(0, 3, 1, 2), size=(oh, ow), mode="bilinear", align_corners=True).permute(0, 2, 3, 1)
        tol = 16 * U * max(h, w) * x.abs().max()
        assert float((ref - want).abs().max()) <= tol, (h, w, oh, ow)
        gy = torch.randn(2, oh, ow, 3, generator=g, dtype=torch.float64)
        gx, _, _ = upsample_bwd_ref(gy, h, w)
        xa = x.clone().requires_grad_(True)
        Fnn.interpolate(xa.permute(0, 3, 1, 2), size=(oh, ow), mode="bilinear", align_corners=True).permute(0, 2, 3, 1).backward(gy)
        assert float((gx - xa.grad).abs().max()) <= 16 * U * max(h, w) * gy.abs().max() * 4, (h, w, oh, ow)


def _two_orders_exact(terms, dst, n_out, ref, what):
    """fp32 index_add in forward and in reversed order must both equal the fp64 sum bit for bit"""
    fwd = torch.zeros(n_out, terms.shape[1]).index_add_(0, dst, terms.float())
    rev = torch.zeros(n_out, terms.shape[1]).index_add_(0, dst.flip(0), terms.float().flip(0))
    assert torch.equal(fwd.double(), ref) and torch.equal(rev.double(), ref), what


@pytest.mark.parametrize("name", ["D", "DG"])
def test_dyadic_sample_forward_inputs_are_exact(name):
    c = cloud(name)
    for r in (64, 8):
        idx, w = sample_taps(c.xy, c.tile, r)
        plane = int_tensor((c.B * r * r, 8), 3)
        ref, A, _ = sample_fwd_ref(plane, idx, w)
        assert_exact_budget(A, _dyadic_m(c.xy)[:, None], f"{name} r={r}")
        terms = (w[:, :, None].double() * plane[idx].double()).reshape(-1, 8)
        assert torch.equal(terms.float().double(), terms), "every product w * v is an fp32 value"
        _two_orders_exact(terms, torch.arange(c.n).repeat_interleave(4), c.n, ref, f"{name} r={r}")


def test_dyadic_heavy_backward_inputs_are_exact():
    c = cloud("E")
    for r in HEAVY_LEVELS:
        idx, w = sample_taps(c.xy, c.tile, r)
        gr = int_tensor((c.n, 4), 4)
        ref, A, _ = sample_bwd_ref(gr, idx, w, r * r)
        m = sample_m_bwd(c, idx, w, r * r)
        assert_exact_budget(A, m, f"heavy r={r}")
        hc = cells_of(torch.tensor([HEAVY_AT]), torch.zeros(1, dtype=torch.long), r)
        assert int(m[hc]) == 3 and float(A[hc].max()) > 2.0 ** 13, "the heavy cell's terms are all m = 3 and large"
        terms = (w.reshape(-1, 1).double() * gr.double().repeat_interleave(4, 0))
        _two_orders_exact(terms, idx.reshape(-1), r * r, ref, f"heavy r={r}")


@pytest.mark.parametrize("name", ["A", "H", "G"])
def test_integer_segment_inputs_are_exact(name):
    c = cloud(name)
    f = int_tensor((c.n, 4), 5)
    for r in (c.R, 1):
        cell = cells_of(c.xy, c.tile, r)
        S, cnt, _, _ = seg_refs(f, cell, c.B * r * r)
        _two_orders_exact(f, cell, c.B * r * r, S, f"{name} r={r}")
    if name == "H":
        assert int(torch.bincount(cells_of(c.xy, c.tile, c.R)).max()) >= 20000
    if name in ("A", "H"):  # the chunk-border cells hold exactly their row counts
        cnt = torch.bincount(cells_of(c.xy, c.tile, c.R), minlength=c.B * c.R * c.R)
        for (cx, cy), k in zip(_count_cells(c.R), COUNTS):
            assert int(cnt[cy * c.R + cx]) == k


def test_path_matrix_covers_every_kernel_instance():
    """The union of the kernels the GPU cases below assert covers every instance the dispatch can pick."""
    want = set(REQUIRED)
    have = set()
    for case in SAMPLE_BWD_CASES:
        have.update(k.replace(" ", "") for k in case[-1])
    for C in SUPPORTED_C:
        have.update(k.replace(" ", "") for k in _seg_kernels(C))
        have.update(f"upsample_{d}_kernel<{RS(C)}>" for d in ("fwd", "bwd"))
        have.add(f"sample_fwd_kernel<{RS(C)}>")
    assert want <= have, sorted(want - have)


# =====================================================================================================
# 2 / 3. segment ops: every C, shift 0 and > 0 down to r = 1, rows sorted and unsorted
# =====================================================================================================
def _seg_kernels(C):
    rs = RS(C)
    return [f"seg_reduce_rows_kernel<{rs}>", f"seg_reduce_fix_kernel<{rs}>", f"seg_max_rows_kernel<{rs}>",
            f"seg_max_fix_kernel<{rs}>", f"seg_rowmap_kernel<{rs},0>", f"seg_rowmap_kernel<{rs},1>",
            f"seg_rowmap_kernel<{rs},2>"]


SEG_CASES = ([("A", C, s, (64, 8, 1)) for C in SUPPORTED_C for s in (True, False)]
             + [("H", C, True, (64, 16, 1)) for C in (4, 32, 128, 512)] + [("H", 64, False, (64, 1))]
             + [("M", C, s, (100,)) for C in (8, 256) for s in (True, False)]
             + [("G", C, s, (64, 4, 1)) for C in (16, 128) for s in (True, False)])


@pytest.mark.gpu
@pytest.mark.parametrize("name,C,rows_sorted,levels", SEG_CASES, ids=[f"{a}-C{b}-{'sorted' if c else 'perm'}" for a, b, c, _ in SEG_CASES])
def test_segment_ops_exact(name, C, rows_sorted, levels):
    c = cloud(name)
    topo = c.topo()
    n = c.n
    perm_dev = None if rows_sorted else topo.perm
    to_rows = (lambda x: x[c.perm]) if rows_sorted else (lambda x: x)       # point order -> row order
    to_pts = (lambda x: x[c.inv]) if rows_sorted else (lambda x: x)        # row order -> point order
    row_of_pt = c.inv if rows_sorted else torch.arange(n)
    pt_of_row = c.perm if rows_sorted else torch.arange(n)
    feat = int_tensor((n, C), C)
    gp = int_tensor((n, C), C + 1)
    rows_dev = to_rows(feat).cuda()
    gp_dev = to_rows(gp).cuda()
    rs = RS(C)
    results = {}

    def geo(r):
        n_seg, shift, morton = c.level(r)
        return n_seg, shift, morton, topo.keys_sorted, topo.cell_start, (topo.perm if shift > 0 else None)

    def run_reduce(mean):
        for r in levels:
            n_seg, shift, morton, keys, cs, _ = geo(r)
            nb = int(_lib().t2h_seg_workspace_bytes(n, n_seg, C))
            ws = nan_workspace(nb)
            plane = nan_f32(n_seg, C)
            _call("t2h_seg_reduce_fwd", _p(rows_dev), n, _p(perm_dev), _p(keys), _p(cs), n_seg, shift, C, morton, r,
                  int(mean), _p(ws), nb, _p(plane))
            results[("reduce", mean, r)] = plane

    def run_max():
        for r in levels:
            n_seg, shift, morton, keys, cs, tie = geo(r)
            nb = int(_lib().t2h_seg_workspace_bytes(n, n_seg, C))
            ws = nan_workspace(nb)
            pooled, plane, arg = nan_f32(n, C), nan_f32(n_seg, C), sentinel_i32(n_seg, C)
            _call("t2h_seg_max_fwd", _p(rows_dev), n, _p(perm_dev), _p(tie), _p(keys), _p(cs), n_seg, shift, C, morton, r,
                  _p(ws), nb, _p(pooled), _p(plane), _p(arg))
            results[("max", r)] = (pooled, plane, arg)

    refs = {}
    for r in levels:
        cell = cells_of(c.xy, c.tile, r)
        refs[r] = (cell,) + seg_refs(feat, cell, c.B * r * r)

    expect(launched(lambda: run_reduce(False)), f"seg_reduce_rows_kernel<{rs}>", f"seg_reduce_fix_kernel<{rs}>")
    expect(launched(lambda: run_reduce(True)), f"seg_reduce_rows_kernel<{rs}>", f"seg_reduce_fix_kernel<{rs}>")
    expect(launched(run_max), f"seg_max_rows_kernel<{rs}>", f"seg_max_fix_kernel<{rs}>", f"seg_rowmap_kernel<{rs},0>")
    for r in levels:
        cell, S, cnt, vmax, arg_pt = refs[r]
        assert_bitwise(results[("reduce", False, r)], S.float(), f"seg_sum r={r}")
        assert_bitwise(results[("reduce", True, r)], mean_ref(S, cnt), f"seg_mean r={r}")
        pooled, plane, arg = results[("max", r)]
        assert_bitwise(plane, vmax, f"seg_max values r={r}")
        a = arg.cpu().long()
        assert bool(((a >= -1) & (a < n)).all()), f"seg_max arg r={r}: unwritten or out-of-range entries"
        got_pt = torch.where(a < 0, a, pt_of_row[a.clamp(min=0)])
        assert_bitwise(got_pt, arg_pt, f"seg_max argmax r={r} (ties -> smallest point index, empty -> -1)")
        assert_bitwise(to_pts(pooled.cpu()), vmax[cell], f"seg_max pooled r={r}")

    # backward of the max: grad_pooled only, grad_plane only, both
    for r in levels:
        cell, S, cnt, vmax, arg_pt = refs[r]
        n_seg, shift, morton, keys, cs, _ = geo(r)
        arg_rows = torch.where(arg_pt < 0, arg_pt, row_of_pt[arg_pt.clamp(min=0)]).int().cuda()
        gl = int_tensor((n_seg, C), C + 2 + r)
        gl_dev = gl.cuda()
        Sg = torch.zeros(n_seg, C, dtype=torch.float64).index_add_(0, cell, gp.double())
        won = arg_pt[cell] == torch.arange(n)[:, None]
        for use_gp, use_gl in ((True, False), (False, True), (True, True)):
            tot = (Sg if use_gp else 0) + (gl.double() if use_gl else 0)
            want = torch.where(won, tot[cell], torch.zeros(()))
            nb = int(_lib().t2h_seg_workspace_bytes(n, n_seg, C)) if use_gp else 0
            ws = nan_workspace(nb) if use_gp else None
            out = nan_f32(n, C)
            names = launched(lambda: _call("t2h_seg_max_bwd", _p(gp_dev if use_gp else None), _p(gl_dev if use_gl else None),
                                           n, _p(perm_dev), _p(keys), _p(cs), n_seg, shift, C, morton, r, _p(arg_rows),
                                           _p(ws), nb, _p(out)))
            expect(names, f"seg_rowmap_kernel<{rs},1>", *([f"seg_reduce_rows_kernel<{rs}>"] if use_gp else []))
            assert_bitwise(to_pts(out.cpu()), want.float(), f"seg_max_bwd r={r} grad_pooled={use_gp} grad_plane={use_gl}")

    # broadcast (mean 0 / 1) and broadcast-add with its max-|x| slot
    for r in levels:
        cell, S, cnt, _, _ = refs[r]
        n_seg, shift, morton, keys, cs, _ = geo(r)
        plane = int_tensor((n_seg, C), C + 3 + r)
        plane_dev = plane.cuda()
        for mean in (0, 1):
            inv = (1.0 / cnt.float().clamp(min=1))[cell][:, None] if mean else torch.ones(n, 1)
            out = nan_f32(n, C)
            expect(launched(lambda: _call("t2h_seg_broadcast", _p(plane_dev), n, _p(perm_dev), _p(keys), _p(cs), n_seg, shift,
                                          C, morton, r, mean, _p(out))), f"seg_rowmap_kernel<{rs},0>")
            assert_bitwise(to_pts(out.cpu()), plane[cell] * inv, f"seg_broadcast r={r} mean={mean}")
            out = nan_f32(n, C)
            slot = sentinel_i32(1)
            expect(launched(lambda: _call("t2h_seg_broadcast_add", _p(plane_dev), _p(gp_dev), n, _p(perm_dev), _p(keys), _p(cs),
                                          n_seg, shift, C, morton, r, mean, _p(out), _p(slot))), f"seg_rowmap_kernel<{rs},2>")
            got = to_pts(out.cpu())
            prod = plane[cell] * inv                                     # fp32(v * inv)
            unfused = prod + gp                                          # two roundings
            fused = (plane[cell].double() * inv.double() + gp.double()).float()  # v * inv exact in fp64, one rounding
            if mean == 0:
                assert_bitwise(got, unfused, f"seg_broadcast_add r={r} mean=0")
            else:
                ulp = (torch.nextafter(fused.abs(), torch.tensor(math.inf)) - fused.abs())
                ok = (got == unfused) | ((got.double() - fused.double()).abs() <= ulp.double())
                assert bool(ok.all()), f"seg_broadcast_add r={r} mean=1: {int((~ok).sum())} elements beyond 1 ulp"
            slot_val = torch.tensor([int(slot.cpu())], dtype=torch.int32).view(torch.float32)
            assert_bitwise(slot_val, got.abs().max().view(1), f"seg_broadcast_add slot r={r}")


# =====================================================================================================
# 2 / 3. bilinear_sample_fwd: every C, dense and ragged, perm NULL and not
# =====================================================================================================
def _sample_fwd_case(c, C, r, rows_sorted, seed, exact):
    topo = c.topo()
    n = c.n
    plane = int_tensor((c.B * r * r, C), seed) if exact else torch.randn(c.B * r * r, C,
                                                                          generator=torch.Generator().manual_seed(seed))
    plane_dev = plane.cuda()
    out = nan_f32(n, C)
    perm = None if rows_sorted else topo.perm
    tile_ids = topo.tile_ids  # ragged batches carry tile ids; None for dense ones
    names = launched(lambda: _call("t2h_bilinear_sample_fwd", _p(plane_dev), r, C, _p(topo.xyz_sorted), 4, _p(perm),
                                   _p(tile_ids), n, c.N or 1, _p(out)))
    expect(names, f"sample_fwd_kernel<{RS(C)}>")
    got = out.cpu()[c.inv] if rows_sorted else out.cpu()
    idx, w = sample_taps(c.xy, c.tile, r)
    ref, A, nt = sample_fwd_ref(plane, idx, w)
    what = f"sample fwd C={C} r={r} {'sorted' if rows_sorted else 'perm'}"
    if exact:
        assert_exact_budget(A, _dyadic_m(c.xy)[:, None], what)  # a row's terms share its point's m
        assert_bitwise(got, ref.float(), what + " (dyadic, exact)")
    else:
        assert_bound(got, ref, A, nt, what)


@pytest.mark.gpu
@pytest.mark.parametrize("C", SUPPORTED_C)
@pytest.mark.parametrize("ragged", [False, True], ids=["dense", "ragged"])
def test_sample_fwd(C, ragged):
    for rows_sorted in (True, False):
        for r in (64, 8):
            _sample_fwd_case(cloud("DG" if ragged else "D"), C, r, rows_sorted, C + r, exact=True)
            _sample_fwd_case(cloud("G" if ragged else "A"), C, r, rows_sorted, C + r + 1, exact=False)


# =====================================================================================================
# 2 / 3. bilinear_sample_bwd: every G2 kernel instance
# =====================================================================================================
def _wtile(C, TW):
    return [f"sample_bwd_wtile_rows_kernel<{C},{TW}>", f"sample_bwd_wtile_merge_kernel<{C},{TW}>"]


def _nine(C):
    lpr = {32: 8, 64: 16}.get(C, 32)
    return [f"sample_bwd_nine_rows_kernel<{lpr}>", f"sample_bwd_nine_fix_kernel<{256 if C >= 128 else 128}>",
            "sample_bwd_nine_gather_kernel"]


def _gather(C, wps):
    return [f"sample_bwd_kernel<{RS(C)},{wps}>"]


# (cloud, C, level r, workspace, kernels that must run); avg rows per cell = points / (B r^2) picks the path
SAMPLE_BWD_CASES = [
    ("A", 32, 64, True, _wtile(32, 4)),        # avg 1
    ("A", 64, 64, True, _wtile(64, 4)),
    ("A", 128, 32, True, _wtile(128, 2)),      # avg 5
    ("G", 32, 64, True, _wtile(32, 4)),        # ragged
    ("H", 32, 32, True, _nine(32)),            # avg 32: the first density past the tile walk
    ("A", 32, 2, True, _nine(32)),             # reso < 4
    ("H", 64, 16, True, _nine(64)),            # avg 128, the 20 000-row cell
    ("A", 64, 2, True, _nine(64)),
    ("H", 128, 16, True, _nine(128)),          # avg 128
    ("A", 128, 1, True, _nine(128)),           # reso 1: one cell per tile
    ("A", 256, 8, True, _nine(256)),
    ("A", 384, 8, True, _nine(384)),
    ("G", 512, 8, True, _nine(512)),           # ragged, empty tiles
    ("A", 1024, 4, True, _nine(1024)),
    ("A", 4, 64, True, _gather(4, 1)),         # Morton, avg 1
    ("A", 8, 32, True, _gather(8, 2)),         # avg 5
    ("H", 4, 64, True, _gather(4, 4)),         # avg 8
    ("A", 16, 16, True, _gather(16, 8)),       # avg 23
    ("H", 16, 8, True, _gather(16, 8)),        # avg 512, the 20 000-row cell
    ("H", 4, 16, True, _gather(4, 8)),         # avg 128
    ("M", 4, 100, True, _gather(4, 1)),        # row-major keys
    ("M", 32, 100, True, _gather(32, 1)),      # row-major keys take the gather even at C = 32
    ("M10", 16, 10, True, _gather(16, 8)),     # row-major, avg 40
    ("A", 32, 64, False, _gather(32, 1)),      # NULL workspace on a Morton level (t2h.h documents the switch)
    ("H", 64, 16, False, _gather(64, 8)),
]


def _sample_bwd(c, C, r, g, with_ws):
    """t2h_bilinear_sample_bwd on rows in sorted order (the model path) -> (grad_plane, kernel names)"""
    topo = c.topo()
    n = c.n
    n_seg, shift, morton = c.level(r)
    g_dev = g[c.perm].cuda()
    nb = int(_lib().t2h_bilinear_sample_bwd_workspace_bytes(r, C, n, n_seg, morton)) if with_ws else 0
    ws = nan_workspace(nb) if with_ws else None
    out = nan_f32(c.B, r, r, C)
    names = launched(lambda: _call("t2h_bilinear_sample_bwd", _p(g_dev), n, r, C, _p(topo.xyz_sorted), 4, None,
                                   _p(topo.keys_sorted), _p(topo.cell_start), n_seg, shift, morton, _p(ws), nb, _p(out)))
    return out, names


@pytest.mark.gpu
@pytest.mark.parametrize("name,C,r,with_ws,kernels", SAMPLE_BWD_CASES,
                         ids=[f"{k[0].split('<')[0].replace('sample_bwd_', '')}-{a}-C{b}-r{c}{'' if d else '-nullws'}"
                              for a, b, c, d, k in SAMPLE_BWD_CASES])
def test_sample_bwd_paths(name, C, r, with_ws, kernels):
    c = cloud(name)
    g = torch.randn(c.n, C, generator=torch.Generator().manual_seed(C * 7 + r))
    out, names = _sample_bwd(c, C, r, g, with_ws)
    expect(names, *kernels, only="sample_bwd")
    idx, w = sample_taps(c.xy, c.tile, r)
    ref, A, nt = sample_bwd_ref(g, idx, w, c.B * r * r)
    assert_bound(out.view(-1, C), ref, A, nt, f"sample bwd {name} C={C} r={r} ws={with_ws}")


HEAVY_LEVELS = (64, 32, 16)
HEAVY_CASES = [(32, 64, _wtile(32, 4)), (128, 32, _wtile(128, 2)), (32, 16, _nine(32)), (64, 16, _nine(64)),
               (256, 16, _nine(256)), (4, 64, _gather(4, 2)), (8, 16, _gather(8, 8))]


@pytest.mark.gpu
@pytest.mark.parametrize("C,r,kernels", HEAVY_CASES, ids=[f"C{a}-r{b}" for a, b, _ in HEAVY_CASES])
def test_sample_bwd_heavy_cell_exact(C, r, kernels):
    """20 000 points at one dyadic coordinate (a cell edge at every level): every path must sum the chunk partials
    of that cell without losing one, bit for bit."""
    c = cloud("E")
    g = int_tensor((c.n, C), C + r)
    out, names = _sample_bwd(c, C, r, g, True)
    expect(names, *kernels, only="sample_bwd")
    idx, w = sample_taps(c.xy, c.tile, r)
    ref, A, _ = sample_bwd_ref(g, idx, w, r * r)
    assert_exact_budget(A, sample_m_bwd(c, idx, w, r * r), f"heavy C={C} r={r}")
    assert_bitwise(out.view(-1, C).cpu(), ref.float(), f"heavy sample bwd C={C} r={r}")


# =====================================================================================================
# 2 / 3. up-sampling: a sweep of sizes for one C, every C once
# =====================================================================================================
def _upsample_sizes():
    sizes = [(1, 1, 1, 1), (1, 1, 80, 80), (40, 40, 1, 1), (1, 40, 80, 1), (40, 1, 1, 80), (40, 40, 80, 80),
             (2, 2, 1, 80), (33, 17, 20, 9), (40, 40, 39, 41), (3, 40, 79, 2)]
    g = np.random.default_rng(7)
    for h in (1, 2, 3, 5, 8, 13, 21, 34, 40):
        for _ in range(6):
            sizes.append((h, int(g.integers(1, 41)), int(g.integers(1, 81)), int(g.integers(1, 81))))
    return sizes


def _upsample_case(C, h, w, oh, ow, seed):
    B = 2
    gen = torch.Generator().manual_seed(seed)
    x = torch.randn(B, h, w, C, generator=gen)
    gy = torch.randn(B, oh, ow, C, generator=gen)
    x_dev, gy_dev = x.cuda(), gy.cuda()
    out, gx = nan_f32(B, oh, ow, C), nan_f32(B, h, w, C)
    _call("t2h_upsample_bilinear_fwd", _p(x_dev), B, h, w, C, oh, ow, _p(out))
    _call("t2h_upsample_bilinear_bwd", _p(gy_dev), B, h, w, C, oh, ow, _p(gx))
    ref, A, nt = upsample_fwd_ref(x, oh, ow)
    assert_bound(out, ref, A, nt, f"upsample fwd C={C} {h}x{w} -> {oh}x{ow}")
    ref, A, nt = upsample_bwd_ref(gy, h, w)
    assert_bound(gx, ref, A, nt, f"upsample bwd C={C} {h}x{w} -> {oh}x{ow}")


@pytest.mark.gpu
def test_upsample_size_sweep():
    """h, w in 1..40 against out_h, out_w in 1..80: down-sampling, out_h != out_w, the degenerate axes out = 1 and
    h = 1, and the candidate window of the gather backward over many size ratios"""
    def sweep():
        for i, s in enumerate(_upsample_sizes()):
            _upsample_case(8, *s, seed=i)
    names = launched(sweep)
    expect(names, f"upsample_fwd_kernel<{RS(8)}>", f"upsample_bwd_kernel<{RS(8)}>")


@pytest.mark.gpu
@pytest.mark.parametrize("C", SUPPORTED_C)
def test_upsample_every_c(C):
    names = launched(lambda: _upsample_case(C, 7, 5, 12, 3, seed=C))
    expect(names, f"upsample_fwd_kernel<{RS(C)}>", f"upsample_bwd_kernel<{RS(C)}>")


# =====================================================================================================
# 4. n_rows * C > 2^31
# =====================================================================================================
def _morton(ix, iy):
    def part(v):
        v = v & 0xFFFF
        v = (v | (v << 8)) & 0x00FF00FF
        v = (v | (v << 4)) & 0x0F0F0F0F
        v = (v | (v << 2)) & 0x33333333
        return (v | (v << 1)) & 0x55555555
    return part(ix) | (part(iy) << 1)


@pytest.mark.gpu
def test_large_index_c512():
    """4.2 M rows x 512 channels (> 2^31 elements): broadcast, sum, max backward and sampling forward, checked exactly
    on a few thousand rows and cells including the last ones.  Features are integer functions of (row, channel)."""
    free, _ = torch.cuda.mem_get_info()
    if free < 48e9:
        pytest.skip(f"needs ~48 GB of free device memory, {free / 1e9:.1f} GB free")
    from tomosar2height_b200.topology import Topology
    from tomosar2height_b200.tests_support import demorton
    B, N, R, C = 16, 262500, 128, 512
    n, n_seg = B * N, B * R * R
    assert n * C > 2 ** 31
    gen = torch.Generator().manual_seed(99)
    xy = (torch.randint(1, 1024, (n, 2), generator=gen).float() / 1024)
    topo = Topology(xy.view(B, N, 2).cuda(), R)
    perm = topo.perm.long().cpu().numpy()
    keys = topo.keys_sorted.long().cpu().numpy()
    cs = topo.cell_start.long().cpu().numpy()
    ch = np.arange(C)

    def feat(rows):  # f(row, c), integer in [-8, 8]
        return ((np.asarray(rows)[:, None] * 7 + ch[None, :] * 3) % 17 - 8).astype(np.float64)

    def pval(prows):  # plane P(prow, c)
        return ((np.asarray(prows)[:, None] * 5 + ch[None, :]) % 17 - 8).astype(np.float64)

    def prow_of_seg(seg):
        b, code = seg // (R * R), seg % (R * R)
        ix, iy = demorton(torch.as_tensor(code))
        return b * R * R + iy.numpy() * R + ix.numpy()

    rng = np.random.default_rng(3)
    pos = np.unique(np.concatenate([rng.integers(0, n, 2000), np.arange(n - 64, n), np.arange(64)]))
    segs = np.unique(np.concatenate([rng.integers(0, n_seg, 1500), np.arange(n_seg - 64, n_seg), keys[-8:]]))
    prow_pos = prow_of_seg(keys[pos])
    pos_dev = torch.as_tensor(pos).cuda()

    def fill(rows_fn, m):
        t = torch.empty(m, C, dtype=torch.float32, device="cuda")
        chd = torch.arange(C, device="cuda")
        for a in range(0, m, 1 << 18):
            r = torch.arange(a, min(a + (1 << 18), m), device="cuda")
            t[a:a + r.numel()] = rows_fn(r[:, None], chd[None, :]).float()
        return t

    P = fill(lambda r, c: (r * 5 + c) % 17 - 8, n_seg)                       # plane in row-major (b, y, x) order
    # sampling forward (rows in original order through perm)
    out = nan_f32(n, C)
    _call("t2h_bilinear_sample_fwd", _p(P), R, C, _p(topo.xyz_sorted), 4, _p(topo.perm), None, n, N, _p(out))
    got = out[torch.as_tensor(perm[pos]).cuda()].double().cpu().numpy()
    idx, w = sample_taps(xy[perm[pos]], torch.as_tensor(perm[pos] // N), R)
    want = sum(w[:, t, None].double().numpy() * pval(idx[:, t].numpy()) for t in range(4))
    assert np.array_equal(got, want), "sample fwd at > 2^31 elements"
    del out
    # broadcast (rows in sorted order)
    out = nan_f32(n, C)
    _call("t2h_seg_broadcast", _p(P), n, None, _p(topo.keys_sorted), _p(topo.cell_start), n_seg, 0, C, 1, R, 0, _p(out))
    assert np.array_equal(out[pos_dev].double().cpu().numpy(), pval(prow_pos)), "seg_broadcast at > 2^31 elements"
    del out
    # sum
    F = fill(lambda r, c: (r * 7 + c * 3) % 17 - 8, n)
    nb = int(_lib().t2h_seg_workspace_bytes(n, n_seg, C))
    ws = nan_workspace(nb)
    plane = nan_f32(n_seg, C)
    _call("t2h_seg_reduce_fwd", _p(F), n, None, _p(topo.keys_sorted), _p(topo.cell_start), n_seg, 0, C, 1, R, 0, _p(ws), nb,
          _p(plane))
    prows = prow_of_seg(segs)
    got = plane[torch.as_tensor(prows).cuda()].double().cpu().numpy()
    want = np.stack([feat(np.arange(cs[s], cs[s + 1])).sum(0) for s in segs])
    assert np.array_equal(got, want), "seg_reduce_fwd at > 2^31 elements"
    del plane
    # max backward with both gradients: arg = the first row of the cell on even channels, the last on odd ones
    prow = torch.arange(n_seg, device="cuda")
    b, rem = prow // (R * R), prow % (R * R)
    seg_of_prow = b * R * R + _morton(rem % R, rem // R)
    cs_dev = topo.cell_start.long()
    beg, end = cs_dev[seg_of_prow], cs_dev[seg_of_prow + 1]
    pick = torch.where(torch.arange(C, device="cuda")[None, :] % 2 == 0, beg[:, None], end[:, None] - 1)
    arg = torch.where((end > beg)[:, None], pick, -1).int()
    del pick
    out = nan_f32(n, C)
    _call("t2h_seg_max_bwd", _p(F), _p(P), n, None, _p(topo.keys_sorted), _p(topo.cell_start), n_seg, 0, C, 1, R, _p(arg),
          _p(ws), nb, _p(out))
    got = out[pos_dev].double().cpu().numpy()
    seg_pos = keys[pos]
    tot = np.stack([feat(np.arange(cs[s], cs[s + 1])).sum(0) for s in seg_pos]) + pval(prow_pos)
    mine = np.where(ch[None, :] % 2 == 0, cs[seg_pos][:, None], cs[seg_pos + 1][:, None] - 1) == pos[:, None]
    assert np.array_equal(got, np.where(mine, tot, 0.0)), "seg_max_bwd at > 2^31 elements"


# =====================================================================================================
# summary
# =====================================================================================================
REQUIRED = sorted({k.replace(" ", "") for case in SAMPLE_BWD_CASES for k in case[-1]}
                  | {f"sample_bwd_wtile_rows_kernel<{c},{tw}>" for c, tw in ((32, 4), (64, 4), (128, 2))}
                  | {f"sample_bwd_nine_rows_kernel<{l}>" for l in (8, 16, 32)}
                  | {f"sample_bwd_kernel<{RS(c)},{wps}>" for c, wps in ((4, 1), (8, 2), (4, 4), (4, 8), (16, 8), (32, 1))}
                  | {k for C in SUPPORTED_C for k in _seg_kernels(C)}
                  | {f"sample_fwd_kernel<{RS(C)}>" for C in SUPPORTED_C}
                  | {f"upsample_{d}_kernel<{RS(C)}>" for C in SUPPORTED_C for d in ("fwd", "bwd")})


_PATH_CASES = (len(SEG_CASES) + 2 * len(SUPPORTED_C) + len(SAMPLE_BWD_CASES) + len(HEAVY_CASES) + 1 + len(SUPPORTED_C))
_DONE = set()


@pytest.fixture(autouse=True)
def _record_case(request):
    yield
    if "gpu" in request.node.keywords:
        _DONE.add(request.node.nodeid)


@pytest.mark.gpu
def test_zz_every_kernel_instance_was_reached(request):
    """When the whole path matrix ran, the union of the kernels seen covers every instance the dispatch can pick."""
    ran = {d for d in _DONE if "test_large_index" not in d}
    if len(ran) < _PATH_CASES or request.session.testsfailed:
        pytest.skip(f"only meaningful when all {_PATH_CASES} path cases ran and passed ({len(ran)} ran)")
    seen = "\n".join(sorted(_SEEN))
    missing = [k for k in REQUIRED if k not in seen]
    print("kernel instances reached:\n  " + "\n  ".join(k for k in REQUIRED if k in seen))
    assert not missing, f"never reached: {missing}"
