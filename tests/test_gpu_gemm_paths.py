"""Every dispatch path of the tensor-core GEMM kernels (t2h_linear.cu) against exact and fp64 references.

The linear forward / input-gradient GEMM, the implicit-GEMM 3x3 convolution, both weight gradients, the bias column
sums and the 3xFP16 helpers pick among many template instances from n_out, the row count, K and the epilogue.  Each
case below reaches one such instance through its natural trigger, asserts by the profiler's kernel names that it did
(and that no other instance of the family ran), and compares the result with a reference that detects one wrong term.
All references are computed on the CPU in fp64, which is exact for the integer data below (every sum < 2^53).

- Integer mode (bitwise).  Operands, gradients, masks, residuals and biases are small integers, nonzero in most
  entries.  Then the TF32 and FP16 `lo` parts are 0, the FP16 power-of-two scale is exact and every product is exact.
  The builders assert that every element's sum|x_k w_k| + |bias| + |residual| <= 2^21, so that every partial sum,
  in any order and any split of the rows, is an integer an fp32 accumulator holds exactly (3 bits of headroom below
  2^24 for an accumulator that keeps 24 bits under its largest addend; `test_a_accumulator_is_exact_for_integers`
  checks that assumption first).  The kernels must then equal the reference bit for bit (+0 and -0 compare equal).
- Split mode (bitwise).  Exactly one operand has 12 significant bits (odd integers in +-[2049, 4095]), the other is
  an integer in +-{1, 2}.  TF32 truncation gives hi = +-(|v| - 1), lo = +-1; the FP16 split of the scaled value
  (8 v, ulp 16) is a round-to-nearest-even tie with lo = +-8.  The dropped lo*lo product is 0, so the result is still
  exact, but a missing or doubled hi*lo / lo*hi product changes an element by at least 1.
- Random data (per-element bound).  |got - ref| <= (c1 2^-22 + (K + 2) 2^-24) A (+ the FP16 floor) for every
  element, A = sum_k |x_k w_k| + |bias| + |residual|.  The constants follow from the operand splits in
  include/t2h.h:
    3xTF32: hi = v with the low 13 mantissa bits cleared, so |lo| < 2^-10 |v|; the tensor core reads lo as TF32
      (truncated), an error < 2^-21 |v|.  x w - (x_h w_h + x_h w_l' + x_l' w_h) = x_l w_l + x_h (w_l - w_l') +
      (x_l - x_l') w_h, below (2^-20 + 2^-21 + 2^-21) |x w| = 8 * 2^-22 |x w|: c1 = 8.
    3xFP16: scaled v = hi + lo + d with |lo| <= 2^-11 |v| (+ 2^-25 for fp16 subnormals), |d| <= 2^-11 |lo|.  The
      dropped lo*lo and the two rounding errors d each contribute at most 2^-22 |x w|: c1 = 3 (the header's 2^-22
      per product is the size of each of these three terms).  An entry tiny against its operand's maximum loses
      up to half an fp16 subnormal step, 2^-25 in scaled units, against a scaled maximum >= 2^14: an absolute
      2^-39 max|x| |w_k| (and 2^-39 max|w| |x_k|) per product.
    Accumulation: every MMA adds 3 x 8 (TF32) or 3 x 16 (FP16) products into the fp32 accumulator and rounds at
      most once per instruction, so fewer than K roundings of at most 2^-24 of the running |sum| <= A; the bias
      and residual additions are two more.
  No element may exceed its bound.

Outputs and workspaces of the direct C-ABI calls are pre-filled with NaN (gap columns of strided outputs with the
bit pattern 0x7fc0dead, which must survive), so an element a kernel never writes, or a workspace slot it reads
without writing, fails the comparison.
"""
import numpy as np
import pytest
import torch

BUDGET = 2.0 ** 21
U = 2.0 ** -24
NAN_BITS = 0x7FC0DEAD
F16_FLOOR = 2.0 ** -39

_SEEN = set()   # every (normalised) kernel name the profiler reported in this session


# =====================================================================================================
# references and operand builders (CPU)
# =====================================================================================================
def split_tf32_np(v):
    """t2h::tc::split_tf32: hi = v with the low 13 mantissa bits cleared, lo = fp32(v - hi)"""
    v = np.asarray(v, dtype=np.float32)
    hi = (v.view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)
    return hi, (v - hi).astype(np.float32)


def f16_scale_exp_np(absmax_bits):
    """f16_scale_exp: e = 14 - floor(log2 max), clamped to [-63, 63]; 0 for a zero / subnormal maximum"""
    biased = (int(absmax_bits) >> 23) & 0xFF
    if biased == 0:
        return 0
    return max(-63, min(63, 14 - (biased - 127)))


def absmax_bits_np(*arrays):
    """bit pattern of max |v| (NaN sorts above infinity, as an unsigned maximum)"""
    return max([int((np.asarray(a, dtype=np.float32).view(np.uint32) & np.uint32(0x7FFFFFFF)).max(initial=0))
                for a in arrays])


def split_f16_np(v, absmax_bits):
    """split_f16x2 under the scale of absmax_bits: s = fp32(v * 2^e), hi = rn16(s), lo = rn16(fp32(s - hi))"""
    v = np.asarray(v, dtype=np.float32)
    s = (v * np.float32(2.0 ** f16_scale_exp_np(absmax_bits))).astype(np.float32)
    hi = s.astype(np.float16)
    lo = (s - hi.astype(np.float32)).astype(np.float32).astype(np.float16)
    return hi, lo


def ints(rng, shape, amax=7, zeros=0.0):
    """integers in +-[1, amax]; a fraction `zeros` of them set to 0"""
    v = rng.integers(1, amax + 1, size=shape) * rng.choice([-1, 1], size=shape)
    if zeros:
        v = np.where(rng.random(shape) < zeros, 0, v)
    return v.astype(np.float64)


def split12(rng, shape):
    """odd integers in +-[2049, 4095]: 12 significant bits, so the TF32 / FP16 lo part is +-1 (unscaled)"""
    return (2 * rng.integers(1025, 2048, size=shape) - 1) * rng.choice([-1.0, 1.0], size=shape)


def mask_values(rng, shape):
    """integers in [-2, 2] with a share of exact -0.0: only the strictly positive entries keep the result"""
    m = rng.integers(-2, 3, size=shape).astype(np.float64)
    neg0 = (m == 0) & (rng.random(shape) < 0.5)
    m[neg0] = -0.0
    return m


def act(x, relu):
    return np.maximum(x, 0.0) if relu else x


def gemm_ref(x, w, bias=None, relu=False, mask=None, res=None):
    """act(x) @ w^T (+ bias) (zeroed where mask <= 0) (+ res) in fp64, and A = sum|x w| + |bias| + |res|"""
    xa = act(x, relu)
    ref = xa @ w.T
    A = np.abs(xa) @ np.abs(w).T
    if bias is not None:
        ref = ref + bias[None, :]
        A = A + np.abs(bias)[None, :]
    if mask is not None:
        ref = np.where(mask > 0, ref, 0.0)
    if res is not None:
        ref = ref + res
        A = A + np.abs(res)
    return ref, A


def assert_budget(A, what):
    assert float(np.max(A, initial=0.0)) <= BUDGET, f"{what}: integer budget exceeded ({float(np.max(A)):.0f} > 2^21)"


def im2col(x, relu=False):
    """channels-last (B, H, W, C) -> (B*H*W, 9*C) with k = (3*ky + kx)*C + c, zero padding 1"""
    B, H, W, C = x.shape
    xp = np.zeros((B, H + 2, W + 2, C))
    xp[:, 1:-1, 1:-1] = act(x, relu)
    cols = [xp[:, ky:ky + H, kx:kx + W] for ky in range(3) for kx in range(3)]
    return np.concatenate(cols, axis=3).reshape(B * H * W, 9 * C)


def tf32_bound(A, K):
    return (8 * 2.0 ** -22 + (K + 2) * U) * A


def f16_bound(A, K, xa_abs, w_abs, x_max, w_max):
    """per element (c1 2^-22 + (K + 2) 2^-24) A + 2^-39 (max|x| sum_k |w_k| + max|w| sum_k |x_k|)"""
    floor = F16_FLOOR * (x_max * w_abs.sum(1)[None, :] + w_max * xa_abs.sum(1)[:, None])
    return (3 * 2.0 ** -22 + (K + 2) * U) * A + floor


# =====================================================================================================
# CPU self-tests of the emulations and builders
# =====================================================================================================
def test_split_tf32_emulation_hand_computed():
    # 4095 = 0x457ff000: the low 13 mantissa bits hold the last set bit -> hi 4094, lo 1; 2049 -> 2048 + 1
    hi, lo = split_tf32_np(np.array([4095.0, -2049.0, 1.0 + 2.0 ** -10, 1.0 + 2.0 ** -11, 3.0], dtype=np.float32))
    assert hi.view(np.uint32).tolist() == [0x457FE000, 0xC5000000, 0x3F802000, 0x3F800000, 0x40400000]
    assert lo.tolist() == [1.0, -1.0, 0.0, 2.0 ** -11, 0.0]
    v = np.float32(1.2345678)
    h, l = split_tf32_np(v)
    assert h.view(np.uint32) == 0x3F9E0000 and np.float32(h + l) == v
    # every 12-bit split operand has lo = +-1 exactly
    v = split12(np.random.default_rng(0), 4096)
    h, l = split_tf32_np(v)
    assert np.array_equal(np.abs(l), np.ones(4096, np.float32)) and np.array_equal(h + l, v.astype(np.float32))


def test_split_f16_emulation_hand_computed():
    assert f16_scale_exp_np(np.float32(4095).view(np.uint32)) == 3
    assert f16_scale_exp_np(np.float32(7).view(np.uint32)) == 12
    assert f16_scale_exp_np(np.float32(2.0 ** -49).view(np.uint32)) == 63
    assert f16_scale_exp_np(np.float32(2.0 ** -50).view(np.uint32)) == 63   # clamped
    assert f16_scale_exp_np(np.float32(2.0 ** 77).view(np.uint32)) == -63
    assert f16_scale_exp_np(np.float32(2.0 ** 78).view(np.uint32)) == -63   # clamped
    assert f16_scale_exp_np(np.float32(1e-40).view(np.uint32)) == 0         # subnormal maximum: no scale
    assert f16_scale_exp_np(0) == 0
    m = int(np.float32(4095).view(np.uint32))
    # 8 * 4095 = 32760 = 2047.5 fp16 steps of 16: tie -> even 2048 -> hi 32768 (0x7800), lo -8 (0xc800)
    # 8 * 4093 = 32744 = 2046.5 steps: tie -> even 2046 -> hi 32736 (0x77fe), lo +8 (0x4800)
    hi, lo = split_f16_np(np.array([4095.0, 4093.0, -2049.0, 0.0]), m)
    assert hi.view(np.uint16).tolist() == [0x7800, 0x77FE, 0xF400, 0x0000]
    assert lo.view(np.uint16).tolist() == [0xC800, 0x4800, 0xC800, 0x0000]
    # tiny entries: 2^-25 scaled is half the smallest fp16 subnormal -> ties to 0 in hi and lo (the FP16 floor)
    hi, lo = split_f16_np(np.array([1.0, 2.0 ** -39, 3 * 2.0 ** -40]), int(np.float32(1.0).view(np.uint32)))
    assert hi.view(np.uint16).tolist() == [0x7400, 0x0000, 0x0001] and lo.view(np.uint16).tolist() == [0, 0, 0x8000]
    v = split12(np.random.default_rng(1), 4096)
    v[0] = 4095.0
    hi, lo = split_f16_np(v, absmax_bits_np(v))
    assert np.array_equal(np.abs(lo.astype(np.float64)), np.full(4096, 8.0))
    assert np.array_equal((hi.astype(np.float64) + lo.astype(np.float64)) / 8, v)


def test_builders_and_references():
    rng = np.random.default_rng(2)
    x, w = ints(rng, (50, 4608)), ints(rng, (8, 4608))
    assert np.count_nonzero(x) == x.size and np.abs(x).max() == 7
    ref, A = gemm_ref(x, w, bias=ints(rng, 8), res=ints(rng, (50, 8)))
    assert_budget(A, "K = 4608")
    with pytest.raises(AssertionError):
        assert_budget(gemm_ref(np.full((2, 42800), 7.0), np.full((2, 42800), -7.0))[1], "over")
    # fp32 sums of the integer products are order-independent: forward and backward order agree with fp64
    prods = (x[:, None, :] * w[None, :, :]).astype(np.float32)
    fwd = np.zeros(prods.shape[:2], np.float32)
    bwd = np.zeros(prods.shape[:2], np.float32)
    for k in range(prods.shape[2]):
        fwd += prods[:, :, k]
        bwd += prods[:, :, -1 - k]
    assert np.array_equal(fwd, x @ w.T) and np.array_equal(bwd, x @ w.T)
    # mask semantics: 0, -0.0 and negatives zero the result
    m = np.array([[1.0, 0.0, -0.0, -2.0]])
    assert gemm_ref(np.ones((1, 1)), np.ones((4, 1)), mask=m)[0].tolist() == [[1.0, 0.0, 0.0, 0.0]]
    # im2col against a direct 3x3 convolution with zero padding
    xc = ints(rng, (2, 8, 16, 3))
    wc = ints(rng, (5, 3, 3, 3))   # (cout, ky, kx, c)
    got = (im2col(xc) @ wc.reshape(5, -1).T).reshape(2, 8, 16, 5)
    want = np.zeros((2, 8, 16, 5))
    xp = np.pad(xc, ((0, 0), (1, 1), (1, 1), (0, 0)))
    for ky in range(3):
        for kx in range(3):
            want += np.einsum("bhwc,oc->bhwo", xp[:, ky:ky + 8, kx:kx + 16], wc[:, ky, kx])
    assert np.array_equal(got, want)


def test_bounds_hold_for_emulated_splits():
    """the per-element bounds contain the emulated 3xTF32 / 3xFP16 products summed in fp32 (one rounding per term)"""
    rng = np.random.default_rng(3)
    K = 256
    x = (rng.standard_normal((64, K)) * np.exp(rng.uniform(-8, 2, (64, 1)))).astype(np.float32)
    w = rng.standard_normal((16, K)).astype(np.float32)
    ref, A = gemm_ref(x.astype(np.float64), w.astype(np.float64))
    xh, xl = split_tf32_np(x)
    wh, wl = split_tf32_np(w)
    xl_t, wl_t = split_tf32_np(xl)[0], split_tf32_np(wl)[0]   # lo read as TF32 (truncated)
    acc = np.zeros((64, 16), np.float32)
    for k in range(K):
        for a, b in ((xl_t, wh), (xh, wl_t), (xh, wh)):
            acc = (acc + (a[:, k, None].astype(np.float64) * b[None, :, k]).astype(np.float32)).astype(np.float32)
    assert (np.abs(acc - ref) <= tf32_bound(A, K)).all()
    bx, bw = absmax_bits_np(x), absmax_bits_np(w)
    sx, sw = 2.0 ** f16_scale_exp_np(bx), 2.0 ** f16_scale_exp_np(bw)
    xh, xl = (t.astype(np.float64) / sx for t in split_f16_np(x, bx))
    wh, wl = (t.astype(np.float64) / sw for t in split_f16_np(w, bw))
    got = xl @ wh.T + xh @ wl.T + xh @ wh.T
    bound = f16_bound(A, K, np.abs(x), np.abs(w), np.abs(x).max(), np.abs(w).max())
    assert (np.abs(got - ref) <= bound).all()


# =====================================================================================================
# GPU plumbing: direct C-ABI calls with sentinel outputs, and the kernels they launched
# =====================================================================================================
def _call(name, *args):
    from tomosar2height_b200 import _lib
    _lib.call(name, *args)


def _p(t):
    from tomosar2height_b200._lib import ptr
    return ptr(t)


def _libh():
    from tomosar2height_b200 import _lib
    return _lib.load()


def norm_name(n):
    """profiler kernel name without spaces, argument list and demangler casts: `ns::k<true,128,0,false,false>`"""
    n = n.replace(" ", "").replace("(bool)0", "false").replace("(bool)1", "true").replace("(int)", "")
    return n.split(">(")[0] + ">" if ">(" in n else n.split("(")[0]


def launched(fn):
    """run fn under the profiler; the set of kernel names it launched"""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = {norm_name(e.name) for e in prof.events()}
    _SEEN.update(names)
    return names


def expect(names, *kernels, only=None):
    """every kernel in `kernels` ran; with only=prefix, no other kernel whose name contains the prefix ran"""
    for k in kernels:
        assert any(n.endswith(k) for n in names), f"kernel {k} did not run; launched: {sorted(names)}"
    if only is not None:
        extra = {n for n in names if only in n and not any(n.endswith(k) for k in kernels)}
        assert not extra, f"unexpected {only} kernels {sorted(extra)} (expected {kernels})"


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda()


def sentinel(rows, ld):
    return torch.full((rows, ld), NAN_BITS, dtype=torch.int32, device="cuda").view(torch.float32)


def placed(a, ld):
    """a (rows, k) in the first k columns of a (rows, ld) buffer whose other columns hold the NaN pattern"""
    buf = sentinel(a.shape[0], ld)
    buf[:, :a.shape[1]] = dev(a)
    return buf[:, :a.shape[1]], buf


def nan_workspace(nbytes):
    return torch.full((max(int(nbytes), 1),), 0xFF, dtype=torch.uint8, device="cuda")


def absmax_slot(x1, x2=None, rows=None):
    slot = torch.full((1,), 12345, dtype=torch.int32, device="cuda")
    _call("t2h_absmax", _p(x1), x1.stride(0), x1.shape[1], _p(x2), 0 if x2 is None else x2.stride(0),
          0 if x2 is None else x2.shape[1], x1.shape[0] if rows is None else rows, _p(slot))
    return slot


def split_weight(w_dev, f16):
    """(hi, lo[, w_slot]) of a contiguous (n, k) device weight by the library's own split kernels"""
    if not f16:
        hi, lo = torch.empty_like(w_dev), torch.empty_like(w_dev)
        _call("t2h_split_tf32", _p(w_dev), w_dev.numel(), _p(hi), _p(lo))
        return hi, lo
    slot = absmax_slot(w_dev)
    hi = torch.empty(w_dev.shape, dtype=torch.float16, device="cuda")
    lo = torch.empty_like(hi)
    _call("t2h_split_f16", _p(w_dev), w_dev.numel(), _p(slot), _p(hi), _p(lo))
    return hi, lo, slot


def assert_exact(got, ref, what):
    got = got.detach().cpu().double().numpy().reshape(ref.shape)
    same = got == ref
    if not same.all():
        i = tuple(np.argwhere(~same)[0])
        raise AssertionError(f"{what}: {int((~same).sum())} of {ref.size} elements differ; first at {i}: "
                             f"got {got[i]!r} want {ref[i]!r}")


def assert_within(got, ref, bound, what):
    got = got.detach().cpu().double().numpy().reshape(ref.shape)
    assert np.isfinite(got).all(), f"{what}: {int((~np.isfinite(got)).sum())} elements unwritten or non-finite"
    err = np.abs(got - ref)
    bad = err > bound
    if bad.any():
        i = tuple(np.argwhere(bad)[np.argmax((err - bound)[bad])])
        raise AssertionError(f"{what}: {int(bad.sum())} of {ref.size} elements outside the bound; worst at {i}: "
                             f"got {got[i]!r} ref {ref[i]!r} bound {bound[i]:.3e}")


def assert_gap_intact(buf, k, what):
    gap = buf[:, k:].view(torch.int32)
    assert bool((gap == NAN_BITS).all()), f"{what}: {int((gap != NAN_BITS).sum())} padding elements were written"


def P(f16, bn, pair=False, ds=False):
    return f"linear_x3_persistent_kernel<{str(f16).lower()},{bn},0,{str(pair).lower()},{str(ds).lower()}>"


T32, T64, T128 = P(False, 32), P(False, 64), P(False, 128)
F32, F64, F128 = P(True, 32), P(True, 64), P(True, 128)
FP, FDS, FW, FWDS = P(True, 128, True), P(True, 128, True, True), P(True, 256, True), P(True, 256, True, True)
LIN = "linear_x3_persistent_kernel"


def run_linear(f16, x1, w, bias=None, x2=None, relu=False, mask=None, res=None, ld_out=None, alias=False,
               out_max=False):
    """one t2h_linear_fwd[_f16] call on device operands (x1, x2, mask, res may be strided views); w is numpy.
    Returns (out view, its NaN-patterned buffer (None when out aliases res), kernel names, out_absmax slot)."""
    rows, k1 = x1.shape
    k2 = 0 if x2 is None else x2.shape[1]
    n_out = w.shape[0]
    split = split_weight(dev(w), f16)
    if alias:
        out, buf = res, None
    else:
        buf = sentinel(rows, ld_out or n_out)
        out = buf[:, :n_out]
    ld = out.stride(0)
    ml = 0 if mask is None else mask.stride(0)
    rl = 0 if res is None else res.stride(0)
    bias_d = None if bias is None else dev(bias)
    if f16:
        x_slot = absmax_slot(x1, x2)
        o_slot = torch.full((1,), 777, dtype=torch.int32, device="cuda") if out_max else None
        fn = lambda: _call("t2h_linear_fwd_f16", _p(x1), x1.stride(0), k1, _p(x2), 0 if x2 is None else x2.stride(0), k2,
                           rows, _p(x_slot), _p(split[0]), _p(split[1]), _p(split[2]), n_out, _p(bias_d), int(relu),
                           _p(mask), ml, _p(res), rl, _p(out), ld, _p(o_slot))
    else:
        o_slot = None
        fn = lambda: _call("t2h_linear_fwd", _p(x1), x1.stride(0), k1, _p(x2), 0 if x2 is None else x2.stride(0), k2,
                           rows, _p(split[0]), _p(split[1]), n_out, _p(bias_d), int(relu), _p(mask), ml, _p(res), rl,
                           _p(out), ld)
    names = launched(fn)
    return out, buf, names, o_slot


# =====================================================================================================
# 0. the hardware assumption behind the bitwise oracle
# =====================================================================================================
@pytest.mark.gpu
@pytest.mark.parametrize("f16", [False, True], ids=["tf32", "f16"])
def test_a_accumulator_is_exact_for_integers(f16):
    """Partial sums up to just below 2^21, built from addends of 1 to 49 over K = 42 784, must come out exact: the
    tcgen05 fp32 accumulator adds integers of that size without loss.  Every other bitwise case relies on this."""
    rng = np.random.default_rng(100)
    rows, K, n = 128, 42784, 32 if not f16 else 132
    x = np.full((rows, K), 7.0)
    x[rng.random((rows, K)) < 0.01] = 1.0
    w = np.full((n, K), 7.0)
    w[:, ::977] = -1.0
    ref, A = gemm_ref(x, w)
    assert_budget(A, "accumulator probe")
    assert np.abs(ref).max() > 2.0 ** 20.9
    out, _, names, _ = run_linear(f16, dev(x), w)
    expect(names, F128 if f16 else T32, only=LIN)
    assert_exact(out, ref, "accumulator probe")


# =====================================================================================================
# 1. linear forward / input-gradient GEMM: every instance, edge shapes and epilogues, integer mode
# =====================================================================================================
# (flavour, rows, k1, k2, n_out, epilogue flags, instance)
#   b bias, r relu_in (negative inputs), m mask (0 / -0.0 / negative), s residual, a residual aliasing out,
#   S strided operands (ld_x1 > k1, ld_x2 > k2, ld_out > n_out, ld_mask != ld_res != ld_out)
FWD_CASES = [
    # 3xTF32: rows around one and two 128-row tiles, every N-tile width and a ragged last N-block
    *[("tf32", r, 28, 0, 32, "b", T32) for r in (1, 127, 128, 129, 255, 256, 257)],
    *[("tf32", 257, 136, 0, n, "b", T32) for n in (4, 28, 32)],
    *[("tf32", 257, 136, 0, n, "b", T64) for n in (36, 60, 64)],
    *[("tf32", 257, 136, 0, n, "b", T128) for n in (68, 132, 200, 252, 256, 260, 512)],
    ("tf32", 300, 4, 0, 32, "b", T32), ("tf32", 300, 4, 0, 132, "b", T128),
    ("tf32", 300, 32, 36, 64, "br", T64), ("tf32", 300, 64, 4, 260, "br", T128),
    *[("tf32", 333, 64, 36, n, e, i) for n, i in ((28, T32), (60, T64), (260, T128))
      for e in ("", "br", "bm", "bs", "bms", "ba", "bmsS", "brmsS")],
    ("tf32", 19201, 64, 0, 32, "bs", T32), ("tf32", 19201, 64, 0, 260, "bm", T128),   # > 148 tiles per grid
    # 3xFP16: one-CTA instances, then CTA pairs (rows >= 256) and their flavours
    *[("f16", r, 136, 0, 32, "b", F32) for r in (1, 129, 257)],
    *[("f16", r, 136, 0, 64, "b", F64) for r in (1, 129, 257)],
    *[("f16", r, 136, 0, n, "b", F128) for r in (1, 127, 128, 129, 255) for n in (132,)],
    ("f16", 255, 136, 0, 512, "bm", F128), ("f16", 200, 8, 0, 68, "b", F128), ("f16", 200, 24, 0, 260, "br", F128),
    *[("f16", r, 136, 0, 132, "b", FP) for r in (256, 257, 300, 385)],
    *[("f16", 300, 136, 0, n, "b", FP) for n in (68, 200, 252, 260)],
    ("f16", 300, 128, 0, 256, "b", FP), ("f16", 300, 136, 0, 256, "b", FW),          # k_chunks 4 | 5
    ("f16", 300, 96, 40, 512, "br", FW), ("f16", 300, 64, 40, 512, "br", FP),        # concat, odd chunk count
    ("f16", 300, 256, 0, 132, "bm", FDS), ("f16", 300, 264, 0, 132, "bm", FP),       # k_chunks 8 | 9 with aux
    ("f16", 300, 256, 0, 512, "bs", FWDS), ("f16", 300, 288, 0, 512, "bs", FW),
    *[("f16", 300, 64, 72, n, e, FDS if n == 260 and set(e) & set("msa") else i)
      for n, i in ((28, F32), (60, F64), (260, FP)) for e in ("", "br", "bm", "bs", "bms", "ba", "bmsS", "brmsS")],
    *[("f16", 129, 64, 72, 260, e, F128) for e in ("bm", "bs", "bms", "ba", "bmsS")],
    *[("f16", 300, 96, 200, 260, e, FP) for e in ("bm", "bs", "bms", "ba", "bmsS")],
    *[("f16", 300, 160, 0, 512, e, FWDS) for e in ("bm", "bs", "bms", "ba", "bmsS")],
    *[("f16", 300, 320, 0, 512, e, FW) for e in ("bm", "bs", "bms", "ba", "bmsS")],
    ("f16", 19201, 64, 0, 132, "bs", FDS), ("f16", 19201, 160, 0, 132, "b", FP),      # odd M-tile count, > 74 pairs
    ("f16", 19201, 160, 0, 512, "bm", FWDS), ("f16", 19201, 320, 0, 512, "b", FW),
]


def _fwd_id(c):
    return f"{c[0]}-r{c[1]}-k{c[2]}+{c[3]}-n{c[4]}-{c[5] or 'plain'}"


@pytest.mark.gpu
@pytest.mark.parametrize("case", FWD_CASES, ids=_fwd_id)
def test_linear_fwd_integer(case):
    flavour, rows, k1, k2, n_out, epi, inst = case
    f16 = flavour == "f16"
    rng = np.random.default_rng(rows * 7919 + k1 * 31 + k2 * 7 + n_out + len(epi))
    strided = "S" in epi
    x1 = ints(rng, (rows, k1), zeros=0.05)
    x2 = ints(rng, (rows, k2), zeros=0.05) if k2 else None
    w = ints(rng, (n_out, k1 + k2))
    bias = ints(rng, n_out) * 100 if "b" in epi else None
    mask = mask_values(rng, (rows, n_out)) if "m" in epi else None
    res = ints(rng, (rows, n_out)) * 1000 if ("s" in epi or "a" in epi) else None
    x = x1 if x2 is None else np.concatenate([x1, x2], 1)
    ref, A = gemm_ref(x, w, bias, "r" in epi, mask, res)
    assert_budget(A, _fwd_id(case))
    x1_d, _ = placed(x1, k1 + 12 if strided else k1)
    x2_d = None if x2 is None else placed(x2, k2 + 4 if strided else k2)[0]
    mask_d = None if mask is None else placed(mask, n_out + 8 if strided else n_out)[0]
    ld_out = n_out + 4 if strided else n_out
    res_d = res_buf = None
    if "a" in epi:
        res_d, res_buf = placed(res, ld_out)
    elif res is not None:
        res_d = placed(res, n_out + 16 if strided else n_out)[0]
    out, buf, names, slot = run_linear(f16, x1_d, w, bias, x2_d, "r" in epi, mask_d, res_d, ld_out, "a" in epi,
                                       out_max=f16)
    expect(names, inst, only=LIN)
    assert_exact(out, ref, _fwd_id(case))
    assert_gap_intact(res_buf if "a" in epi else buf, n_out, _fwd_id(case))
    if slot is not None:
        assert slot.item() == int(np.float32(np.abs(ref).max()).view(np.int32)), "out_absmax"


@pytest.mark.gpu
@pytest.mark.parametrize("rows,n_out,K,inst", [(129, 132, 64, F128), (300, 132, 288, FP), (300, 132, 64, FDS),
                                               (129, 512, 64, F128), (385, 512, 160, FWDS), (300, 512, 160, FWDS),
                                               (300, 512, 320, FW), (19201, 260, 288, FP)])
def test_out_absmax_ignores_padding_rows(rows, n_out, K, inst):
    """The residual cancels the bias on every valid row, so |out| <= 4 K + 7 there, while the padding rows of the
    last tile (and the empty rank-1 tile of an odd pair count) hold the bias alone: out_absmax must be max |out| of
    the valid rows, bit for bit."""
    rng = np.random.default_rng(rows + n_out + K)
    x = ints(rng, (rows, K), amax=2)
    w = ints(rng, (n_out, K), amax=2)
    bias = ints(rng, n_out) * 4096
    res = np.broadcast_to(-bias, (rows, n_out)) + ints(rng, (rows, n_out))
    ref, A = gemm_ref(x, w, bias, res=res)
    assert_budget(A, "cancel")
    out, _, names, slot = run_linear(True, dev(x), w, bias, res=dev(res), out_max=True)
    expect(names, inst, only=LIN)
    assert_exact(out, ref, "cancelled bias")
    assert np.abs(ref).max() < 4096
    assert slot.item() == int(np.float32(np.abs(ref).max()).view(np.int32)), "out_absmax counted padding rows"


# split mode: (flavour, which operand carries the 12-bit values, n_out, instance)
SPLIT_FWD = [("tf32", "x", 132, T128), ("tf32", "w", 132, T128), ("tf32", "x", 28, T32), ("tf32", "w", 60, T64),
             ("f16", "x", 132, FP), ("f16", "w", 132, FP), ("f16", "x", 512, FW), ("f16", "w", 512, FW),
             ("f16", "x", 64, F64), ("f16", "w", 32, F32)]


@pytest.mark.gpu
@pytest.mark.parametrize("flavour,side,n_out,inst", SPLIT_FWD)
def test_linear_fwd_split_operand(flavour, side, n_out, inst):
    """One operand with 12 significant bits: the lo*hi / hi*lo products carry +-1 per term and must all be there."""
    rng = np.random.default_rng(len(side) + n_out)
    rows, K = 300, 200
    big = split12(rng, (rows, K) if side == "x" else (n_out, K))
    small = ints(rng, (n_out, K) if side == "x" else (rows, K), amax=2)
    x, w = (big, small) if side == "x" else (small, big)
    ref, A = gemm_ref(x, w)
    assert_budget(A, "split fwd")
    out, _, names, _ = run_linear(flavour == "f16", dev(x), w)
    expect(names, inst, only=LIN)
    assert_exact(out, ref, f"{flavour} split {side}")


@pytest.mark.gpu
def test_library_splits_match_emulation():
    """t2h_split_tf32 and t2h_split_f16 equal the numpy emulation bit for bit (random, 12-bit, tiny and scaled data)"""
    rng = np.random.default_rng(5)
    for v in (rng.standard_normal(4096) * 3, split12(rng, 4096), np.concatenate([[1.0], rng.standard_normal(4095) *
                                                                               2.0 ** -30]), rng.standard_normal(4096) * 1e20):
        v = v.astype(np.float32)
        v_d = dev(v.reshape(64, 64))
        got = {}
        names = launched(lambda: got.update(tf32=split_weight(v_d, False), f16=split_weight(v_d, True)))
        expect(names, "split_tf32_kernel", "split_f16_kernel", "::absmax_kernel")
        hi, lo = got["tf32"]
        h, l = split_tf32_np(v)
        assert np.array_equal(hi.cpu().numpy().reshape(-1).view(np.uint32), h.view(np.uint32))
        assert np.array_equal(lo.cpu().numpy().reshape(-1).view(np.uint32), l.view(np.uint32))
        hi, lo, slot = got["f16"]
        assert slot.item() == absmax_bits_np(v)
        h, l = split_f16_np(v, absmax_bits_np(v))
        assert np.array_equal(hi.cpu().numpy().reshape(-1).view(np.uint16), h.view(np.uint16))
        assert np.array_equal(lo.cpu().numpy().reshape(-1).view(np.uint16), l.view(np.uint16))


# =====================================================================================================
# 2. random data: per-element bound for the combined paths
# =====================================================================================================
RANDOM_CASES = [("tf32", 300, 64, 36, 28, T32), ("tf32", 300, 64, 36, 60, T64), ("tf32", 1000, 512, 0, 260, T128),
                ("f16", 300, 64, 72, 132, FDS), ("f16", 129, 64, 72, 260, F128), ("f16", 1000, 512, 0, 512, FW),
                ("f16", 300, 128, 32, 512, FWDS), ("f16", 300, 1024, 0, 132, FP), ("f16", 300, 96, 40, 32, F32)]


@pytest.mark.gpu
@pytest.mark.parametrize("flavour,rows,k1,k2,n_out,inst", RANDOM_CASES)
def test_linear_fwd_random_bound(flavour, rows, k1, k2, n_out, inst):
    """general fp32 data, both operands split, ReLU, concatenation, mask and residual: every element in its bound"""
    rng = np.random.default_rng(rows + k1 + k2 + n_out)
    f32 = lambda *s: rng.standard_normal(s).astype(np.float32).astype(np.float64)
    x1, x2 = f32(rows, k1), (f32(rows, k2) if k2 else None)
    w = f32(n_out, k1 + k2) / np.sqrt(k1 + k2)
    bias, mask, res = f32(n_out), f32(rows, n_out), f32(rows, n_out)
    x = x1 if x2 is None else np.concatenate([x1, x2], 1)
    ref, A = gemm_ref(x, w.astype(np.float32).astype(np.float64), bias, True, mask, res)
    out, _, names, _ = run_linear(flavour == "f16", dev(x1), w, bias, None if x2 is None else dev(x2), True,
                                  dev(mask), dev(res))
    expect(names, inst, only=LIN)
    K = k1 + k2
    if flavour == "f16":
        xa = np.abs(act(x, True))
        bound = f16_bound(A, K, xa, np.abs(w), np.abs(x).max(), np.abs(w).max())
    else:
        bound = tf32_bound(A, K)
    assert_within(out, ref, bound, f"{flavour} random")


# =====================================================================================================
# 3. FP16 operand scaling at its edges
# =====================================================================================================
@pytest.mark.gpu
def test_f16_zero_and_subnormal_operands():
    rng = np.random.default_rng(7)
    rows, K, n = 300, 136, 132
    bias, res = ints(rng, n) * 3, ints(rng, (rows, n))
    w = ints(rng, (n, K))
    for x, wt in ((np.zeros((rows, K)), w), (ints(rng, (rows, K)), np.zeros((n, K)))):
        out, _, names, slot = run_linear(True, dev(x), wt, bias, res=dev(res), out_max=True)
        expect(names, FDS, only=LIN)
        assert_exact(out, bias[None, :] + res, "zero operand")
        assert slot.item() == int(np.float32(np.abs(bias[None, :] + res).max()).view(np.int32))
    # a subnormal maximum gets no scale (and cannot be represented in fp16): the result is the bias, and without
    # a bias it is finite and no farther from the tiny exact value than that value itself
    xs = (rng.standard_normal((rows, K)) * 1e-39).astype(np.float32)
    assert absmax_bits_np(xs) < (1 << 23)
    out, _, _, _ = run_linear(True, dev(xs), w, bias)
    assert_exact(out, np.broadcast_to(bias, (rows, n)), "subnormal maximum with bias")
    out, _, _, _ = run_linear(True, dev(xs), w)
    ref, A = gemm_ref(xs.astype(np.float64), w)
    assert_within(out, ref, A, "subnormal maximum")


@pytest.mark.gpu
@pytest.mark.parametrize("x_max,w_max", [(2.0 ** -49, 1.0), (1.0, 2.0 ** -49), (2.0 ** -49, 2.0 ** -49),
                                         (2.0 ** 78 * (1 - 2.0 ** -24), 2.0 ** -49),
                                         (2.0 ** -49, 2.0 ** 78 * (1 - 2.0 ** -24)), (2.0 ** 40, 2.0 ** -40)])
def test_f16_scale_limits_within_documented_bound(x_max, w_max):
    """maxima at the clamp limits of f16_scale_exp (2^-49 and just under 2^78) against the documented bound"""
    rng = np.random.default_rng(8)
    rows, K, n = 300, 256, 260
    x = rng.uniform(-1, 1, (rows, K)) * np.exp2(rng.uniform(-12, 0, (rows, 1)))
    x = (x / np.abs(x).max() * x_max).astype(np.float32)
    x.reshape(-1)[17] = np.float32(x_max)
    w = (rng.uniform(-1, 1, (n, K)) * w_max).astype(np.float32)
    w.reshape(-1)[5] = np.float32(-w_max)
    x64, w64 = x.astype(np.float64), w.astype(np.float64)
    ref, A = gemm_ref(x64, w64)
    out, _, names, _ = run_linear(True, dev(x), w)
    expect(names, FP, only=LIN)
    bound = f16_bound(A, K, np.abs(x64), np.abs(w64), np.abs(x64).max(), np.abs(w64).max())
    assert_within(out, ref, bound, f"max|x| {x_max:.3g} max|w| {w_max:.3g}")


@pytest.mark.gpu
def test_f16_absolute_floor_is_reached():
    """An entry 2^-39 against an operand maximum of 1 (scaled: 2^-25, half the smallest fp16 subnormal) is lost in
    both hi and lo (round to nearest even): the error of those rows is exactly the documented absolute floor
    2^-39 max|x| |w|, so a smaller floor would not hold."""
    rows, K, n = 256, 128, 132
    x = np.zeros((rows, K), np.float32)
    x[0, 0] = 1.0
    x[1:, 3] = 2.0 ** -39
    w = np.ones((n, K), np.float32)
    ref, _ = gemm_ref(x.astype(np.float64), w.astype(np.float64))
    out, _, names, _ = run_linear(True, dev(x), w)
    expect(names, FP, only=LIN)
    err = np.abs(out.cpu().double().numpy() - ref)
    assert np.array_equal(err[0], np.zeros(n))
    assert np.array_equal(err[1:], np.full((rows - 1, n), F16_FLOOR * 1.0 * 1.0)), "floor not reached exactly"


# =====================================================================================================
# 4. 3x3 convolution (implicit GEMM), integer mode
# =====================================================================================================
CONV_CASES = [
    # (flavour, B, H, W, cin, cout, epilogue, instance)
    ("tf32", 1, 8, 16, 32, 4, "b", T32), ("tf32", 3, 16, 48, 32, 32, "br", T32), ("tf32", 3, 8, 16, 64, 64, "bm", T64),
    ("tf32", 1, 16, 48, 64, 128, "bs", T128), ("tf32", 3, 16, 16, 512, 256, "b", T128), ("tf32", 1, 8, 48, 32, 36, "brs", T64),
    ("f16", 1, 8, 16, 32, 4, "b", F32), ("f16", 3, 8, 16, 64, 32, "bm", F32), ("f16", 1, 16, 48, 32, 64, "bs", F64),
    ("f16", 1, 8, 16, 64, 128, "brm", F128), ("f16", 1, 8, 16, 512, 256, "bs", F128),
    ("f16", 3, 8, 16, 64, 128, "b", FP), ("f16", 3, 8, 16, 32, 256, "bm", FP), ("f16", 3, 16, 48, 512, 128, "brs", FP),
    ("f16", 1, 16, 16, 64, 132, "bs", FP),
]


def _conv_id(c):
    return f"{c[0]}-B{c[1]}H{c[2]}W{c[3]}-c{c[4]}to{c[5]}-{c[6]}"


@pytest.mark.gpu
@pytest.mark.parametrize("case", CONV_CASES, ids=_conv_id)
def test_conv3x3_fwd_integer(case):
    flavour, B, H, W, cin, cout, epi, inst = case
    f16 = flavour == "f16"
    rng = np.random.default_rng(B * 1000 + H * 100 + W + cin + cout)
    x = ints(rng, (B, H, W, cin), zeros=0.05)
    w = ints(rng, (cout, 9 * cin))
    bias = ints(rng, cout) * 100 if "b" in epi else None
    rows = B * H * W
    mask = mask_values(rng, (rows, cout)) if "m" in epi else None
    res = ints(rng, (rows, cout)) * 1000 if "s" in epi else None
    cols = im2col(x, "r" in epi)
    ref, A = gemm_ref(cols, w, bias, False, mask, res)
    assert_budget(A, _conv_id(case))
    x_d = dev(x)
    out = torch.full((B, H, W, cout), float("nan"), device="cuda")
    split = split_weight(dev(w), f16)
    bias_d, mask_d, res_d = (None if a is None else dev(a) for a in (bias, mask, res))
    relu = int("r" in epi)
    if f16:
        x_slot = absmax_slot(x_d.view(rows, cin))
        o_slot = torch.full((1,), 777, dtype=torch.int32, device="cuda")
        fn = lambda: _call("t2h_conv3x3_fwd_f16", _p(x_d), B, H, W, cin, _p(x_slot), _p(split[0]), _p(split[1]),
                           _p(split[2]), cout, _p(bias_d), relu, _p(mask_d), _p(res_d), _p(out), _p(o_slot))
    else:
        fn = lambda: _call("t2h_conv3x3_fwd", _p(x_d), B, H, W, cin, _p(split[0]), _p(split[1]), cout, _p(bias_d),
                           relu, _p(mask_d), _p(res_d), _p(out))
    expect(launched(fn), inst, only=LIN)
    assert_exact(out.view(rows, cout), ref, _conv_id(case))
    if f16:
        assert o_slot.item() == int(np.float32(np.abs(ref).max()).view(np.int32)), "conv out_absmax"


@pytest.mark.gpu
@pytest.mark.parametrize("flavour", ["tf32", "f16"])
def test_conv3x3_fwd_random_bound(flavour):
    """random fp32 data at the deepest K (cin = 512, K = 4608) on the per-element bound"""
    rng = np.random.default_rng(11)
    B, H, W, cin, cout = 1, 8, 32, 512, 128
    x = rng.standard_normal((B, H, W, cin)).astype(np.float32).astype(np.float64)
    w = (rng.standard_normal((cout, 9 * cin)) / 64).astype(np.float32).astype(np.float64)
    bias = rng.standard_normal(cout).astype(np.float32).astype(np.float64)
    cols = im2col(x, True)
    ref, A = gemm_ref(cols, w, bias)
    out = torch.full((B, H, W, cout), float("nan"), device="cuda")
    x_d = dev(x)
    split = split_weight(dev(w), flavour == "f16")
    if flavour == "f16":
        x_slot = absmax_slot(x_d.view(-1, cin))
        _call("t2h_conv3x3_fwd_f16", _p(x_d), B, H, W, cin, _p(x_slot), _p(split[0]), _p(split[1]), _p(split[2]), cout,
              _p(dev(bias)), 1, None, None, _p(out), None)
        bound = f16_bound(A, 9 * cin, np.abs(cols), np.abs(w), np.abs(x).max(), np.abs(w).max())
    else:
        _call("t2h_conv3x3_fwd", _p(x_d), B, H, W, cin, _p(split[0]), _p(split[1]), cout, _p(dev(bias)), 1, None, None,
              _p(out))
        bound = tf32_bound(A, 9 * cin)
    assert_within(out.view(-1, cout), ref, bound, f"conv {flavour} random")


# =====================================================================================================
# 5. weight gradients (+ bias gradient) and their row-split reduction, integer mode
# =====================================================================================================
def expect_wgrad(names, inst):
    """`inst` ran and no other weight-gradient GEMM instance (the reduce kernels are checked separately)"""
    expect(names, inst)
    extra = {n for n in names if ("wgrad_x3_kernel" in n or "wgrad_f16_pair_kernel" in n) and not n.endswith(inst)}
    assert not extra, f"unexpected weight-gradient kernels {sorted(extra)} (expected {inst})"


def wg_inst(f16, k_in, pair=False):
    if pair:
        return "wgrad_f16_pair_kernel"
    if f16:
        return "wgrad_x3_kernel<128,true>"
    return f"wgrad_x3_kernel<{32 if k_in <= 32 else 64 if k_in <= 64 else 128},false>"


def run_wgrad(f16, g_d, x_d, n_out, k_in, relu, ld_w, with_bias, rows=None):
    rows = g_d.shape[0] if rows is None else rows
    nb = int(_libh().t2h_linear_wgrad_workspace_bytes(rows, n_out, k_in))
    ws = nan_workspace(nb)
    gw_buf = sentinel(n_out, ld_w)
    gw = gw_buf[:, :k_in]
    gb = torch.full((n_out,), float("nan"), device="cuda") if with_bias else None
    if f16:
        g_slot, x_slot = absmax_slot(g_d, rows=rows), absmax_slot(x_d, rows=rows)
        fn = lambda: _call("t2h_linear_wgrad_f16", _p(g_d), g_d.stride(0), _p(g_slot), _p(x_d), x_d.stride(0), _p(x_slot),
                           rows, n_out, k_in, int(relu), _p(ws), nb, _p(gw), ld_w, _p(gb))
    else:
        fn = lambda: _call("t2h_linear_wgrad", _p(g_d), g_d.stride(0), _p(x_d), x_d.stride(0), rows, n_out, k_in, int(relu),
                           _p(ws), nb, _p(gw), ld_w, _p(gb))
    return gw, gw_buf, gb, launched(fn)


# (flavour, rows, n_out, k_in, relu, pair, reduce instance)
WGRAD_CASES = [
    ("tf32", 1, 32, 28, False, False, 1), ("tf32", 31, 4, 32, True, False, 1), ("tf32", 33, 36, 64, False, False, 1),
    ("tf32", 100, 132, 60, True, False, 1), ("tf32", 1000, 32, 28, False, False, 8), ("tf32", 1000, 132, 132, True, False, 8),
    ("tf32", 5000, 4, 32, True, False, 32), ("tf32", 4737, 28, 64, False, False, 32), ("tf32", 4737, 260, 260, True, False, 32),
    ("tf32", 2049, 128, 68, False, False, 32), ("tf32", 20000, 64, 136, True, False, 32),
    ("f16", 1, 132, 68, False, False, 1), ("f16", 100, 32, 132, True, False, 1), ("f16", 1000, 132, 260, False, False, 8),
    ("f16", 5000, 128, 68, True, False, 32), ("f16", 4737, 260, 128, False, False, 32),
    ("f16", 300, 256, 256, False, True, 1), ("f16", 5000, 256, 256, True, True, 8), ("f16", 20000, 256, 256, False, True, 32),
    ("f16", 2049, 512, 256, True, True, 8), ("f16", 1000, 256, 512, False, True, 8),
]


def _wg_id(c):
    return f"{c[0]}-r{c[1]}-n{c[2]}-k{c[3]}{'-relu' if c[4] else ''}{'-pair' if c[5] else ''}-red{c[6]}"


@pytest.mark.gpu
@pytest.mark.parametrize("case", WGRAD_CASES, ids=_wg_id)
def test_linear_wgrad_integer(case):
    flavour, rows, n_out, k_in, relu, pair, tpo = case
    f16 = flavour == "f16"
    rng = np.random.default_rng(rows * 3 + n_out * 5 + k_in)
    amax = 7 if rows <= 40000 else 1
    g = ints(rng, (rows, n_out), amax=amax, zeros=0.1)
    x = ints(rng, (rows, k_in), amax=amax, zeros=0.1)
    xa = act(x, relu)
    ref_w, ref_b = g.T @ xa, g.sum(0)
    assert_budget(np.abs(g).T @ np.abs(xa), _wg_id(case))
    g_d, _ = placed(g, n_out + 4)           # ld_g > n_out
    x_d, _ = placed(x, k_in + 8)            # ld_x > k_in
    gw, gw_buf, gb, names = run_wgrad(f16, g_d, x_d, n_out, k_in, relu, k_in + 12, True)
    expect_wgrad(names, wg_inst(f16, k_in, pair))
    expect(names, f"wgrad_reduce_kernel<{tpo}>", only="wgrad_reduce_kernel")
    assert_exact(gw, ref_w, _wg_id(case) + " grad_w")
    assert_exact(gb, ref_b, _wg_id(case) + " grad_b")
    assert_gap_intact(gw_buf, k_in, _wg_id(case))


@pytest.mark.gpu
@pytest.mark.parametrize("flavour,side,n_out,k_in,pair", [("tf32", "g", 132, 132, False), ("tf32", "x", 60, 28, False),
                                                          ("f16", "g", 132, 260, False), ("f16", "x", 132, 132, False),
                                                          ("f16", "g", 256, 256, True), ("f16", "x", 256, 256, True)])
def test_linear_wgrad_split_operand(flavour, side, n_out, k_in, pair):
    rng = np.random.default_rng(n_out + k_in + len(side))
    rows = 250
    if side == "g":
        g, x = split12(rng, (rows, n_out)), ints(rng, (rows, k_in), amax=2)
    else:
        g, x = ints(rng, (rows, n_out), amax=2), split12(rng, (rows, k_in))
    assert_budget(np.abs(g).T @ np.abs(x), "split wgrad")
    gw, _, gb, names = run_wgrad(flavour == "f16", dev(g), dev(x), n_out, k_in, False, k_in, True)
    expect_wgrad(names, wg_inst(flavour == "f16", k_in, pair))
    assert_exact(gw, g.T @ x, f"{flavour} split {side} grad_w")
    assert_exact(gb, g.sum(0), f"{flavour} split {side} grad_b")


@pytest.mark.gpu
@pytest.mark.parametrize("flavour", ["tf32", "f16"])
def test_linear_wgrad_zero_rows(flavour):
    """rows = 0: the NaN-filled grad_w (with its padding) and grad_b come back as zeros, padding untouched"""
    for n_out, k_in in ((32, 132), (256, 256)):
        g_d = torch.ones(1, n_out, device="cuda")    # valid pointers (an empty tensor's is NULL), no rows
        x_d = torch.ones(1, k_in, device="cuda")
        gw, gw_buf, gb, names = run_wgrad(flavour == "f16", g_d, x_d, n_out, k_in, False, k_in + 4, True, rows=0)
        expect(names, "wgrad_reduce_kernel<1>", only="wgrad_")
        assert_exact(gw, np.zeros((n_out, k_in)), "grad_w at rows = 0")
        assert_exact(gb, np.zeros(n_out), "grad_b at rows = 0")
        assert_gap_intact(gw_buf, k_in, "grad_w at rows = 0")


@pytest.mark.gpu
@pytest.mark.parametrize("flavour,B,H,W,cin,cout,relu", [
    ("tf32", 1, 6, 16, 32, 4, True), ("tf32", 3, 8, 48, 32, 32, False), ("tf32", 1, 2, 16, 64, 64, True),
    ("tf32", 3, 16, 16, 512, 128, False), ("tf32", 2, 10, 32, 32, 256, True),
    ("f16", 1, 6, 16, 32, 4, True), ("f16", 3, 8, 48, 64, 128, False), ("f16", 1, 16, 16, 512, 256, True),
    ("f16", 2, 10, 32, 32, 132, False)])
def test_conv3x3_wgrad_integer(flavour, B, H, W, cin, cout, relu):
    """conv weight / bias gradient, including H % 8 != 0 (2 x 16 pixel units) and the deepest K = 4608"""
    f16 = flavour == "f16"
    rng = np.random.default_rng(B + H + W + cin + cout)
    x = ints(rng, (B, H, W, cin), zeros=0.1)
    rows = B * H * W
    g = ints(rng, (rows, cout), zeros=0.1)
    cols = im2col(x, relu)
    ref_w, ref_b = g.T @ cols, g.sum(0)
    assert_budget(np.abs(g).T @ np.abs(cols), "conv wgrad")
    g_d, x_d = dev(g), dev(x)
    nb = int(_libh().t2h_conv3x3_wgrad_workspace_bytes(B, H, W, cin, cout))
    ws = nan_workspace(nb)
    gw = torch.full((cout, 9 * cin), float("nan"), device="cuda")
    gb = torch.full((cout,), float("nan"), device="cuda")
    if f16:
        g_slot, x_slot = absmax_slot(g_d), absmax_slot(x_d.view(rows, cin))
        fn = lambda: _call("t2h_conv3x3_wgrad_f16", _p(g_d), _p(g_slot), _p(x_d), _p(x_slot), B, H, W, cin, cout, int(relu),
                           _p(ws), nb, _p(gw), _p(gb))
    else:
        fn = lambda: _call("t2h_conv3x3_wgrad", _p(g_d), _p(x_d), B, H, W, cin, cout, int(relu), _p(ws), nb, _p(gw), _p(gb))
    expect(launched(fn), wg_inst(f16, 9 * cin), only="wgrad_x3_kernel")
    assert_exact(gw, ref_w, "conv grad_w")
    assert_exact(gb, ref_b, "conv grad_b")


# =====================================================================================================
# 6. helpers: column sums, operand maxima
# =====================================================================================================
@pytest.mark.gpu
@pytest.mark.parametrize("n", [4, 32, 33, 64, 65, 128, 129, 256, 260])
def test_colsum_integer(n):
    cw = 32 if n <= 32 else 64 if n <= 64 else 128 if n <= 128 else 256
    rng = np.random.default_rng(n)
    for rows, amax in ((1, 7), (9, 7), (4737, 7), (100003, 7), (10 ** 6, 2)):
        if rows == 10 ** 6 and n not in (4, 33):
            continue
        g = ints(rng, (rows, n), amax=amax, zeros=0.1)
        assert_budget(np.abs(g).sum(0), "colsum")
        g_d, _ = placed(g, n + 3 + (n % 4 == 0))   # ld_g > n, any alignment
        nb = int(_libh().t2h_colsum_workspace_bytes(rows, n))
        ws = nan_workspace(nb)
        out = torch.full((n,), float("nan"), device="cuda")
        names = launched(lambda: _call("t2h_colsum", _p(g_d), g_d.stride(0), rows, n, _p(ws), nb, _p(out)))
        expect(names, f"colsum_partial_kernel<{cw}>", "colsum_final_kernel", only="colsum_")
        assert_exact(out, g.sum(0), f"colsum rows {rows} n {n}")


@pytest.mark.gpu
def test_absmax_and_add_absmax_edges():
    rng = np.random.default_rng(13)
    NAN_PAT = np.array([0x7FC0BEEF], np.uint32).view(np.float32)[0]
    # -0.0 only: the maximum is +0
    z = np.full((100, 8), -0.0, np.float32)
    assert absmax_slot(dev(z)).item() == 0
    for rows, k, ld in ((1, 4, 4), (4097, 96, 132), (300000, 64, 68)):
        x = (rng.standard_normal((rows, k)) * 3).astype(np.float32)
        x[rows // 2, k - 1] = -0.0
        xd, buf = placed(x, ld)
        buf[:, k:] = 1e30                                  # outside the matrix: must be ignored
        assert absmax_slot(xd).item() == absmax_bits_np(x), "absmax strided"
        x[rows - 1, 1] = NAN_PAT                            # a NaN wins over every finite value and infinity
        x[0, 0] = -np.inf
        xd, buf = placed(x, ld)
        assert absmax_slot(xd).item() > 0x7F800000, "absmax NaN: the maximum must be a NaN pattern"
    a1, a2 = rng.standard_normal((777, 32)).astype(np.float32), (rng.standard_normal((777, 36)) * 5).astype(np.float32)
    assert absmax_slot(dev(a1), dev(a2)).item() == absmax_bits_np(a1, a2)
    # add_absmax: out = a + b exactly as fp32, slot = max |out|; a NaN sum wins (its payload is the device's)
    for n in (0, 4, 4096, 1 << 20):
        a = rng.standard_normal(max(n, 4)).astype(np.float32)
        b = rng.standard_normal(max(n, 4)).astype(np.float32)
        a[n // 3] = b[n // 3] = -0.0
        if n >= 4096:
            a[n - 1] = NAN_PAT
        a_d, b_d = dev(a), dev(b)
        out = torch.full((max(n, 4),), float("nan"), device="cuda")
        slot = torch.full((1,), 99, dtype=torch.int32, device="cuda")
        names = launched(lambda: _call("t2h_add_absmax", _p(a_d), _p(b_d), n, _p(out), _p(slot)))
        want = (a[:n] + b[:n]).astype(np.float32)
        got = out[:n].cpu().numpy()
        if n:
            expect(names, "add_absmax_kernel")
        fin = ~np.isnan(want)
        assert np.array_equal(got[fin].view(np.uint32), want[fin].view(np.uint32)) and np.isnan(got[~fin]).all()
        if fin.all():
            assert slot.item() == absmax_bits_np(want), f"add_absmax slot n={n}"
        else:
            assert slot.item() == absmax_bits_np(got) and slot.item() > 0x7F800000, f"add_absmax NaN slot n={n}"


# =====================================================================================================
# 7. autograd level (integer mode): the transposed / mirrored weight splits and their use_f16 decisions
# =====================================================================================================
@pytest.mark.gpu
@pytest.mark.parametrize("use_f16", [False, True])
def test_linear_autograd_integer(use_f16, monkeypatch):
    from tomosar2height_b200 import linear as L
    monkeypatch.setattr(L, "USE_F16", use_f16)
    monkeypatch.setattr(L, "USE_F16_WGRAD", use_f16)
    L._cache.invalidate()
    rng = np.random.default_rng(17)
    rows, k1, k2, n = 1000, 64, 128, 136
    x1n, x2n = ints(rng, (rows, k1), zeros=0.1), ints(rng, (rows, k2), zeros=0.1)
    wn, bn, resn, gyn = ints(rng, (n, k1 + k2)), ints(rng, n), ints(rng, (rows, n)), ints(rng, (rows, n))
    x1, x2, w, b, res = (dev(a).requires_grad_(True) for a in (x1n, x2n, wn, bn, resn))
    gy = dev(gyn)
    got = {}
    names = launched(lambda: got.setdefault("y", L.linear(x1, w, b, x2=x2, relu_in=True, residual=res)).backward(gy))
    xa = np.maximum(np.concatenate([x1n, x2n], 1), 0)
    y = xa @ wn.T + bn + resn
    assert_budget(np.abs(xa) @ np.abs(wn).T + np.abs(bn) + np.abs(resn), "autograd fwd")
    dx = gyn @ wn * (np.concatenate([x1n, x2n], 1) > 0)
    assert_budget(np.abs(gyn) @ np.abs(wn), "autograd dx")
    assert_budget(np.abs(gyn).T @ np.abs(xa), "autograd dw")
    assert_exact(got["y"], y, "y")
    assert_exact(x1.grad, dx[:, :k1], "dx1")
    assert_exact(x2.grad, dx[:, k1:], "dx2")
    assert_exact(w.grad, gyn.T @ xa, "dw")
    assert_exact(b.grad, gyn.sum(0), "db")
    assert_exact(res.grad, gyn, "dres")
    # forward 192 -> 136 (with its residual) and dx2 128 <- 136 (with its ReLU mask) take the fp16 flavour when it
    # is enabled, on CTA pairs with two staging slots; dx1 64 <- 136 never does, and neither does the 64-wide wgrad
    expect(names, FDS if use_f16 else T128, T64, only=LIN)
    if use_f16:
        expect(names, "wgrad_x3_kernel<64,false>", "wgrad_x3_kernel<128,true>", only="wgrad_x3_kernel")
    else:
        expect(names, "wgrad_x3_kernel<64,false>", "wgrad_x3_kernel<128,false>", only="wgrad_x3_kernel")


@pytest.mark.gpu
@pytest.mark.parametrize("use_f16", [False, True])
def test_conv3x3_autograd_integer(use_f16, monkeypatch):
    from tomosar2height_b200 import linear as L
    from tomosar2height_b200.conv import conv3x3
    monkeypatch.setattr(L, "USE_F16", use_f16)
    monkeypatch.setattr(L, "USE_F16_WGRAD", use_f16)
    L._cache.invalidate()
    rng = np.random.default_rng(19)
    B, C, H, W, cout = 2, 64, 8, 32, 96
    xn, wn, bn = ints(rng, (B, C, H, W), zeros=0.1), ints(rng, (cout, C, 3, 3)), ints(rng, cout)
    gyn = ints(rng, (B, cout, H, W))
    x, w, b = (dev(a).requires_grad_(True) for a in (xn, wn, bn))
    y = conv3x3(x, w, b, relu_in=True)
    names = launched(lambda: y.backward(dev(gyn)))
    xd, wd, bd = (torch.from_numpy(a).requires_grad_(True) for a in (xn, wn, bn))
    yd = torch.nn.functional.conv2d(torch.relu(xd), wd, bd, padding=1)
    yd.backward(torch.from_numpy(gyn))
    assert_budget(9 * C * 49 + 7, "conv autograd fwd")
    assert_budget(9 * cout * 49, "conv autograd dx")
    assert_budget(B * H * W * 49, "conv autograd dw")
    assert_exact(y, yd.detach().numpy(), "conv y")
    assert_exact(x.grad, xd.grad.numpy(), "conv dx")
    assert_exact(w.grad, wd.grad.numpy(), "conv dw")
    assert_exact(b.grad, bd.grad.numpy(), "conv db")
    # forward 64 -> 96 on 512 pixels, input gradient 96 -> 64 with the ReLU mask
    expect(launched(lambda: conv3x3(x.detach(), w.detach(), b.detach(), relu_in=True)), FP if use_f16 else T128, only=LIN)
    expect(names, F64 if use_f16 else T64, only=LIN)
    expect(names, "wgrad_x3_kernel<128,true>" if use_f16 else "wgrad_x3_kernel<128,false>", only="wgrad_x3_kernel")


# =====================================================================================================
# 8. more than 2^31 elements
# =====================================================================================================
@pytest.mark.gpu
def test_large_index_rows_times_ld():
    """4.2 M rows x 512 outputs (> 2^31 elements) with a residual in both flavours, and the weight gradient over the
    same rows, checked exactly on a few thousand sampled rows including the last ones.  Operands are integer
    functions of (row, column); the gradient is nonzero on every 1024th row and the last 64, within the budget."""
    free, _ = torch.cuda.mem_get_info()
    if free < 48e9:
        pytest.skip(f"needs ~48 GB of free device memory, {free / 1e9:.1f} GB free")
    rows, K, n = 4_200_000, 128, 512
    assert rows * n > 2 ** 31
    rng = np.random.default_rng(23)
    wn = ints(rng, (n, K))
    bn = ints(rng, n)

    def xf(r, c):
        return (r * 7 + c * 3) % 15 - 7

    def rf(r, c):
        return (r * 5 + c) % 17 - 8

    def fill(fn, m, k):
        t = torch.empty(m, k, dtype=torch.float32, device="cuda")
        cc = torch.arange(k, device="cuda")
        for a in range(0, m, 1 << 18):
            r = torch.arange(a, min(a + (1 << 18), m), device="cuda")
            t[a:a + r.numel()] = fn(r[:, None], cc[None, :]).float()
        return t

    x = fill(xf, rows, K)
    res = fill(rf, rows, n)
    pos = np.unique(np.concatenate([rng.integers(0, rows, 3000), np.arange(rows - 300, rows), np.arange(64)]))
    xs = xf(pos[:, None], np.arange(K)[None, :]).astype(np.float64)
    ref, A = gemm_ref(xs, wn, bn, res=rf(pos[:, None], np.arange(n)[None, :]).astype(np.float64))
    assert_budget(A, "large fwd")
    pos_d = torch.as_tensor(pos).cuda()
    for f16, inst in ((False, T128), (True, FDS)):
        out, _, names, _ = run_linear(f16, x, wn, bn, res=res)
        expect(names, inst, only=LIN)
        assert_exact(out[pos_d], ref, f"{'f16' if f16 else 'tf32'} forward at > 2^31 elements")
        del out
        torch.cuda.empty_cache()
    del res
    keep = torch.arange(rows, device="cuda")
    keep = ((keep % 1024 == 0) | (keep >= rows - 64)).float()[:, None]
    g = fill(rf, rows, n) * keep
    kr = np.flatnonzero((np.arange(rows) % 1024 == 0) | (np.arange(rows) >= rows - 64))
    gk = rf(kr[:, None], np.arange(n)[None, :]).astype(np.float64)
    xk = xf(kr[:, None], np.arange(K)[None, :]).astype(np.float64)
    assert_budget(np.abs(gk).T @ np.abs(xk), "large wgrad")
    for f16, inst in ((False, "wgrad_x3_kernel<128,false>"), (True, "wgrad_x3_kernel<128,true>")):
        gw, _, gb, names = run_wgrad(f16, g, x, n, K, False, K, True)
        expect(names, inst, only="wgrad_x3_kernel")
        assert_exact(gw, gk.T @ xk, "grad_w at > 2^31 elements")
        assert_exact(gb, gk.sum(0), "grad_b at > 2^31 elements")


# =====================================================================================================
# summary
# =====================================================================================================
REQUIRED = sorted({T32, T64, T128, F32, F64, F128, FP, FDS, FW, FWDS,
                   "wgrad_x3_kernel<32,false>", "wgrad_x3_kernel<64,false>", "wgrad_x3_kernel<128,false>",
                   "wgrad_x3_kernel<128,true>", "wgrad_f16_pair_kernel",
                   "wgrad_reduce_kernel<1>", "wgrad_reduce_kernel<8>", "wgrad_reduce_kernel<32>",
                   "colsum_partial_kernel<32>", "colsum_partial_kernel<64>", "colsum_partial_kernel<128>",
                   "colsum_partial_kernel<256>", "colsum_final_kernel",
                   "::absmax_kernel", "add_absmax_kernel", "split_tf32_kernel", "split_f16_kernel"})
# compiled in, reachable only in an -DT2H_ABLATION_ENV build (environment switches of the design study)
EXCLUDED = ("linear_tf32x3_kernel", "linear_x3_persistent_kernel<true,128,2,false,false>",
            "linear_x3_persistent_kernel<true,128,4,false,false>")

_DONE = set()


@pytest.fixture(autouse=True)
def _record_case(request):
    yield
    if "gpu" in request.node.keywords:
        _DONE.add(request.node.nodeid)


@pytest.mark.gpu
def test_zz_every_kernel_instance_was_reached(request):
    """When every GPU case of this file ran and passed, the kernels seen cover every instance the product dispatch
    can pick, and none of the ablation-only instances."""
    cases = {i.nodeid for i in request.session.items if i.fspath == request.node.fspath and "gpu" in i.keywords
             and "test_large_index" not in i.nodeid and "test_zz" not in i.nodeid}
    if not cases <= _DONE or request.session.testsfailed:
        pytest.skip(f"only meaningful when all {len(cases)} path cases ran and passed ({len(cases & _DONE)} ran)")
    seen = sorted(_SEEN)
    reached = lambda k: any(s.endswith(k) for s in seen)
    missing = [k for k in REQUIRED if not reached(k)]
    print("kernel instances reached:\n  " + "\n  ".join(k for k in REQUIRED if reached(k)))
    assert not missing, f"never reached: {missing}"
    unexpected = [k for k in EXCLUDED if any(k in s for s in seen)]
    assert not unexpected, f"ablation-only instances ran: {unexpected}"
