"""tcgen05 3xTF32 linear layer (t2h_linear_*) vs an fp64 evaluation of the same layer."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _split(w):
    from tomosar2height_b200 import _lib
    hi, lo = torch.empty_like(w), torch.empty_like(w)
    _lib.call("t2h_split_tf32", _lib.ptr(w), w.numel(), _lib.ptr(hi), _lib.ptr(lo))
    return hi, lo


def _linear_raw(x1, w, bias=None, x2=None, relu_in=False, mask=None, residual=None):
    from tomosar2height_b200 import _lib
    rows, k1 = x1.shape
    k2 = 0 if x2 is None else x2.shape[1]
    n_out = w.shape[0]
    hi, lo = _split(w.contiguous())
    out = torch.empty(rows, n_out, device=x1.device, dtype=torch.float32)
    _lib.call("t2h_linear_fwd", _lib.ptr(x1), x1.stride(0), k1, _lib.ptr(x2), 0 if x2 is None else x2.stride(0), k2, rows,
              _lib.ptr(hi), _lib.ptr(lo), n_out, _lib.ptr(bias), int(relu_in), _lib.ptr(mask),
              0 if mask is None else mask.stride(0), _lib.ptr(residual), 0 if residual is None else residual.stride(0),
              _lib.ptr(out), out.stride(0))
    return out


@pytest.mark.parametrize("rows,K,N", [(128, 32, 32), (1000, 64, 32), (4096, 32, 64), (777, 128, 256), (3000, 512, 1024),
                                     (2500, 1024, 512), (130, 96, 48), (5000, 256, 128)])
def test_linear_fwd_matches_fp64(rows, K, N):
    g = torch.Generator().manual_seed(rows + K + N)
    x = torch.randn(rows, K, generator=g).cuda()
    w = (torch.randn(N, K, generator=g) / K ** 0.5).cuda()
    b = torch.randn(N, generator=g).cuda()
    y = _linear_raw(x, w, b)
    ref = x.double() @ w.double().t() + b.double()
    err = (y.double() - ref).abs().max().item() / ref.abs().max().item()
    assert err < 1e-5, err
    # cuBLAS fp32 for comparison: the 3xTF32 result must be as close to fp64 as plain fp32 is (within 4x)
    err32 = ((x @ w.t() + b).double() - ref).abs().max().item() / ref.abs().max().item()
    assert err < 20 * err32 + 1e-6, (err, err32)


def test_linear_epilogues_and_concat():
    g = torch.Generator().manual_seed(0)
    rows = 1500
    a = torch.randn(rows, 32, generator=g).cuda()
    b2 = torch.randn(rows, 32, generator=g).cuda()
    w = (torch.randn(32, 64, generator=g) / 8).cuda()
    bias = torch.randn(32, generator=g).cuda()
    res = torch.randn(rows, 32, generator=g).cuda()
    mask = torch.randn(rows, 32, generator=g).cuda()
    y = _linear_raw(a, w, bias, x2=b2, relu_in=True, mask=mask, residual=res)
    x = torch.cat([a, b2], 1).double().relu()
    ref = (x @ w.double().t() + bias.double()) * (mask > 0).double() + res.double()
    assert (y.double() - ref).abs().max().item() < 2e-6 * ref.abs().max().item()
    # strided views (columns of a wider buffer) as inputs / outputs
    wide = torch.randn(rows, 128, generator=g).cuda()
    y2 = _linear_raw(wide[:, 64:96], w[:, :32].contiguous(), None)
    ref2 = wide[:, 64:96].double() @ w[:, :32].double().t()
    assert (y2.double() - ref2).abs().max().item() < 2e-6 * ref2.abs().max().item()


@pytest.mark.parametrize("rows,K,N", [(128, 32, 32), (1000, 64, 32), (5000, 32, 64), (3000, 128, 256), (2000, 512, 1024),
                                     (4100, 1024, 512), (130, 96, 48), (9000, 256, 128), (40, 64, 64), (33, 256, 256),
                                     (70000, 512, 256), (129, 256, 512)])
@pytest.mark.parametrize("relu_in", [False, True])
@pytest.mark.parametrize("flavour", ["f16", "tf32"])
def test_linear_autograd_matches_fp64(rows, K, N, relu_in, flavour, monkeypatch):
    from tomosar2height_b200.linear import linear
    from tomosar2height_b200 import linear as L
    monkeypatch.setattr(L, "USE_F16", flavour == "f16")        # wide layers: 3xFP16 (default) or 3xTF32 everywhere
    monkeypatch.setattr(L, "USE_F16_WGRAD", flavour == "f16")
    g = torch.Generator().manual_seed(rows * 7 + K + N)
    x = torch.randn(rows, K, generator=g).cuda().requires_grad_(True)
    w = (torch.randn(N, K, generator=g) / K ** 0.5).cuda().requires_grad_(True)
    b = torch.randn(N, generator=g).cuda().requires_grad_(True)
    res = torch.randn(rows, N, generator=g).cuda().requires_grad_(True)
    gy = torch.randn(rows, N, generator=g).cuda()
    y = linear(x, w, b, relu_in=relu_in, residual=res)
    y.backward(gy)
    xd, wd, bd, rd = (t.detach().double().requires_grad_(True) for t in (x, w, b, res))
    yd = (xd.relu() if relu_in else xd) @ wd.t() + bd + rd
    yd.backward(gy.double())

    def rel(a, ref):
        return (a.double() - ref).abs().max().item() / ref.abs().max().item()

    # tensor-core fp32 accumulation rounds once per MMA k-step: allow a slow growth with depth
    tol = 1e-5 * max(1.0, max(K, N) / 256)
    assert rel(y, yd) < tol, rel(y, yd)
    assert rel(x.grad, xd.grad) < tol, rel(x.grad, xd.grad)
    assert rel(w.grad, wd.grad) < tol, rel(w.grad, wd.grad)
    assert rel(b.grad, bd.grad) < 1e-5
    assert torch.equal(res.grad, gy)


def test_linear_concat_autograd():
    from tomosar2height_b200.linear import linear
    g = torch.Generator().manual_seed(5)
    rows = 2345
    a = torch.randn(rows, 32, generator=g).cuda().requires_grad_(True)
    b2 = torch.randn(rows, 32, generator=g).cuda().requires_grad_(True)
    w = (torch.randn(32, 64, generator=g) / 8).cuda().requires_grad_(True)
    gy = torch.randn(rows, 32, generator=g).cuda()
    y = linear(a, w, None, x2=b2, relu_in=True)
    y.backward(gy)
    ad, bd, wd = (t.detach().double().requires_grad_(True) for t in (a, b2, w))
    yd = torch.cat([ad, bd], 1).relu() @ wd.t()
    yd.backward(gy.double())
    for got, ref in ((y, yd), (a.grad, ad.grad), (b2.grad, bd.grad), (w.grad, wd.grad)):
        assert (got.double() - ref).abs().max().item() < 1e-5 * ref.abs().max().item()


def test_weight_split_cache_tracks_updates():
    from tomosar2height_b200.linear import linear
    w = torch.randn(32, 32).cuda().requires_grad_(True)
    x = torch.randn(256, 32).cuda()
    y0 = linear(x, w)
    with torch.no_grad():
        w.mul_(2.0)  # optimizer-style in-place update bumps the version counter
    y1 = linear(x, w)
    assert (y1 - 2 * y0).abs().max().item() < 1e-5 * y0.abs().max().item()


def test_linear_odd_widths_are_padded():
    """1-wide output head (pixel.py:51) and a K that is not a multiple of 4 still run on the tensor cores."""
    from tomosar2height_b200.linear import linear
    from tomosar2height_b200 import _lib
    g = torch.Generator().manual_seed(11)
    x = torch.randn(2, 50, 50, 30, generator=g).cuda().requires_grad_(True)
    w = (torch.randn(1, 30, generator=g) / 5).cuda().requires_grad_(True)
    b = torch.randn(1, generator=g).cuda().requires_grad_(True)
    before = _lib.launch_count
    y = linear(x, w, b, relu_in=True)
    assert y.shape == (2, 50, 50, 1) and _lib.launch_count > before
    y.square().sum().backward()
    xd, wd, bd = (t.detach().double().requires_grad_(True) for t in (x, w, b))
    yd = xd.relu() @ wd.t() + bd
    yd.square().sum().backward()
    for got, ref in ((y, yd), (x.grad, xd.grad), (w.grad, wd.grad), (b.grad, bd.grad)):
        assert (got.double() - ref).abs().max().item() < 1e-5 * ref.abs().max().item()


# ---- 3xFP16 flavour (t2h_absmax / t2h_split_f16 / t2h_linear_fwd_f16) ------------------------------------
def _absmax_raw(x1, x2=None):
    from tomosar2height_b200 import _lib
    slot = torch.full((1,), 12345, dtype=torch.int32, device=x1.device)  # the call must reset it
    _lib.call("t2h_absmax", _lib.ptr(x1), x1.stride(0), x1.shape[1], _lib.ptr(x2), 0 if x2 is None else x2.stride(0),
              0 if x2 is None else x2.shape[1], x1.shape[0], _lib.ptr(slot))
    return slot


def _linear_f16_raw(x1, w, bias=None, x2=None, relu_in=False, mask=None, residual=None, want_out_max=True):
    from tomosar2height_b200 import _lib
    rows, k1 = x1.shape
    k2 = 0 if x2 is None else x2.shape[1]
    n_out = w.shape[0]
    w = w.contiguous()
    w_slot = _absmax_raw(w)
    hi = torch.empty(w.shape, dtype=torch.float16, device=w.device)
    lo = torch.empty_like(hi)
    _lib.call("t2h_split_f16", _lib.ptr(w), w.numel(), _lib.ptr(w_slot), _lib.ptr(hi), _lib.ptr(lo))
    x_slot = _absmax_raw(x1, x2)
    out = torch.empty(rows, n_out, device=x1.device, dtype=torch.float32)
    out_slot = torch.full((1,), 777, dtype=torch.int32, device=x1.device) if want_out_max else None
    _lib.call("t2h_linear_fwd_f16", _lib.ptr(x1), x1.stride(0), k1, _lib.ptr(x2), 0 if x2 is None else x2.stride(0), k2, rows,
              _lib.ptr(x_slot), _lib.ptr(hi), _lib.ptr(lo), _lib.ptr(w_slot), n_out, _lib.ptr(bias), int(relu_in),
              _lib.ptr(mask), 0 if mask is None else mask.stride(0), _lib.ptr(residual),
              0 if residual is None else residual.stride(0), _lib.ptr(out), out.stride(0), _lib.ptr(out_slot))
    return out, out_slot


def test_absmax_is_exact_and_handles_strides():
    g = torch.Generator().manual_seed(5)
    for rows, k, ld in [(1, 4, 4), (1000, 32, 32), (4097, 96, 128), (300000, 64, 64)]:
        buf = (torch.randn(rows, ld, generator=g) * 3).cuda()
        buf[:, k:] = 1e6  # outside the matrix: must be ignored
        x = buf[:, :k]
        slot = _absmax_raw(x)
        assert slot.view(torch.float32).item() == x.abs().max().item()
    a, b = torch.randn(777, 32, generator=g).cuda(), (torch.randn(777, 64, generator=g) * 5).cuda()
    assert _absmax_raw(a, b).view(torch.float32).item() == max(a.abs().max().item(), b.abs().max().item())
    assert _absmax_raw(torch.zeros(64, 8).cuda()).item() == 0


@pytest.mark.parametrize("rows,K,N", [(777, 128, 256), (3000, 512, 1024), (2500, 1024, 512), (5000, 256, 128),
                                     (130, 160, 132), (100000, 256, 512)])
def test_linear_f16_matches_fp64(rows, K, N):
    g = torch.Generator().manual_seed(rows + K + N)
    x = torch.randn(rows, K, generator=g).cuda()
    w = (torch.randn(N, K, generator=g) / K ** 0.5).cuda()
    b = torch.randn(N, generator=g).cuda()
    y, out_slot = _linear_f16_raw(x, w, b)
    ref = x.double() @ w.double().t() + b.double()
    err = (y.double() - ref).abs().max().item() / ref.abs().max().item()
    err32 = ((x @ w.t() + b).double() - ref).abs().max().item() / ref.abs().max().item()
    assert err < 1e-5 and err < 20 * err32 + 1e-6, (err, err32)
    # the epilogue publishes max |out| exactly (the operand scale of a following layer)
    assert out_slot.view(torch.float32).item() == y.abs().max().item()


@pytest.mark.parametrize("scale", [1e-12, 1e-4, 1.0, 1e6, 1e20])
def test_linear_f16_operand_scaling(scale):
    """power-of-two operand scaling: the relative accuracy does not depend on the magnitude of the operands
    (gradients are ~1e-9, fp16 underflows below 6e-8 and overflows above 65504)."""
    g = torch.Generator().manual_seed(11)
    x = (torch.randn(2000, 256, generator=g) * scale).cuda()
    w = (torch.randn(128, 256, generator=g) * (0.05 / scale ** 0.5)).cuda()
    y, _ = _linear_f16_raw(x, w)
    ref = x.double() @ w.double().t()
    assert torch.isfinite(y).all()
    assert (y.double() - ref).abs().max().item() < 2e-6 * ref.abs().max().item()


def test_linear_f16_rows_of_very_different_magnitude():
    """rows spanning six orders of magnitude share one tensor scale: small rows keep ~1e-5 of THEIR OWN scale
    (absolute floor 2^-39 of the tensor maximum, documented in include/t2h.h)."""
    g = torch.Generator().manual_seed(12)
    x = torch.randn(4096, 256, generator=g) * torch.exp(torch.empty(4096, 1).uniform_(-12, 3, generator=g))
    w = torch.randn(256, 256, generator=g) / 16
    y, _ = _linear_f16_raw(x.cuda(), w.cuda())
    ref = x.double() @ w.double().t()
    row_scale = ref.abs().amax(1, keepdim=True)
    assert ((y.cpu().double() - ref).abs() / row_scale).max().item() < 1e-4


@pytest.mark.parametrize("n_out", [200, 256, 512])  # 128-wide tiles (ragged last tile) / 256 x 256 pair tiles
def test_linear_f16_epilogues_concat_and_ragged_k(n_out):
    g = torch.Generator().manual_seed(1)
    rows = 1500
    a = torch.randn(rows, 96, generator=g).cuda()    # 3 chunks + 2 chunks = odd number of 32-wide chunks
    b2 = torch.randn(rows, 64, generator=g).cuda()
    w = (torch.randn(n_out, 160, generator=g) / 12).cuda()
    bias = torch.randn(n_out, generator=g).cuda()
    res = torch.randn(rows, n_out, generator=g).cuda()
    mask = torch.randn(rows, n_out, generator=g).cuda()
    x = torch.cat([a, b2], 1).double().relu()
    full = x @ w.double().t() + bias.double()
    y, slot = _linear_f16_raw(a, w, bias, x2=b2, relu_in=True, mask=mask)
    ref = full * (mask > 0).double()
    assert (y.double() - ref).abs().max().item() < 2e-6 * full.abs().max().item()
    assert slot.view(torch.float32).item() == y.abs().max().item()
    y, slot = _linear_f16_raw(a, w, bias, x2=b2, relu_in=True, residual=res)
    ref = full + res.double()
    assert (y.double() - ref).abs().max().item() < 2e-6 * ref.abs().max().item()
    assert slot.view(torch.float32).item() == y.abs().max().item()
    y, _ = _linear_f16_raw(a, w, bias, x2=b2, relu_in=True, mask=mask, residual=res, want_out_max=False)  # general epilogue
    ref = full * (mask > 0).double() + res.double()
    assert (y.double() - ref).abs().max().item() < 2e-6 * ref.abs().max().item()
    # K = 136 (multiple of 8, not of 32): the last chunk is zero-filled by TMA
    xs = torch.randn(rows, 136, generator=g).cuda()
    ws = (torch.randn(96 if n_out == 200 else n_out, 136, generator=g) / 11).cuda()
    y, _ = _linear_f16_raw(xs, ws)
    ref = xs.double() @ ws.double().t()
    assert (y.double() - ref).abs().max().item() < 2e-6 * ref.abs().max().item()


def test_absmax_registry_is_reused_and_never_stale():
    from tomosar2height_b200 import linear as L
    from tomosar2height_b200 import _lib
    g = torch.Generator().manual_seed(2)
    x = torch.randn(3000, 256, generator=g).cuda()
    w1 = torch.nn.Parameter((torch.randn(256, 256, generator=g) / 16).cuda())
    w2 = torch.nn.Parameter((torch.randn(128, 256, generator=g) / 16).cuda())
    assert L.use_f16(256, 256)
    h = L.linear(x, w1)
    slot = L._absmax.get(h.detach())
    assert slot is not None and slot.view(torch.float32).item() == h.abs().max().item()
    L.linear(h, w2, relu_in=True)                # fills the weight-split cache of w2
    before = _lib.launch_count
    y = L.linear(h, w2, relu_in=True)            # uses the published maximum: one launch (the GEMM), no absmax pass
    assert _lib.launch_count - before == 1
    ref = h.double().relu() @ w2.double().t()
    assert (y.double() - ref).abs().max().item() < 2e-6 * ref.abs().max().item()
    with torch.no_grad():
        h.mul_(1000.0)                            # modified in place: the registered maximum must not be used
    assert L._absmax.get(h) is None
    y = L.linear(h, w2, relu_in=True)
    ref = h.double().relu() @ w2.double().t()
    assert torch.isfinite(y).all() and (y.double() - ref).abs().max().item() < 2e-6 * ref.abs().max().item()


def test_fork2_sums_gradient_branches_and_publishes_their_maximum():
    from tomosar2height_b200 import linear as L
    g = torch.Generator().manual_seed(4)
    x = torch.randn(5000, 256, generator=g).cuda().requires_grad_(True)
    w = torch.nn.Parameter((torch.randn(128, 256, generator=g) / 16).cuda())
    h = L.linear(x, torch.nn.Parameter((torch.randn(256, 256, generator=g) / 16).cuda()))
    a, b = L.fork2(h)
    seen = {}
    h.register_hook(lambda gr: seen.setdefault("g", gr))
    (L.linear(a, w).square().sum() + (b * 3.0).sum()).backward()
    gr = seen["g"]
    ref = (2 * (h.detach().double() @ w.double().t()) @ w.double()) + 3.0
    assert (gr.double() - ref).abs().max().item() < 1e-5 * ref.abs().max().item()
    slot = L._absmax.get(gr)
    assert slot is not None and slot.view(torch.float32).item() == gr.abs().max().item()
    # without autograd the fork is the identity
    with torch.no_grad():
        p, q = L.fork2(h)
    assert p is h and q is h


@pytest.mark.parametrize("rows,K,N", [(70000, 512, 256), (40000, 1024, 512), (50000, 256, 512), (300, 288, 256)])
def test_linear_f16_wide_tiles_with_mask_and_residual(rows, K, N):
    """256 x 256 pair tiles: four output blocks per epilogue group and tile, mask / residual blocks through one
    (K >= 512) or two (K <= 256) staging slots per group, many tiles per CTA pair."""
    g = torch.Generator().manual_seed(rows + K)
    x = torch.randn(rows, K, generator=g).cuda()
    w = (torch.randn(N, K, generator=g) / K ** 0.5).cuda()
    bias = torch.randn(N, generator=g).cuda()
    aux = torch.randn(rows, N, generator=g).cuda()
    full = x.double() @ w.double().t() + bias.double()
    tol = 2e-6 * max(1.0, K / 256)
    y, _ = _linear_f16_raw(x, w, bias, mask=aux)
    assert (y.double() - full * (aux > 0).double()).abs().max().item() < tol * full.abs().max().item()
    y, slot = _linear_f16_raw(x, w, bias, residual=aux)
    ref = full + aux.double()
    assert (y.double() - ref).abs().max().item() < tol * ref.abs().max().item()
    assert slot.view(torch.float32).item() == y.abs().max().item()
    y, _ = _linear_f16_raw(x, w, bias, relu_in=True)
    ref = x.double().relu() @ w.double().t() + bias.double()
    assert (y.double() - ref).abs().max().item() < tol * ref.abs().max().item()
