"""GPU parity of the tcgen05 implicit-GEMM kernel (csrc/igemm2.cu) through the C ABI.

Reference = torch fp32 conv / matmul on the SAME fp16-rounded inputs, so the only differences
are accumulation order and the final fp16 rounding of the output: tolerance 2e-3 * max|ref|
(fp16 has 11 significand bits: one rounding is <= 2^-11 = 4.9e-4 relative).
"""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _err(a, b):
    return (a.float() - b.float()).abs().max().item() / (b.float().abs().max().item() + 1e-12)


def _rand(shape, dev, scale=1.0):
    return (torch.randn(shape, device=dev) * scale).to(torch.float16)


@pytest.mark.parametrize("m,k,n", [(128, 64, 64), (1000, 128, 128), (4096, 256, 768), (300, 512, 256), (77, 64, 64)])
def test_plain_gemm_with_bias_and_residual(cuda, m, k, n):
    from cesm_emulator_b200 import kernels as K
    torch.manual_seed(0)
    a = _rand((1, 1, m, k), cuda)
    w = _rand((n, k), cuda, 0.1)
    bias = torch.randn(n, device=cuda)
    res = _rand((1, 1, m, n), cuda)
    out = K.igemm(a, w, bias=bias, residual=res)
    ref = a.float().view(m, k) @ w.float().t() + bias + res.float().view(m, n)
    assert _err(out.view(m, n), ref) < 2e-3


@pytest.mark.parametrize("n,h,w,cin,cout", [(2, 128, 128, 64, 64), (3, 64, 64, 128, 128), (2, 32, 32, 256, 256),
                                             (6, 8, 8, 512, 512), (2, 48, 72, 64, 128), (1, 24, 36, 128, 64),
                                             (2, 192, 288, 64, 64),
                                             # CTA pairs: odd row-tile counts (one ghost tile) and a single tile (no pair)
                                             (3, 8, 14, 64, 64), (1, 8, 14, 128, 128), (5, 16, 30, 64, 256)])
def test_conv3x3(cuda, n, h, w, cin, cout):
    from cesm_emulator_b200 import kernels as K
    torch.manual_seed(1)
    x = _rand((n, h, w, cin), cuda)
    wt = _rand((cout, cin, 3, 3), cuda, 0.05)
    bias = torch.randn(cout, device=cuda)
    wg = wt.permute(0, 2, 3, 1).reshape(cout, 9 * cin).contiguous()
    out = K.igemm(x, wg, taps=K.TAPS_3x3, bias=bias)
    ref = F.conv2d(x.float().permute(0, 3, 1, 2), wt.float(), bias, padding=1).permute(0, 2, 3, 1)
    assert _err(out, ref) < 2e-3


def test_conv3x3_concat(cuda):
    from cesm_emulator_b200 import kernels as K
    torch.manual_seed(2)
    n, h, w, c0, c1, cout = 2, 64, 64, 128, 64, 128
    x0, x1 = _rand((n, h, w, c0), cuda), _rand((n, h, w, c1), cuda)
    wt = _rand((cout, c0 + c1, 3, 3), cuda, 0.05)
    wg = wt.permute(0, 2, 3, 1).reshape(cout, 9 * (c0 + c1)).contiguous()
    out = K.igemm(x0, wg, a1=x1, taps=K.TAPS_3x3)
    xin = torch.cat([x0, x1], -1).float().permute(0, 3, 1, 2)
    ref = F.conv2d(xin, wt.float(), None, padding=1).permute(0, 2, 3, 1)
    assert _err(out, ref) < 2e-3


@pytest.mark.parametrize("n,h,w,c", [(2, 128, 128, 64), (3, 64, 64, 128), (2, 192, 288, 64), (2, 16, 16, 256)])
def test_downsample_conv4x4s2(cuda, n, h, w, c):
    from cesm_emulator_b200 import kernels as K
    torch.manual_seed(3)
    x = _rand((n, h, w, c), cuda)
    wt = _rand((c, c, 4, 4), cuda, 0.05)
    bias = torch.randn(c, device=cuda)
    taps = [(kh - 1, kw - 1) for kh in range(4) for kw in range(4)]
    wg = wt.permute(0, 2, 3, 1).reshape(c, 16 * c).contiguous()
    out = K.igemm(x, wg, taps=taps, stride=2, bias=bias)
    ref = F.conv2d(x.float().permute(0, 3, 1, 2), wt.float(), bias, stride=2, padding=1).permute(0, 2, 3, 1)
    assert out.shape == ref.shape
    assert _err(out, ref) < 2e-3


@pytest.mark.parametrize("n,h,w,c", [(2, 32, 32, 128), (3, 64, 64, 64), (2, 48, 72, 128)])
def test_upsample_convT4x4s2(cuda, n, h, w, c):
    """ConvTranspose2d(4, s2, p1) as four 2x2 phase convolutions scattered into the output."""
    from cesm_emulator_b200 import kernels as K
    torch.manual_seed(4)
    x = _rand((n, h, w, c), cuda)
    wt = _rand((c, c, 4, 4), cuda, 0.05)  # [cin, cout, kh, kw] (ConvTranspose layout)
    bias = torch.randn(c, device=cuda)
    out = torch.empty((n, 2 * h, 2 * w, c), dtype=torch.float16, device=cuda)
    # out[2m+ph] = sum_ih x[ih] * w[kh], kh = 2m+ph+1-2ih  ->  ph=0: (dh=0,kh=1),(dh=-1,kh=3); ph=1: (dh=1,kh=0),(dh=0,kh=2)
    sel = {0: [(0, 1), (-1, 3)], 1: [(1, 0), (0, 2)]}
    for ph in (0, 1):
        for pw in (0, 1):
            taps, wcols = [], []
            for dh, kh in sel[ph]:
                for dw, kw in sel[pw]:
                    taps.append((dh, dw))
                    wcols.append(wt[:, :, kh, kw].t())  # [cout, cin]
            wg = torch.stack(wcols, 1).reshape(c, 4 * c).contiguous()
            K.igemm(x, wg, taps=taps, out=out, out_hw=(h, w), out_place=(2, 2, ph, pw), bias=bias)
    ref = F.conv_transpose2d(x.float().permute(0, 3, 1, 2), wt.float(), bias, stride=2, padding=1).permute(0, 2, 3, 1)
    assert _err(out, ref) < 2e-3


@pytest.mark.parametrize("n,h,w,cin,cout,frames", [(6, 64, 64, 64, 64, 3), (6, 48, 72, 128, 128, 3), (4, 16, 24, 64, 256, 2),
                                                    (2, 192, 288, 64, 64, 1), (6, 8, 8, 128, 128, 3),
                                                    (3, 8, 14, 64, 64, 1), (1, 8, 14, 64, 128, 1), (9, 16, 30, 128, 64, 3)])
def test_conv3x3_fused_groupnorm_stats_and_flipped_taps(cuda, n, h, w, cin, cout, frames):
    """Persistent kernel extras: (a) the per-sample per-group (sum, sum of squares) of the fp16
    outputs from the epilogue equal those of the stored tensor; (b) the data-gradient form
    (negated taps, residual added in the epilogue) matches conv_transpose."""
    from cesm_emulator_b200 import kernels as K
    torch.manual_seed(7)
    G = 8
    x = _rand((n, h, w, cin), cuda)
    wt = _rand((cout, cin, 3, 3), cuda, 0.05)
    bias = torch.randn(cout, device=cuda)
    wg = wt.permute(0, 2, 3, 1).reshape(cout, 9 * cin).contiguous()
    sums = torch.full((n // frames, G, 2), 123.0, device=cuda)
    out = K.igemm(x, wg, taps=K.TAPS_3x3, bias=bias, gn_sums=sums, gn_frames=frames)
    ref = F.conv2d(x.float().permute(0, 3, 1, 2), wt.float(), bias, padding=1).permute(0, 2, 3, 1)
    assert _err(out, ref) < 2e-3
    o = out.float().view(n // frames, frames * h * w, G, cout // G)
    want = torch.stack([o.sum(dim=(1, 3)), (o * o).sum(dim=(1, 3))], dim=-1)
    assert _err(sums, want) < 1e-4
    assert _err(sums, K.gn_stats(out, n // frames, G)) < 1e-4
    # data gradient: dx = conv_transpose(dy, W) + r  ==  conv with negated taps and [ci][t][co] weights
    dy = _rand((n, h, w, cout), cuda)
    r = _rand((n, h, w, cin), cuda)
    wd = wt.permute(1, 2, 3, 0).reshape(cin, 9 * cout).contiguous()
    dx = K.igemm(dy, wd, taps=[(-a, -b) for a, b in K.TAPS_3x3], residual=r)
    ref_dx = F.conv_transpose2d(dy.float().permute(0, 3, 1, 2), wt.float(), padding=1).permute(0, 2, 3, 1) + r.float()
    assert _err(dx, ref_dx) < 2e-3


@pytest.mark.parametrize("m,k,n", [(331776, 64, 768), (82944, 256, 128), (20736, 256, 256), (1000, 1024, 64)])
def test_gemm_large_and_streamed_weights(cuda, m, k, n):
    """Projection shapes of the baseline model at full grid: resident (98 KB) and streamed weights."""
    from cesm_emulator_b200 import kernels as K
    torch.manual_seed(8)
    a = _rand((1, 1, m, k), cuda)
    w = _rand((n, k), cuda, 0.1)
    out = K.igemm(a, w)
    idx = torch.randint(0, m, (4096,), device=cuda)
    ref = a.float().view(m, k)[idx] @ w.float().t()
    assert _err(out.view(m, n)[idx], ref) < 2e-3


@pytest.mark.parametrize("rows,cout", [(128 * 5, 768), (1000, 768), (128 * 300 + 17, 768), (4096, 256)])
def test_fused_qkv_backward(cuda, rows, cout):
    """cesm_qkv_bwd: data gradient + weight gradient of the C=64 -> cout projection in one pass over dy,
    against fp32 matmuls of the same fp16 operands (ragged row counts exercise the TMA zero fill and the
    predicated row stores; two calls accumulate into dW)."""
    from cesm_emulator_b200 import kernels as K
    torch.manual_seed(2)
    dy = (torch.randn(rows, cout, device=cuda) * 0.5).half()
    x = torch.randn(rows, 64, device=cuda).half()
    w = (torch.randn(cout, 64, device=cuda) * 0.1).half()      # to_qkv.weight [cout, cin]
    wt = w.t().contiguous()                                         # data-gradient operand [cin, cout]
    dx, dw = K.qkv_bwd(dy, x, wt)
    dx_ref = dy.float() @ w.float()
    dw_ref = dy.float().t() @ x.float()
    assert (dx.float() - dx_ref).abs().max().item() <= 1e-2 * dx_ref.abs().max().item()
    assert (dw - dw_ref).abs().max().item() <= 2e-4 * dw_ref.abs().max().item()
    base = torch.randn(cout, 64, device=cuda)
    acc = base.clone()
    K.qkv_bwd(dy, x, wt, dw_into=acc)
    K.qkv_bwd(dy, x, wt, dw_into=acc)
    assert (acc - base - 2 * dw_ref).abs().max().item() <= 4e-4 * dw_ref.abs().max().item()
