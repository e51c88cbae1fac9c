"""GPU parity of every non-GEMM kernel and of the tcgen05 weight-gradient kernel, through the C ABI.

Each check feeds the CUDA kernel and a torch fp32 restatement (oracle functions where they exist)
the SAME fp16-rounded inputs.  Tolerances (relative to max|ref|): 2e-3 for fp16 outputs (one or two fp16
roundings of 2^-12 each plus fp32 reassociation) unless a test states otherwise, 2e-3 for fp32 outputs.
"""
import math

import pytest
import torch
import torch.nn.functional as F

from oracle import cesm_oracle as O

pytestmark = pytest.mark.gpu
BF = torch.float16


def err(a, b):
    a, b = a.float(), b.float()
    return (a - b).abs().max().item() / (b.abs().max().item() + 1e-20)


def rnd(shape, dev, scale=1.0, dtype=BF):
    return (torch.randn(shape, device=dev) * scale).to(dtype)


# ------------------------------------------------------------------------------------------------
# weight gradients (tcgen05, MN-major operands)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,h,w,cin,cout", [(2, 32, 32, 64, 64), (3, 64, 64, 128, 128), (2, 16, 16, 256, 256),
                                             (6, 8, 8, 512, 512), (2, 48, 72, 64, 128), (1, 24, 36, 128, 64),
                                             (2, 128, 128, 64, 64)])
def test_wgrad_conv3x3(cuda, n, h, w, cin, cout):
    from cesm_emulator_b200 import kernels as K
    torch.manual_seed(0)
    x, dy = rnd((n, h, w, cin), cuda), rnd((n, h, w, cout), cuda, 0.1)
    dw = K.wgrad(x, dy, taps=K.TAPS_3x3)  # [cout, 9, cin]
    wt = torch.zeros(cout, cin, 3, 3, device=cuda, requires_grad=True)
    y = F.conv2d(x.float().permute(0, 3, 1, 2), wt, padding=1)
    (ref,) = torch.autograd.grad(y, wt, dy.float().permute(0, 3, 1, 2))
    assert err(dw.view(cout, 3, 3, cin).permute(0, 3, 1, 2), ref) < 2e-3


def test_wgrad_concat_and_1x1(cuda):
    from cesm_emulator_b200 import kernels as K
    torch.manual_seed(1)
    n, h, w, c0, c1, cout = 2, 32, 32, 128, 64, 128
    x0, x1, dy = rnd((n, h, w, c0), cuda), rnd((n, h, w, c1), cuda), rnd((n, h, w, cout), cuda, 0.1)
    dw = K.wgrad(x0, dy, x1=x1, taps=K.TAPS_3x3)
    wt = torch.zeros(cout, c0 + c1, 3, 3, device=cuda, requires_grad=True)
    y = F.conv2d(torch.cat([x0, x1], -1).float().permute(0, 3, 1, 2), wt, padding=1)
    (ref,) = torch.autograd.grad(y, wt, dy.float().permute(0, 3, 1, 2))
    assert err(dw.view(cout, 3, 3, c0 + c1).permute(0, 3, 1, 2), ref) < 2e-3
    # plain linear: dW = dy^T x
    m, k, nn = 5000, 256, 768
    a, g = rnd((1, 1, m, k), cuda), rnd((1, 1, m, nn), cuda, 0.1)
    dwl = K.wgrad(a, g)
    assert err(dwl.view(nn, k), g.float().view(m, nn).t() @ a.float().view(m, k)) < 2e-3


def test_wgrad_strided_and_transposed(cuda):
    from cesm_emulator_b200 import kernels as K
    torch.manual_seed(2)
    n, h, w, c = 2, 32, 32, 128
    # Downsample conv 4x4 s2 p1
    x, dy = rnd((n, h, w, c), cuda), rnd((n, h // 2, w // 2, c), cuda, 0.1)
    taps = [(kh - 1, kw - 1) for kh in range(4) for kw in range(4)]
    dw = K.wgrad(x, dy, taps=taps, stride=2)
    wt = torch.zeros(c, c, 4, 4, device=cuda, requires_grad=True)
    y = F.conv2d(x.float().permute(0, 3, 1, 2), wt, stride=2, padding=1)
    (ref,) = torch.autograd.grad(y, wt, dy.float().permute(0, 3, 1, 2))
    assert err(dw.view(c, 4, 4, c).permute(0, 3, 1, 2), ref) < 2e-3
    # Upsample ConvTranspose 4x4 s2 p1: weight [cin, cout, kh, kw]
    x, dy = rnd((n, h, w, c), cuda), rnd((n, 2 * h, 2 * w, c), cuda, 0.1)
    wt = torch.zeros(c, c, 4, 4, device=cuda, requires_grad=True)
    y = F.conv_transpose2d(x.float().permute(0, 3, 1, 2), wt, stride=2, padding=1)
    (ref,) = torch.autograd.grad(y, wt, dy.float().permute(0, 3, 1, 2))
    got = torch.zeros_like(ref)
    sel = {0: [(0, 1), (-1, 3)], 1: [(1, 0), (0, 2)]}
    for ph in (0, 1):
        for pw in (0, 1):
            taps, khw = [], []
            for dh, kh in sel[ph]:
                for dw_, kw in sel[pw]:
                    taps.append((dh, dw_))
                    khw.append((kh, kw))
            d = K.wgrad(x, dy, taps=taps, grid_hw=(h, w), dy_place=(2, 2, ph, pw))  # [cout, 4, cin]
            for t, (kh, kw) in enumerate(khw):
                got[:, :, kh, kw] = d[:, t, :].t()
    assert err(got, ref) < 2e-3


def test_pack_unpack_weight(cuda):
    from cesm_emulator_b200 import kernels as K
    torch.manual_seed(3)
    co, ci = 128, 64
    w = torch.randn(co, ci, 1, 3, 3, device=cuda)
    offs = [kh * 3 + kw for kh in range(3) for kw in range(3)]
    p = K.pack_weight(w, co, 9, ci, ci * 9, 9, offs)
    assert torch.equal(p.view(co, 9, ci), w.view(co, ci, 9).permute(0, 2, 1).to(BF))
    # dgrad layout: [ci][flipped tap][co]
    pd = K.pack_weight(w, ci, 9, co, 9, ci * 9, [8 - o for o in offs])
    assert torch.equal(pd.view(ci, 9, co), w.view(co, ci, 9).flip(-1).permute(1, 2, 0).to(BF))
    g = torch.randn(co, 9, ci, device=cuda)
    dst = torch.zeros_like(w)
    K.unpack_wgrad(g, dst, co, 9, ci, ci * 9, 9, offs)
    assert torch.equal(dst.view(co, ci, 9), g.permute(0, 2, 1))
    K.unpack_wgrad(g, dst, co, 9, ci, ci * 9, 9, offs, accumulate=True)
    assert torch.equal(dst.view(co, ci, 9), 2 * g.permute(0, 2, 1))
    x = rnd((777, 256), cuda)
    assert err(K.colsum(x), x.float().sum(0)) < 1e-4


# ------------------------------------------------------------------------------------------------
# GroupNorm + FiLM + SiLU (+ residual) and channel LayerNorm
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,P,C,film,res", [(2, 3 * 16 * 16, 64, True, False), (2, 3 * 8 * 8, 128, False, True),
                                            (1, 1000, 256, True, True), (3, 65, 512, False, False)])
def test_groupnorm_fwd_bwd(cuda, B, P, C, film, res):
    from cesm_emulator_b200 import kernels as K
    torch.manual_seed(4)
    G = 8
    x = rnd((B, P, C), cuda, 2.0) + 0.5
    gamma = torch.randn(C, device=cuda) * 0.5 + 1
    beta = torch.randn(C, device=cuda) * 0.2
    fl = torch.randn(B, 2 * C, device=cuda) * 0.3 if film else None
    r = rnd((B, P, C), cuda) if res else None
    dout = rnd((B, P, C), cuda)
    sums = K.gn_stats(x, B, G)
    out = K.gn_apply_fwd(x, sums, gamma, beta, fl, r, B, G, 1e-5)
    dx, dg, db, dfl, dcb = K.gn_bwd(x, dout, sums, gamma, beta, fl, B, G, 1e-5, conv_bias_grad=True)

    xr = x.float().requires_grad_(True)
    gr, br = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
    flr = fl.clone().requires_grad_(True) if film else None
    y = F.group_norm(xr.transpose(1, 2), G, gr, br, 1e-5)  # [B, C, P]
    if film:
        y = y * (flr[:, :C, None] + 1) + flr[:, C:, None]
    y = F.silu(y).transpose(1, 2)
    ref = y + (r.float() if res else 0)
    assert err(out, ref) < 2e-3
    grads = torch.autograd.grad(y, [xr, gr, br] + ([flr] if film else []), dout.float())
    assert err(dx, grads[0]) < 2e-3
    assert err(dg, grads[1]) < 2e-3 and err(db, grads[2]) < 2e-3
    if film:
        assert err(dfl, grads[3]) < 2e-3
    # bias gradient of the producing conv = sum over samples and pixels of dx (here of the exact dx)
    assert err(dcb, grads[0].sum(dim=(0, 1))) < 2e-3
    # accumulate mode (the engine hands in the parameters' .grad views): the apply kernel adds the
    # parameter gradients itself, on top of what is already there
    base = [torch.randn(C, device=cuda) for _ in range(3)]
    into = [t.clone() for t in base]
    dx2, _, _, dfl2, _ = K.gn_bwd(x, dout, sums, gamma, beta, fl, B, G, 1e-5, conv_bias_grad=True, into=tuple(into))
    assert err(dx2, dx) < 2e-3  # the per-channel sums are fp32 atomics: run-to-run rounding differs
    for got, b0, want in zip(into, base, (dg, db, dcb)):
        assert err(got - b0, want) < 1e-4
    if film:
        assert err(dfl2, dfl) < 1e-4


@pytest.mark.parametrize("M,C", [(1000, 64), (513, 128), (300, 256), (77, 512)])
def test_layernorm_fwd_bwd(cuda, M, C):
    from cesm_emulator_b200 import kernels as K
    torch.manual_seed(5)
    x = rnd((M, C), cuda, 2.0) + 0.3
    gamma = torch.randn(C, device=cuda) * 0.5 + 1
    dy, dres = rnd((M, C), cuda), rnd((M, C), cuda)
    out = K.ln_fwd(x, gamma, 1e-5)
    dx, dg = K.ln_bwd(x, gamma, dy, dres, 1e-5)
    xr, gr = x.float().requires_grad_(True), gamma.clone().requires_grad_(True)
    y = O.channel_layer_norm(xr.t()[None], gr[None, :, None])[0].t()
    assert err(out, y) < 2e-3
    gx, gg = torch.autograd.grad(y, [xr, gr], dy.float())
    assert err(dx, gx + dres.float()) < 2e-3
    assert err(dg, gg) < 2e-3
    dx2, _ = K.ln_bwd(x, gamma, dy, None, 1e-5)
    assert err(dx2, gx) < 2e-3


# ------------------------------------------------------------------------------------------------
# attention cores
# ------------------------------------------------------------------------------------------------
def _tattn_ref(qkv, bias, freqs, B, Fr, HW, H, D):
    """oracle.attention without the projections: qkv [B*F*HW, 3HD] -> out [B*F*HW, HD]."""
    x = qkv.view(B, Fr, HW, 3 * H * D).permute(0, 2, 1, 3)  # b hw f c
    q, k, v = (t.reshape(B, HW, Fr, H, D).transpose(-2, -3) for t in x.chunk(3, dim=-1))
    q = q * D ** -0.5
    ang = O.rotary_angles(freqs, Fr)
    q, k = O.apply_rotary(q, ang), O.apply_rotary(k, ang)
    sim = torch.einsum("...hid,...hjd->...hij", q, k) + bias
    attn = (sim - sim.amax(-1, keepdim=True).detach()).softmax(-1)
    out = torch.einsum("...hij,...hjd->...hid", attn, v)
    out = out.transpose(-2, -3).reshape(B, HW, Fr, H * D)
    return out.permute(0, 2, 1, 3).reshape(B * Fr * HW, H * D)


def _toeplitz_bias(H, Fr, dev):
    """A bias of RelativePositionBias's structure (video_net.py:302-310): a function of key - query per head."""
    diag = torch.randn(H, 2 * Fr - 1, device=dev)
    i = torch.arange(Fr, device=dev)
    return diag[:, (i[None, :] - i[:, None]) + Fr - 1].contiguous(), diag


def _fold_diagonals(g, Fr):
    """[H, F, F] -> [H, 2F-1]: sums over entries with the same key - query."""
    i = torch.arange(Fr, device=g.device)
    idx = ((i[None, :] - i[:, None]) + Fr - 1).reshape(-1)
    return torch.zeros(g.shape[0], 2 * Fr - 1, device=g.device, dtype=g.dtype).index_add_(1, idx, g.reshape(g.shape[0], -1))


@pytest.mark.parametrize("B,Fr,HW,H", [(2, 3, 64, 8), (1, 1, 100, 8), (2, 12, 33, 8), (1, 40, 16, 4), (1, 16, 64, 8),
                                       (1, 32, 40, 8), (2, 64, 24, 8), (1, 128, 6, 8), (1, 100, 5, 2), (1, 5, 300, 8)])
def test_temporal_attention_core(cuda, B, Fr, HW, H):
    """F <= 4: the register-resident kernels with an arbitrary [H, F, F] bias.  F > 4: the shared-memory / mma.sync
    flash kernels (csrc/tattn_long.cu), which take the relative-position bias by diagonal -- Toeplitz bias, and its
    gradient compared per diagonal (the only form any consumer uses: buckets depend on key - query)."""
    from cesm_emulator_b200 import kernels as K
    torch.manual_seed(6)
    D = 32
    qkv = rnd((B * Fr * HW, 3 * H * D), cuda)
    bias = torch.randn(H, Fr, Fr, device=cuda) if Fr <= 4 else _toeplitz_bias(H, Fr, cuda)[0]
    freqs = (1.0 / (10000 ** (torch.arange(0, D, 2).float() / D))).to(cuda)
    ang = torch.arange(Fr, device=cuda, dtype=torch.float32)[:, None] * freqs[None]
    cs, sn = ang.cos().contiguous(), ang.sin().contiguous()
    dout = rnd((B * Fr * HW, H * D), cuda)
    out, lse = K.tattn_fwd(qkv, bias, cs, sn, B, Fr, HW, H, D, D ** -0.5)
    dqkv, dbias = K.tattn_bwd(qkv, bias, cs, sn, out, lse, dout, B, Fr, HW, H, D, D ** -0.5)
    qr, br = qkv.float().requires_grad_(True), bias.clone().requires_grad_(True)
    ref = _tattn_ref(qr, br, freqs, B, Fr, HW, H, D)
    assert err(out, ref) < 2e-3
    gq, gb = torch.autograd.grad(ref, [qr, br], dout.float())
    assert err(dqkv, gq) < 3e-3
    if Fr <= 4:
        assert err(dbias, gb) < 2e-3
    else:
        assert err(_fold_diagonals(dbias, Fr), _fold_diagonals(gb, Fr)) < 3e-3
        lse_ref = torch.logsumexp(_tattn_scores(qr.detach(), bias, freqs, B, Fr, HW, H, D), dim=-1)  # [B, HW, H, F]
        assert err(lse.view(B, Fr, HW, H).permute(0, 2, 3, 1), lse_ref) < 2e-3


@pytest.mark.parametrize("B,Fr,HW", [(2, 3, 64), (1, 3, 48 * 72), (1, 2, 160), (3, 1, 32), (2, 3, 16)])
def test_temporal_attention_fused_with_projection_forward(cuda, B, Fr, HW):
    """csrc/tattn_proj.cu: o = attention(xn Wq^T, xn Wk^T, xn Wv^T) without materialising q|k|v (the no-grad
    forward), against the fp32 torch restatement of projection + attention on the same fp16-rounded xn / W
    (video_net.py:403-453)."""
    from cesm_emulator_b200 import kernels as K
    torch.manual_seed(7)
    H, D, C = 8, 32, 64
    rows = B * Fr * HW
    xn = rnd((rows, C), cuda)
    w = rnd((3 * H * D, C), cuda, 0.15)
    bias = torch.randn(H, Fr, Fr, device=cuda)
    freqs = (1.0 / (10000 ** (torch.arange(0, D, 2).float() / D))).to(cuda)
    ang = torch.arange(Fr, device=cuda, dtype=torch.float32)[:, None] * freqs[None]
    cs, sn = ang.cos().contiguous(), ang.sin().contiguous()
    out = K.tattn_proj_fwd(xn, w, bias, cs, sn, B, Fr, HW, H, D, D ** -0.5)
    ref = _tattn_ref(xn.float() @ w.float().t(), bias, freqs, B, Fr, HW, H, D)
    assert err(out, ref) < 2e-3
    # and the unfused kernels on the materialised projection agree (same arithmetic, q|k|v rounded to fp16 in between)
    qkv = K.igemm(xn.view(1, 1, rows, C), w).view(rows, 3 * H * D)
    out2, _ = K.tattn_fwd(qkv, bias, cs, sn, B, Fr, HW, H, D, D ** -0.5)
    assert err(out, out2) < 3e-3


def _tattn_scores(qkv, bias, freqs, B, Fr, HW, H, D):
    x = qkv.view(B, Fr, HW, 3 * H * D).permute(0, 2, 1, 3)
    q, k, _ = (t.reshape(B, HW, Fr, H, D).transpose(-2, -3) for t in x.chunk(3, dim=-1))
    ang = O.rotary_angles(freqs, Fr)
    q, k = O.apply_rotary(q * D ** -0.5, ang), O.apply_rotary(k, ang)
    return torch.einsum("...hid,...hjd->...hij", q, k) + bias


def _linattn_ref(qkv, NI, n, H, D):
    q, k, v = (t.reshape(NI, n, H, D).permute(0, 2, 3, 1) for t in qkv.view(NI, n, 3 * H * D).chunk(3, dim=-1))
    q = q.softmax(dim=-2) * D ** -0.5
    k = k.softmax(dim=-1)
    ctx = torch.einsum("bhdn,bhen->bhde", k, v)
    out = torch.einsum("bhde,bhdn->bhen", ctx, q)
    return out.permute(0, 3, 1, 2).reshape(NI * n, H * D)


@pytest.mark.parametrize("NI,n,H", [(2, 256, 8), (3, 1024, 8), (1, 4096, 8), (6, 64, 8), (2, 24 * 36, 8), (2, 50, 8),
                                     (1, 7 * 9, 4), (6, 96 * 144, 8)])
def test_linear_attention_core(cuda, NI, n, H):
    from cesm_emulator_b200 import kernels as K
    torch.manual_seed(7)
    D = 32
    qkv = rnd((NI * n, 3 * H * D), cuda, 1.5)
    dout = rnd((NI * n, H * D), cuda)
    out, ws = K.linattn_fwd(qkv, NI, n, H, D, D ** -0.5)
    dqkv = K.linattn_bwd(qkv, ws, dout, NI, n, H, D, D ** -0.5)
    qr = qkv.float().requires_grad_(True)
    ref = _linattn_ref(qr, NI, n, H, D)
    assert err(out, ref) < 3e-3
    (g,) = torch.autograd.grad(ref, qr, dout.float())
    assert err(dqkv, g) < 3e-3


# ------------------------------------------------------------------------------------------------
# boundary convs, small linears, DDPM elementwise
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,Fr,H,W,f0", [(2, 3, 32, 32, 1), (1, 1, 48, 72, 1), (2, 3, 20, 36, 3)])
def test_input_conv(cuda, B, Fr, H, W, f0):
    from cesm_emulator_b200 import kernels as K
    torch.manual_seed(8)
    x = torch.randn(B, 1, f0, H, W, device=cuda)
    c = torch.randn(B, 1, Fr, H, W, device=cuda)
    w = torch.randn(64, 2, 1, 7, 7, device=cuda) * 0.1
    b = torch.randn(64, device=cuda)
    out = K.input_conv_fwd(x, c, w, b, B, Fr, H, W, 7)
    wr, br = w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    xin = torch.cat([x.expand(-1, -1, Fr, -1, -1), c], dim=1)
    ref = F.conv3d(xin, wr, br, padding=(0, 3, 3))  # [B,64,F,H,W]
    ref_cl = ref.permute(0, 2, 3, 4, 1).reshape(B * Fr, H, W, 64)
    assert err(out, ref_cl) < 2e-3
    dy = rnd((B * Fr, H, W, 64), cuda)
    dw, db = K.input_conv_wgrad(x, c, dy, B, Fr, H, W, 7)
    gw, gb = torch.autograd.grad(ref_cl, [wr, br], dy.float())
    assert err(dw, gw) < 2e-3 and err(db, gb) < 2e-3


@pytest.mark.parametrize("B,Fr,H,W,f0", [(2, 3, 32, 32, 1), (1, 1, 48, 72, 1), (2, 3, 20, 36, 3)])
def test_input_conv_tensor_core_path(cuda, B, Fr, H, W, f0):
    """ops.InputConvFn: (hi, lo) fp16 im2col patches through the tcgen05 GEMM and its weight-gradient
    kernel.  Against fp32 conv3d the forward differs only by the fp16 rounding of the weights and of the
    output; with fp16-representable weights and bias the patch split must recover the fp32 inputs, so the
    result then matches the old fp32-input CUDA-core kernel to output rounding."""
    from cesm_emulator_b200 import kernels as K, ops
    torch.manual_seed(8)
    x = torch.randn(B, 1, f0, H, W, device=cuda) * 3
    c = torch.randn(B, 1, Fr, H, W, device=cuda)
    w = (torch.randn(64, 2, 1, 7, 7, device=cuda) * 0.1).half().float()
    b = torch.randn(64, device=cuda)
    wp, bp = w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    out = ops.InputConvFn.apply(x, c, wp, bp, Fr)
    old = K.input_conv_fwd(x, c, w, b, B, Fr, H, W, 7)
    assert err(out, old) < 1e-3  # one fp16 ulp of the largest output
    assert (out.float() - old.float()).abs().mean().item() < 2e-3 * old.float().abs().mean().item()
    dy = rnd((B * Fr, H, W, 64), cuda)
    gw, gb = torch.autograd.grad(out, [wp, bp], dy)
    dw, db = K.input_conv_wgrad(x, c, dy, B, Fr, H, W, 7)
    assert err(gw, dw) < 1e-4 and err(gb, db) < 1e-4
    # patch layout: [hi | lo | 1 | 1 | 0...], hi + lo == x to ~2^-17
    pt = K.input_patches(x, c, B, Fr, H, W, 7).float()
    assert torch.equal(pt[..., 196:198], torch.ones_like(pt[..., 196:198])) and not pt[..., 198:].any()
    centre = 3 * 7 + 3  # tap (3,3) of plane 0 is the pixel itself
    xs = x.expand(-1, -1, Fr, -1, -1).reshape(B * Fr, H, W)
    assert (pt[..., centre] + pt[..., 98 + centre] - xs).abs().max().item() < 1e-4 * 3 * 4


def test_output_conv(cuda):
    from cesm_emulator_b200 import kernels as K
    torch.manual_seed(9)
    B, Fr, H, W = 2, 3, 16, 24
    a = rnd((B * Fr, H, W, 64), cuda)
    w = torch.randn(1, 64, 1, 1, 1, device=cuda) * 0.2
    b = torch.randn(1, device=cuda)
    eps = K.out_conv_fwd(a, w, b, B, Fr, H, W)
    ar, wr, br = a.float().requires_grad_(True), w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    full = (ar.view(B, Fr, H, W, 64) * wr.view(64)).sum(-1) + br
    ref = full[:, Fr // 2][:, None]
    assert err(eps, ref) < 2e-3
    de = torch.randn(B, 1, H, W, device=cuda)
    da, dw, db = K.out_conv_bwd(a, w, de, B, Fr, H, W)
    ga, gw, gb = torch.autograd.grad(ref, [ar, wr, br], de)
    assert err(da, ga) < 1e-2 and err(dw, gw) < 2e-3 and err(db, gb) < 2e-3


def test_time_embedding_and_small_linear(cuda):
    from cesm_emulator_b200 import kernels as K
    torch.manual_seed(10)
    t = torch.tensor([0, 1, 17, 999], device=cuda)
    assert err(K.sinusoidal(t, 64), O.sinusoidal_pos_emb(t, 64)) < 1e-5
    for act in (False, True):
        x = torch.randn(4, 256, device=cuda)
        W = torch.randn(512, 256, device=cuda) * 0.1
        b = torch.randn(512, device=cuda)
        y = K.small_linear_fwd(x, W, b, act)
        xr, Wr, br = x.clone().requires_grad_(True), W.clone().requires_grad_(True), b.clone().requires_grad_(True)
        ref = F.linear(F.silu(xr) if act else xr, Wr, br)
        assert err(y, ref) < 1e-4
        dy = torch.randn_like(y)
        dx, dW, db = K.small_linear_bwd(x, W, dy, act, True)
        gx, gW, gb = torch.autograd.grad(ref, [xr, Wr, br], dy)
        assert err(dx, gx) < 1e-4 and err(dW, gW) < 1e-4 and err(db, gb) < 1e-4


def test_ddpm_elementwise(cuda):
    from cesm_emulator_b200 import kernels as K
    torch.manual_seed(11)
    buf = {k: v.to(cuda) for k, v in O.diffusion_buffers(1000).items()}
    B, H, W = 3, 16, 24
    x0, noise = torch.randn(B, 1, H, W, device=cuda), torch.randn(B, 1, H, W, device=cuda)
    t = torch.tensor([0, 500, 999], device=cuda)
    xt = K.q_sample(x0, noise, t, buf["sqrt_alphas_cumprod"], buf["sqrt_one_minus_alphas_cumprod"])
    assert err(xt, O.q_sample(buf, x0, t, noise)) < 1e-6
    eps = torch.randn_like(x0)
    loss, diff = K.mse_fwd(eps, noise)
    assert abs(loss.item() - F.mse_loss(eps, noise).item()) < 1e-5
    g = torch.tensor([0.5], device=cuda)
    assert err(K.scale_by_scalar(diff, g, 2.0 / eps.numel()), (eps - noise) * 2 / eps.numel() * 0.5) < 1e-6
    z = torch.randn_like(x0)
    got = K.p_sample(xt, eps, z, t, buf["betas"], buf["sqrt_one_minus_alphas_cumprod"], buf["sqrt_recip_alphas"],
                     buf["posterior_variance"])
    beta = buf["betas"][t].view(-1, 1, 1, 1)
    mean = buf["sqrt_recip_alphas"][t].view(-1, 1, 1, 1) * (xt - beta / buf["sqrt_one_minus_alphas_cumprod"][t].view(-1, 1, 1, 1) * eps)
    ref = mean + torch.sqrt(buf["posterior_variance"][t].view(-1, 1, 1, 1)) * z
    assert err(got, ref) < 1e-6
    assert err(got[0], mean[0]) < 1e-6  # t == 0 adds no noise (model.py:178-179): posterior_variance[0] == 0
    assert buf["posterior_variance"][0].item() == 0.0


# ------------------------------------------------------------------------------------------------
# optimizer-step kernels: tiled batched re-layouts and the fused clip + AdamW
# ------------------------------------------------------------------------------------------------
def _descs(entries, cuda):
    from cesm_emulator_b200 import _lib
    arr = (_lib.PackDesc * len(entries))()
    for d, (src, dst, O, T, I, so, si, taps) in zip(arr, entries):
        d.src, d.dst, d.O, d.T, d.I, d.so, d.si = src, dst, O, T, I, so, si
        for i, o in enumerate(taps):
            d.tap_off[i] = int(o)
    return torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).to(cuda)


def test_batched_relayouts_match_single(cuda):
    """Every descriptor family the model registers (ops.py): forward [co][t][ci], data-gradient
    [ci][t][co] incl. the concat split, 1x1, 4x4 down-sampling and the 4-of-16-tap sub-pixel phases,
    ragged channel counts; pack is bit-exact, un-pack adds exactly and zeroes its scratch."""
    from cesm_emulator_b200 import _lib, kernels as K
    torch.manual_seed(5)
    cases = []  # (weight shape [A][B][T'], O, T, I, so, si, taps, src_off)
    for co, ci, kk in ((128, 64, 9), (64, 192, 9), (96, 40, 9), (768, 64, 1), (64, 256, 1), (64, 64, 16)):
        cases.append(((co, ci, kk), co, kk, ci, ci * kk, kk, list(range(kk)), 0))          # forward
        cases.append(((co, ci, kk), ci, kk, co, kk, ci * kk, list(range(kk)), 0))          # data gradient
    cases.append(((64, 128, 9), 64, 9, 64, 9, 128 * 9, list(range(9)), 64 * 9))            # concat split, 2nd half
    for ph in ([0, 2, 8, 10], [5, 7, 13, 15]):
        cases.append(((64, 64, 16), 64, 4, 64, 16, 64 * 16, ph, 0))                        # sub-pixel phase
    ws, outs, ents = [], [], []
    for shape, O, T, I, so, si, taps, off in cases:
        w = torch.randn(*shape, device=cuda)
        out = torch.empty(O, T * I, device=cuda, dtype=BF)
        ws.append(w); outs.append(out)
        ents.append((w.data_ptr() + 4 * off, out.data_ptr(), O, T, I, so, si, taps))
    tab = _descs(ents, cuda)
    _lib.call("cesm_pack_weights_batched", tab.data_ptr(), len(ents), K._stream())
    for (shape, O, T, I, so, si, taps, off), w, out in zip(cases, ws, outs):
        ref = K.pack_weight(w.reshape(-1)[off:], O, T, I, so, si, taps)
        assert torch.equal(out, ref), (shape, O, T, I)
    # un-pack: dst += scratch, scratch = 0
    grads, scr, ents = [], [], []
    shared = torch.randn(64, 64, 16, device=cuda)  # both sub-pixel phases add into ONE parameter gradient
    for shape, O, T, I, so, si, taps, off in cases:
        g = shared if T == 4 else torch.randn(*shape, device=cuda)
        s_ = torch.randn(O, T, I, device=cuda)
        grads.append(g); scr.append(s_)
        ents.append((s_.data_ptr(), g.data_ptr() + 4 * off, O, T, I, so, si, taps))
    want, shared_ref = [], shared.clone()
    for (shape, O, T, I, so, si, taps, off), g, s_ in zip(cases, grads, scr):
        r = shared_ref if T == 4 else g.clone()
        K.unpack_wgrad(s_, r.reshape(-1)[off:], O, T, I, so, si, taps, accumulate=True)
        want.append(r)
    tab = _descs(ents, cuda)
    _lib.call("cesm_unpack_wgrads_batched", tab.data_ptr(), len(ents), K._stream())
    for g, r, s_ in zip(grads, want, scr):
        assert torch.equal(g, r)
        assert not s_.any()


def _opt_state(cuda, lr, wd, scale=1.0, interval=0):
    from cesm_emulator_b200 import kernels as K
    st = torch.zeros(K.OPT_STATE_FLOATS)
    st[K.OPT_LR], st[K.OPT_WD], st[K.OPT_SCALE], st[K.OPT_INTERVAL] = lr, wd, scale, interval
    return st.to(cuda)


@pytest.mark.parametrize("n,max_norm,scale", [(10_001, 1.0, 1.0), (4096, None, 65536.0), (1_234_567, 0.05, 1024.0)])
def test_fused_adamw_matches_torch(cuda, n, max_norm, scale):
    """cesm_adamw_step against torch.optim.AdamW + clip_grad_norm_ (train.py:865, 1078-1083); the kernel is handed
    gradients multiplied by the loss scale and must unscale them first (GradScaler.unscale_, train.py:864)."""
    from cesm_emulator_b200 import _lib, kernels as K
    torch.manual_seed(1)
    hp = dict(lr=2e-4, betas=(0.9, 0.999), weight_decay=1e-4, eps=1e-8)
    p0 = torch.randn(n, device=cuda)
    ref = torch.nn.Parameter(p0.clone())
    opt = torch.optim.AdamW([ref], **hp)
    p, m, v = p0.clone(), torch.zeros(n, device=cuda), torch.zeros(n, device=cuda)
    state = _opt_state(cuda, hp["lr"], hp["weight_decay"], scale)
    partials = torch.zeros(_lib.load().cesm_adamw_partials(), device=cuda)
    for step in range(4):
        g = torch.randn(n, device=cuda) * (0.5 + step)
        ref.grad = g.clone()
        norm = torch.linalg.vector_norm(g)
        if max_norm is not None:
            torch.nn.utils.clip_grad_norm_([ref], max_norm)
        opt.step()
        K.adamw_step(p, g * scale, m, v, partials, state, *hp["betas"], hp["eps"], max_norm)
        assert state[K.OPT_STEP].item() == step + 1 and state[K.OPT_FOUND_INF].item() == 0
        assert abs(state[K.OPT_NORM].item() - norm.item()) < 1e-4 * norm.item()
        assert (p - ref.data).abs().max().item() < 2e-6, step
        if step == 1:  # a new learning rate written to the device state is honoured by the next call
            for gr in opt.param_groups:
                gr["lr"] = 5e-4
            state[K.OPT_LR] = 5e-4
    assert err(m, opt.state[ref]["exp_avg"]) < 1e-4 and err(v, opt.state[ref]["exp_avg_sq"]) < 1e-4


def test_fused_adamw_follows_grad_scaler(cuda):
    """The device-side loss-scale logic against torch.amp.GradScaler driving torch AdamW (train.py:862-867,
    1084): an overflowing gradient skips the update and halves the scale; `growth_interval` clean steps double it."""
    from cesm_emulator_b200 import _lib, kernels as K
    torch.manual_seed(2)
    n, interval = 5000, 3
    hp = dict(lr=1e-3, betas=(0.9, 0.999), weight_decay=1e-2, eps=1e-8)
    p0 = torch.randn(n, device=cuda)
    ref = torch.nn.Parameter(p0.clone())
    opt = torch.optim.AdamW([ref], **hp)
    scaler = torch.amp.GradScaler("cuda", init_scale=65536.0, growth_interval=interval)
    scaler.scale(torch.zeros(1, device=cuda))  # lazy initialisation of the scale tensor
    p, m, v = p0.clone(), torch.zeros(n, device=cuda), torch.zeros(n, device=cuda)
    state = _opt_state(cuda, hp["lr"], hp["weight_decay"], 65536.0, interval)
    partials = torch.zeros(_lib.load().cesm_adamw_partials(), device=cuda)
    overflow_at = {2, 7}
    for step in range(12):
        g = torch.randn(n, device=cuda) * 0.1
        S = scaler.get_scale()
        assert state[K.OPT_SCALE].item() == S, (step, state[K.OPT_SCALE].item(), S)
        gs = g * S
        if step in overflow_at:
            gs[step] = float("inf")
        ref.grad = gs.clone()
        # torch flow (scaler.scale(loss).backward() produced gs)
        scaler.unscale_(opt)
        torch.nn.utils.clip_grad_norm_([ref], 1.0)
        scaler.step(opt)
        scaler.update()
        K.adamw_step(p, gs, m, v, partials, state, *hp["betas"], hp["eps"], 1.0)
        assert state[K.OPT_FOUND_INF].item() == float(step in overflow_at)
        assert (p - ref.data).abs().max().item() < 2e-6, step
    assert state[K.OPT_SKIPPED].item() == 2 and state[K.OPT_STEP].item() == 10
    assert state[K.OPT_SCALE].item() == scaler.get_scale()


# ------------------------------------------------------------------------------------------------
# on-device data path (SURVEY 8(f) rank 3)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K,crop", [(3, None), (3, (16, 24)), (5, (16, 16)), (4, (8, 40))])
def test_device_data_path(cuda, K, crop):
    """One gather kernel over the HBM-resident (T, M, H, W) arrays reproduces the host data path bit for bit:
    same windows, time reversal, crops and random stream (two generators with the same seed)."""
    from cesm_emulator_b200.synthetic import SyntheticEnsemble
    kw = dict(members=3, times=12, lat=24, lon=40, seed=5, K=K, crop_hw=crop, time_reverse_p=0.5)
    host, ds = SyntheticEnsemble(**kw), SyntheticEnsemble(**kw)
    dev = ds.to_device(cuda)
    h, w = ds.out_hw()
    B = 4
    cond = torch.empty(B, 1, K, h, w, device=cuda)
    x0 = torch.empty(B, 1, h, w, device=cuda)
    g = torch.Generator().manual_seed(1)
    seen_rev = 0
    for _ in range(6):
        idx = torch.randint(0, len(ds), (B,), generator=g).tolist()
        ref_c, ref_x = host.batch(idx)
        dev.batch_into(idx, cond, x0)
        assert torch.equal(cond.cpu(), ref_c) and torch.equal(x0.cpu(), ref_x)
        seen_rev += int(dev._plan_dev[:, 5].sum().item())
    assert seen_rev > 0  # the augmentation branch was exercised
    # no augmentation: centre crop, no reversal
    idx = [0, 1, len(ds) - 1, 7]
    ref_c, ref_x = host.batch(idx, augment=False)
    dev.batch_into(idx, cond, x0, augment=False)
    assert torch.equal(cond.cpu(), ref_c) and torch.equal(x0.cpu(), ref_x)


def test_device_data_path_matches_reference_dataset_class(cuda):
    """The gather kernel against windows produced by the REFERENCE's dataset class (dataset_single_member.py:
    168-196; fixture written by tests/golden/make_dataset_golden.py from the imported class)."""
    import numpy as np
    from cesm_emulator_b200.synthetic import SyntheticEnsemble
    from test_host_logic import _ScriptedDraws, _dataset_fixture
    g, cond_np, tgt_np = _dataset_fixture()
    cases = [(3, None, 0.0, True, "plain_K3"), (4, None, 1.0, True, "rev_K4"), (5, None, 1.0, True, "rev_K5"),
             (3, (8, 10), 0.0, False, "center_crop"), (3, (64, 10), 0.0, False, "clamped_crop"),
             (3, (8, 10), 0.5, True, "random_crop")]
    for K, crop, p, augment, key in cases:
        ds = SyntheticEnsemble.from_arrays(cond_np, tgt_np, K=K, crop_hw=crop, time_reverse_p=p)
        if key == "random_crop":
            ds._aug = _ScriptedDraws(g["random_crop_origin"])
        dev = ds.to_device(cuda)
        h, w = ds.out_hw()
        n = len(ds)
        cond = torch.empty(n, 1, K, h, w, device=cuda)
        x0 = torch.empty(n, 1, h, w, device=cuda)
        dev.batch_into(list(range(n)), cond, x0, augment=augment)
        assert np.array_equal(cond.cpu().numpy(), g[key + "_cond"]), key
        assert np.array_equal(x0.cpu().numpy(), g[key + "_x0"]), key


def test_device_data_path_survives_host_run_ahead(cuda):
    """The training loop never syncs inside an epoch: the host may issue dozens of batches while the GPU is still
    busy with the first.  Every batch must still be the one the host path would have produced (the pinned plan
    ring is guarded by events; a bare 8-slot ring was overwritten before its async copies ran)."""
    from cesm_emulator_b200.synthetic import SyntheticEnsemble
    kw = dict(members=3, times=12, lat=24, lon=40, seed=5, K=3, crop_hw=(16, 24), time_reverse_p=0.5)
    host, ds = SyntheticEnsemble(**kw), SyntheticEnsemble(**kw)
    dev = ds.to_device(cuda)
    B, n = 4, 40
    g = torch.Generator().manual_seed(2)
    idxs = [torch.randint(0, len(ds), (B,), generator=g).tolist() for _ in range(n)]
    refs = [host.batch(i) for i in idxs]
    conds = [torch.empty(B, 1, 3, 16, 24, device=cuda) for _ in range(n)]
    x0s = [torch.empty(B, 1, 16, 24, device=cuda) for _ in range(n)]
    big = torch.randn(8192, 8192, device=cuda)
    torch.cuda.synchronize()
    for _ in range(20):          # ~tens of ms of queued GPU work: the stream lags far behind the host
        big = big @ big * 1e-4
    for i in range(n):
        dev.batch_into(idxs[i], conds[i], x0s[i])
    torch.cuda.synchronize()
    for i in range(n):
        assert torch.equal(conds[i].cpu(), refs[i][0]) and torch.equal(x0s[i].cpu(), refs[i][1]), i


@pytest.mark.parametrize("rows_shape", [(2, 16, 24), (1, 5, 7), (16, 48, 72)])
def test_layernorm_folded_into_projection(cuda, rows_shape):
    """kernels.igemm(ln_fold=): x + LN(x) W^T from ONE GEMM whose epilogue takes the row statistics from its residual
    (the one-frame temporal-attention block, video_net.py:78-87 + :380-453), against the two-kernel form and fp32 torch."""
    from cesm_emulator_b200 import kernels as K
    torch.manual_seed(11)
    C, eps = 64, 1e-5
    x = (rnd((*rows_shape, C), cuda) * 1.5 + 0.7).contiguous()          # rows with a non-zero mean
    gamma = 1.0 + 0.2 * torch.randn(C, device=cuda)
    w = torch.randn(C, C, device=cuda) * 0.1
    wln = (w * gamma[None, :]).to(K.H16)
    colsum = wln.float().sum(dim=1)
    y = K.igemm(x, wln, residual=x, ln_fold=(colsum, eps))
    xf = x.float()
    mu = xf.mean(-1, keepdim=True)
    var = xf.var(-1, unbiased=False, keepdim=True)
    ref = xf + ((xf - mu) / (var + eps).sqrt() * gamma) @ w.t()
    assert err(y, ref) < 2e-3
    two = K.igemm(K.ln_fwd(x, gamma, eps), w.to(K.H16), residual=x)
    assert err(y, two.float()) < 2e-3
    with pytest.raises(AssertionError):
        K.igemm(x, wln, residual=x.clone(), ln_fold=(colsum, eps))       # the residual must be the GEMM input itself


@pytest.mark.parametrize("NI,n,C,H", [(2, 16 * 24, 64, 8), (3, 100, 64, 4), (2, 36 * 18, 128, 8), (1, 17, 128, 4),
                                      (16, 48 * 72, 64, 8)])
def test_linear_attention_with_output_projection(cuda, NI, n, C, H):
    """The tail of the spatial-attention block as sampling runs it: cesm_linattn_fwd, then the 1x1 projection GEMM
    with bias and residual (y = x + bout + W_out * attention), against fp32 torch."""
    from cesm_emulator_b200 import kernels as K
    torch.manual_seed(13)
    D = 32
    hid = H * D
    qkv = rnd((NI * n, 3 * hid), cuda)
    x = rnd((NI * n, C), cuda)
    wout = torch.randn(C, hid, device=cuda) * 0.1
    bout = torch.randn(C, device=cuda)
    o, _ = K.linattn_fwd(qkv, NI, n, H, D, D ** -0.5)
    y = K.igemm(o.view(NI, 1, n, hid), wout.to(K.H16), bias=bout, residual=x.view(NI, 1, n, C)).view(-1, C)
    # fp32 restatement (video_net.py:338-347)
    q, k, v = qkv.float().view(NI, n, 3, H, D).unbind(2)
    qs = q.softmax(-1) * D ** -0.5
    ks = k.softmax(1)
    ctx = torch.einsum("bnhd,bnhe->bhde", ks, v)
    out = torch.einsum("bhde,bnhd->bnhe", ctx, qs).reshape(NI * n, hid)
    ref = x.float() + out @ wout.t() + bout
    assert err(y, ref) < 3e-3


def test_film_projections_batched(cuda):
    """ops.FilmAllFn (all FiLM linears of a pass in one launch, one fused backward) against torch."""
    from cesm_emulator_b200 import ops
    torch.manual_seed(6)
    B, Kd = 3, 256
    Ns = [128, 128, 256, 512, 128]
    t = torch.randn(B, Kd, device=cuda, requires_grad=True)
    Ws = [(torch.randn(n, Kd, device=cuda) * 0.05).requires_grad_(True) for n in Ns]
    bs = [torch.randn(n, device=cuda).requires_grad_(True) for n in Ns]
    outs = ops.FilmAllFn.apply(t, *[p for w, b in zip(Ws, bs) for p in (w, b)])
    refs = [F.linear(F.silu(t), w, b) for w, b in zip(Ws, bs)]
    for o, r in zip(outs, refs):
        assert o.shape == r.shape and err(o, r) < 1e-5
    gs = [torch.randn_like(r) for r in refs]
    loss = sum((o * g).sum() for o, g in zip(outs, gs))
    got = torch.autograd.grad(loss, [t] + Ws + bs)
    want = torch.autograd.grad(sum((r * g).sum() for r, g in zip(refs, gs)), [t] + Ws + bs)
    for a, b_ in zip(got, want):
        assert err(a, b_) < 1e-5
