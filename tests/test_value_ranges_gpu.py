"""GPU parity of the normalisation and softmax kernels at the values a trained, loss-scaled network produces rather than
the N(0, 1) of a random initialisation: SiLU pre-activations out to |u| ~ 24, sharp and shifted softmax logits, and
normalisation statistics of tensors whose mean is many standard deviations from zero.

References are float64 torch on the same fp16-rounded inputs the kernels read; errors are max|got - ref| / max|ref| per
tensor, against the bars of tests/test_kernels_gpu.py (2e-3 for outputs and norm gradients, 3e-3 for attention
gradients and linear-attention outputs).  Every assertion message carries the measured error."""
import math

import pytest
import torch
import torch.nn.functional as F

from test_kernels_gpu import _fold_diagonals, _linattn_ref, _tattn_ref, _tattn_scores, _toeplitz_bias

pytestmark = pytest.mark.gpu
H16, F64 = torch.float16, torch.float64
EPS = 1e-5
U_BINS = [(0.0, 2.0), (2.0, 6.0), (6.0, 12.0), (12.0, 24.0), (24.0, math.inf)]


def _err(got, ref, mask=None):
    """max|got - ref| / max|ref|; with `mask` the numerator is taken over the masked elements only."""
    d = (got.double() - ref.double()).abs()
    if mask is not None:
        d = d[mask]
    num = d.max().item() if d.numel() else 0.0
    return num / (ref.double().abs().max().item() + 1e-300)


def _gn_ref(x, gamma, beta, film, res, B, G, dout):
    """float64 GroupNorm + FiLM + SiLU (+ residual) and its gradients -> (out, u, grads[x, gamma, beta(, film)])."""
    C = x.shape[-1]
    xr = x.to(F64).requires_grad_(True)
    gr, br = gamma.to(F64).requires_grad_(True), beta.to(F64).requires_grad_(True)
    leaves = [xr, gr, br]
    u = F.group_norm(xr.transpose(1, 2), G, gr, br, EPS)
    if film is not None:
        flr = film.to(F64).requires_grad_(True)
        leaves.append(flr)
        u = u * (flr[:, :C, None] + 1) + flr[:, C:, None]
    u = u.transpose(1, 2)
    y = F.silu(u)
    out = y + (res.to(F64) if res is not None else 0)
    grads = torch.autograd.grad(y, leaves, dout.to(F64))
    return out.detach(), u.detach(), grads


def _gn_run(K, x, gamma, beta, film, res, dout, B, G):
    sums = K.gn_stats(x, B, G)
    out = K.gn_apply_fwd(x, sums, gamma, beta, film, res, B, G, EPS)
    dx, dg, db, dfl, dcb = K.gn_bwd(x, dout, sums, gamma, beta, film, B, G, EPS, conv_bias_grad=True)
    return sums, out, dx, dg, db, dfl, dcb


# ------------------------------------------------------------------------------------------------
# A. GroupNorm + FiLM + SiLU with saturated pre-activations
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("film_res", [False, True], ids=["plain", "film_res"])
@pytest.mark.parametrize("B,P,C,G", [(2, 3 * 128 * 128, 64, 8), (2, 3 * 32 * 32, 256, 8), (2, 3 * 8 * 8, 512, 8),
                                     (2, 3 * 192 * 288, 64, 8)])
def test_groupnorm_silu_saturated(cuda, B, P, C, G, film_res):
    """gamma / beta (and FiLM scale / shift) put u = GN(x) gamma + beta (FiLM'd) over about +-24 with most elements at
    6 <= |u| <= 18, where silu'(u) is 1 or 0 up to a small difference of tanh(u/2) from 1.  `out` and `dx` are also
    checked per |u| bin (numerator over the bin, denominator the whole tensor's max|ref|)."""
    from cesm_emulator_b200 import kernels as K
    g = torch.Generator(device=cuda).manual_seed(P + C)
    x = torch.randn(B, P, C, device=cuda, generator=g).to(H16)
    sign = torch.where(torch.rand(C, device=cuda, generator=g) < 0.5, -1.0, 1.0)
    gamma = sign * (3.0 + 4.0 * torch.rand(C, device=cuda, generator=g))
    beta = 24.0 * torch.rand(C, device=cuda, generator=g) - 12.0
    film = res = None
    if film_res:
        film = torch.cat([0.6 * torch.rand(B, C, device=cuda, generator=g) - 0.3,
                          6.0 * torch.rand(B, C, device=cuda, generator=g) - 3.0], dim=1)
        res = torch.randn(B, P, C, device=cuda, generator=g).to(H16)
    dout = torch.randn(B, P, C, device=cuda, generator=g).to(H16)
    _, out, dx, dg, db, dfl, dcb = _gn_run(K, x, gamma, beta, film, res, dout, B, G)
    ref, u, grads = _gn_ref(x, gamma, beta, film, res, B, G, dout)
    au = u.abs()
    assert au.max().item() > 20 and ((au >= 6) & (au <= 18)).double().mean().item() > 0.4  # the regime under test
    errs = {"out": _err(out, ref), "dx": _err(dx, grads[0]), "dgamma": _err(dg, grads[1]), "dbeta": _err(db, grads[2]),
            "dconv_bias": _err(dcb, grads[0].sum(dim=(0, 1)))}
    if film is not None:
        errs["dfilm"] = _err(dfl, grads[3])
    for lo, hi in U_BINS:
        m = (au >= lo) & (au < hi)
        errs[f"out|u|[{lo:g},{hi:g})"] = _err(out, ref, m)
        errs[f"dx|u|[{lo:g},{hi:g})"] = _err(dx, grads[0], m)
    print(f"groupnorm saturated B={B} P={P} C={C} film_res={film_res}: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    bad = {k: v for k, v in errs.items() if not v < 2e-3}
    assert not bad, f"errors above 2e-3: {bad}; all: {errs}"


# ------------------------------------------------------------------------------------------------
# B. softmax kernels with sharp and shifted logits
# ------------------------------------------------------------------------------------------------
def _rope(Fr, D, dev):
    freqs = (1.0 / (10000 ** (torch.arange(0, D, 2).float() / D))).to(dev)
    ang = torch.arange(Fr, device=dev, dtype=torch.float32)[:, None] * freqs[None]
    return freqs, ang.cos().contiguous(), ang.sin().contiguous()


@pytest.mark.parametrize("shift", [-300.0, 300.0])
@pytest.mark.parametrize("B,Fr,HW,H", [(2, 1, 256, 8), (2, 3, 64, 8), (2, 12, 33, 8), (1, 128, 6, 8)])
def test_temporal_attention_sharp_and_shifted(cuda, B, Fr, HW, H, shift):
    """q and k scaled so the scaled logits have a standard deviation of about 10 (rows nearly one-hot), every 7th row
    with q = 0, and a constant added to every bias entry (F <= 4) or diagonal (F > 4).  The bias is fp32, so the shift
    cancels exactly in the softmax: the output must also match the kernel's own output without it."""
    from cesm_emulator_b200 import kernels as K
    D = 32
    g = torch.Generator(device=cuda).manual_seed(Fr * 1000 + HW)
    rows = B * Fr * HW
    qkv = torch.randn(rows, 3 * H * D, device=cuda, generator=g)
    qkv[:, :2 * H * D] *= math.sqrt(10.0)
    qkv[::7, :H * D] = 0.0
    qkv = qkv.to(H16)
    if Fr <= 4:
        bias0 = torch.randn(H, Fr, Fr, device=cuda, generator=g)
    else:
        diag = torch.randn(H, 2 * Fr - 1, device=cuda, generator=g)
        i = torch.arange(Fr, device=cuda)
        bias0 = diag[:, (i[None, :] - i[:, None]) + Fr - 1].contiguous()
    bias = (bias0 + shift).contiguous()
    freqs, cs, sn = _rope(Fr, D, cuda)
    dout = torch.randn(rows, H * D, device=cuda, generator=g).to(H16)
    out, lse = K.tattn_fwd(qkv, bias, cs, sn, B, Fr, HW, H, D, D ** -0.5)
    dqkv, dbias = K.tattn_bwd(qkv, bias, cs, sn, out, lse, dout, B, Fr, HW, H, D, D ** -0.5)
    out0, _ = K.tattn_fwd(qkv, bias0, cs, sn, B, Fr, HW, H, D, D ** -0.5)
    qr, br = qkv.to(F64).requires_grad_(True), bias.to(F64).requires_grad_(True)
    ref = _tattn_ref(qr, br, freqs, B, Fr, HW, H, D)
    gq, gb = torch.autograd.grad(ref, [qr, br], dout.to(F64))
    s = _tattn_scores(qkv.to(F64), bias.to(F64), freqs, B, Fr, HW, H, D)
    assert s.std().item() > 7, s.std().item()
    errs = {"out": _err(out, ref), "shift_invariance": _err(out, out0), "dqkv": _err(dqkv, gq)}
    if Fr <= 4:
        errs["dbias"] = _err(dbias, gb)
    else:
        errs["dbias_diag"] = _err(_fold_diagonals(dbias.double(), Fr), _fold_diagonals(gb, Fr))
        lse_ref = torch.logsumexp(s, dim=-1)
        errs["lse"] = _err(lse.view(B, Fr, HW, H).permute(0, 2, 3, 1), lse_ref)
    print(f"tattn sharp F={Fr} shift={shift:+g}: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    bars = {"out": 2e-3, "shift_invariance": 2e-3, "dqkv": 3e-3, "dbias": 2e-3, "dbias_diag": 3e-3, "lse": 2e-3}
    bad = {k: v for k, v in errs.items() if not v < bars[k]}
    assert not bad, f"errors above their bars: {bad}; all: {errs}"


@pytest.mark.parametrize("B,Fr,HW", [(2, 1, 256), (1, 2, 160), (2, 3, 64)])
def test_temporal_attention_fused_projection_sharp(cuda, B, Fr, HW):
    """csrc/tattn_proj.cu with W scaled so the q / k projections give logits of standard deviation about 10."""
    from cesm_emulator_b200 import kernels as K
    H, D, C = 8, 32, 64
    g = torch.Generator(device=cuda).manual_seed(Fr * 100 + HW)
    rows = B * Fr * HW
    xn = torch.randn(rows, C, device=cuda, generator=g).to(H16)
    w = torch.randn(3 * H * D, C, device=cuda, generator=g) * C ** -0.5
    w[:2 * H * D] *= math.sqrt(10.0)
    w = w.to(H16)
    bias = torch.randn(H, Fr, Fr, device=cuda, generator=g)
    freqs, cs, sn = _rope(Fr, D, cuda)
    out = K.tattn_proj_fwd(xn, w, bias, cs, sn, B, Fr, HW, H, D, D ** -0.5)
    qkv = xn.to(F64) @ w.to(F64).t()
    ref = _tattn_ref(qkv, bias.to(F64), freqs, B, Fr, HW, H, D)
    s = _tattn_scores(qkv, bias.to(F64), freqs, B, Fr, HW, H, D)
    e = _err(out, ref)
    print(f"tattn_proj sharp F={Fr}: logit std {s.std().item():.1f}, out {e:.2e}")
    assert s.std().item() > 7, s.std().item()
    assert e < 2e-3, f"out error {e:.3e}"


def _mattn_ref64(qkv, dout, NI, n, H):
    t = qkv.to(F64).view(NI, n, 3, H, 32).permute(2, 0, 3, 1, 4)
    q, k, v = (t[i].clone().requires_grad_(True) for i in range(3))
    s = (q * 32 ** -0.5) @ k.transpose(-1, -2)
    lse = torch.logsumexp(s, dim=-1)
    o = torch.softmax(s, dim=-1) @ v
    o.backward(dout.to(F64).view(NI, n, H, 32).permute(0, 2, 1, 3))
    lay = lambda a: a.permute(0, 2, 1, 3).reshape(NI * n, H * 32)
    return lay(o.detach()), lse.detach().permute(0, 2, 1).reshape(NI * n, H), [lay(a.grad) for a in (q, k, v)]


@pytest.mark.parametrize("NI,n,H", [(6, 1024, 8), (2, 216, 8), (1, 16, 8), (3, 45, 4)])
def test_mid_attention_sharp(cuda, NI, n, H):
    """csrc/mid_attn.cu with q scaled x8 (logit standard deviation about 8)."""
    from cesm_emulator_b200 import kernels as K
    g = torch.Generator(device=cuda).manual_seed(n + H)
    qkv = torch.randn(NI * n, 3 * H * 32, device=cuda, generator=g)
    qkv[:, :H * 32] *= 8.0
    qkv = qkv.to(H16)
    dout = torch.randn(NI * n, H * 32, device=cuda, generator=g).to(H16)
    out, lse = K.mattn_fwd(qkv, NI, n, H, 32, 32 ** -0.5)
    dqkv = K.mattn_bwd(qkv, out, lse, dout, NI, n, H, 32, 32 ** -0.5)
    o_r, lse_r, (dq, dk, dv) = _mattn_ref64(qkv, dout, NI, n, H)
    hid = H * 32
    errs = {"out": _err(out, o_r), "lse": _err(lse, lse_r), "dq": _err(dqkv[:, :hid], dq),
            "dk": _err(dqkv[:, hid:2 * hid], dk), "dv": _err(dqkv[:, 2 * hid:], dv)}
    print(f"mattn sharp NI={NI} n={n}: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    bars = {"out": 2e-3, "lse": 2e-3, "dq": 3e-3, "dk": 3e-3, "dv": 3e-3}
    bad = {k: v for k, v in errs.items() if not v < bars[k]}
    assert not bad, f"errors above their bars: {bad}; all: {errs}"


@pytest.mark.parametrize("NI,n", [(16, 48 * 72), (2, 192 * 288)])
def test_linear_attention_shifted(cuda, NI, n):
    """Linear attention with a per-row constant added to q (shifts its softmax over d), k of standard deviation 4 plus a
    per-(image, head, d) constant of +-32 over all pixels (shifts its softmax over pixels)."""
    from cesm_emulator_b200 import kernels as K
    H, D = 8, 32
    hid = H * D
    g = torch.Generator(device=cuda).manual_seed(n)
    qkv = torch.randn(NI * n, 3 * hid, device=cuda, generator=g)
    qkv[:, :hid] += 40.0 * torch.rand(NI * n, 1, device=cuda, generator=g) - 20.0
    kc = torch.where(torch.rand(NI, 1, hid, device=cuda, generator=g) < 0.5, -32.0, 32.0)
    k = qkv[:, hid:2 * hid].view(NI, n, hid)
    k.mul_(4.0).add_(kc)
    qkv = qkv.to(H16)
    dout = torch.randn(NI * n, hid, device=cuda, generator=g).to(H16)
    out, ws = K.linattn_fwd(qkv, NI, n, H, D, D ** -0.5)
    dqkv = K.linattn_bwd(qkv, ws, dout, NI, n, H, D, D ** -0.5)
    qr = qkv.to(F64).requires_grad_(True)
    ref = _linattn_ref(qr, NI, n, H, D)
    (gq,) = torch.autograd.grad(ref, qr, dout.to(F64))
    errs = {"out": _err(out, ref), "dqkv": _err(dqkv, gq)}
    print(f"linattn shifted NI={NI} n={n}: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    bad = {k: v for k, v in errs.items() if not v < 3e-3}
    assert not bad, f"errors above 3e-3: {bad}; all: {errs}"


# ------------------------------------------------------------------------------------------------
# C. normalisation statistics at offset means
# ------------------------------------------------------------------------------------------------
RATIOS = [0.0, 4.0, 16.0, 32.0]   # mean / std of a group or row; plus one exactly constant group / row
CONST = 3.3


def _offset_groups(B, P, C, G, g, dev, sigma=0.5):
    """x = mu_g + sigma z with group mean / std cycling through RATIOS and the last group constant."""
    cpg = C // G
    mu = torch.tensor([RATIOS[i % len(RATIOS)] * sigma for i in range(G)], device=dev)
    sig = torch.full((G,), sigma, device=dev)
    mu[-1], sig[-1] = CONST, 0.0
    sgn = torch.where(torch.arange(G, device=dev) % 2 == 0, 1.0, -1.0)
    mu_c, sig_c = (mu * sgn).repeat_interleave(cpg), sig.repeat_interleave(cpg)
    return (mu_c + sig_c * torch.randn(B, P, C, device=dev, generator=g)).to(H16)


@pytest.mark.parametrize("B,P,C,film", [(2, 3 * 32 * 32, 64, True), (2, 3 * 16 * 16, 256, False), (1, 1000, 512, True)])
def test_groupnorm_offset_means(cuda, B, P, C, film):
    """gn_stats -> gn_apply_fwd / gn_bwd on groups with mean / std 0, 4, 16, 32 and one constant group (torch: xhat = 0
    there; the kernels' variance is sum(x^2)/n - mean^2 from fp32 sums)."""
    from cesm_emulator_b200 import kernels as K
    G = 8
    g = torch.Generator(device=cuda).manual_seed(C + P)
    x = _offset_groups(B, P, C, G, g, cuda)
    gamma = torch.randn(C, device=cuda, generator=g) * 0.5 + 1
    beta = torch.randn(C, device=cuda, generator=g) * 0.2
    fl = torch.randn(B, 2 * C, device=cuda, generator=g) * 0.3 if film else None
    dout = torch.randn(B, P, C, device=cuda, generator=g).to(H16)
    _, out, dx, dg, db, dfl, dcb = _gn_run(K, x, gamma, beta, fl, None, dout, B, G)
    ref, _, grads = _gn_ref(x, gamma, beta, fl, None, B, G, dout)
    errs = {"out": _err(out, ref), "dx": _err(dx, grads[0]), "dgamma": _err(dg, grads[1]), "dbeta": _err(db, grads[2]),
            "dconv_bias": _err(dcb, grads[0].sum(dim=(0, 1)))}
    if film:
        errs["dfilm"] = _err(dfl, grads[3])
    print(f"groupnorm offset B={B} P={P} C={C}: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    bad = {k: v for k, v in errs.items() if not v < 2e-3}
    assert not bad, f"errors above 2e-3: {bad}; all: {errs}"


@pytest.mark.parametrize("n,h,w,frames", [(6, 32, 32, 3), (2, 48, 72, 1)])
def test_conv_fused_groupnorm_sums_offset_means(cuda, n, h, w, frames):
    """K.igemm(gn_sums=) on a 3x3 conv whose bias supplies group means of 0, 4, 16, 32 output standard deviations and
    whose last group has zero weights (a constant group): the sums against float64 sums of the stored fp16 output, and
    gn_apply_fwd fed those sums against float64 GroupNorm + SiLU of that output."""
    from cesm_emulator_b200 import kernels as K
    G, cin, cout = 8, 64, 64
    g = torch.Generator(device=cuda).manual_seed(h * w)
    x = torch.randn(n, h, w, cin, device=cuda, generator=g).to(H16)
    wt = torch.randn(cout, 9 * cin, device=cuda, generator=g) * (9 * cin) ** -0.5   # output std ~ 1
    cpg = cout // G
    wt[-cpg:] = 0.0
    wt = wt.to(H16)
    mu = torch.tensor([RATIOS[i % len(RATIOS)] * (1 if i % 2 == 0 else -1) for i in range(G)], device=cuda)
    mu[-1] = CONST
    bias = mu.repeat_interleave(cpg) + 0.1 * torch.randn(cout, device=cuda, generator=g)
    bias[-cpg:] = CONST
    sums = torch.full((n // frames, G, 2), 123.0, device=cuda)
    y = K.igemm(x, wt, taps=K.TAPS_3x3, bias=bias, gn_sums=sums, gn_frames=frames)
    yd = y.to(F64).view(n // frames, frames * h * w, G, cpg)
    want = torch.stack([yd.sum(dim=(1, 3)), (yd * yd).sum(dim=(1, 3))], dim=-1)
    Bs = n // frames
    yv = y.view(Bs, frames * h * w, cout)
    gamma = torch.randn(cout, device=cuda, generator=g) * 0.5 + 1
    beta = torch.randn(cout, device=cuda, generator=g) * 0.2
    out = K.gn_apply_fwd(yv, sums, gamma, beta, None, None, Bs, G, EPS)
    ref = F.silu(F.group_norm(yv.to(F64).transpose(1, 2), G, gamma.to(F64), beta.to(F64), EPS)).transpose(1, 2)
    errs = {"sum": _err(sums[..., 0], want[..., 0]), "sumsq": _err(sums[..., 1], want[..., 1]), "gn_out": _err(out, ref)}
    print(f"igemm gn_sums offset n={n} {h}x{w}: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    assert errs["sum"] < 1e-4 and errs["sumsq"] < 1e-4, f"sums: {errs}"
    assert errs["gn_out"] < 2e-3, f"GroupNorm from the fused sums: {errs}"


def _offset_rows(M, C, g, dev, sigma=0.5):
    r = torch.tensor(RATIOS, device=dev)[torch.arange(M, device=dev) % len(RATIOS)] * sigma
    r = r * torch.where(torch.arange(M, device=dev) % 3 == 0, -1.0, 1.0)
    x = r[:, None] + sigma * torch.randn(M, C, device=dev, generator=g)
    x[M // 2] = CONST
    return x.to(H16)


def _ln64(x, gamma):
    mean = x.mean(dim=-1, keepdim=True)
    var = ((x - mean) ** 2).mean(dim=-1, keepdim=True)
    return (x - mean) / (var + EPS).sqrt() * gamma


@pytest.mark.parametrize("M,C", [(1000, 64), (300, 256), (200, 1024)])
def test_layernorm_offset_means(cuda, M, C):
    """ln_fwd / ln_bwd (C = 1024 included) on rows with mean / std 0, 4, 16, 32 and one constant row."""
    from cesm_emulator_b200 import kernels as K
    g = torch.Generator(device=cuda).manual_seed(M + C)
    x = _offset_rows(M, C, g, cuda)
    gamma = torch.randn(C, device=cuda, generator=g) * 0.5 + 1
    dy = torch.randn(M, C, device=cuda, generator=g).to(H16)
    dres = torch.randn(M, C, device=cuda, generator=g).to(H16)
    out = K.ln_fwd(x, gamma, EPS)
    dx, dg = K.ln_bwd(x, gamma, dy, dres, EPS)
    xr, gr = x.to(F64).requires_grad_(True), gamma.to(F64).requires_grad_(True)
    y = _ln64(xr, gr)
    gx, gg = torch.autograd.grad(y, [xr, gr], dy.to(F64))
    errs = {"out": _err(out, y), "dx": _err(dx, gx + dres.to(F64)), "dgamma": _err(dg, gg)}
    print(f"layernorm offset M={M} C={C}: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    bad = {k: v for k, v in errs.items() if not v < 2e-3}
    assert not bad, f"errors above 2e-3: {bad}; all: {errs}"


@pytest.mark.parametrize("rows_shape", [(2, 16, 24), (16, 48, 72)])
def test_layernorm_fold_offset_means(cuda, rows_shape):
    """igemm(ln_fold=): x + LN(x) W^T with the row statistics taken in the GEMM epilogue, on rows with mean / std 0, 4,
    16, 32 and one constant row, against float64 with the same fp16 W * gamma the kernel reads."""
    from cesm_emulator_b200 import kernels as K
    C = 64
    g = torch.Generator(device=cuda).manual_seed(rows_shape[0])
    M = rows_shape[0] * rows_shape[1] * rows_shape[2]
    x = _offset_rows(M, C, g, cuda).view(*rows_shape, C).contiguous()
    gamma = 1.0 + 0.2 * torch.randn(C, device=cuda, generator=g)
    w = torch.randn(C, C, device=cuda, generator=g) * 0.1
    wln = (w * gamma[None, :]).to(H16)
    colsum = wln.float().sum(dim=1)
    y = K.igemm(x, wln, residual=x, ln_fold=(colsum, EPS)).view(M, C)
    xd = x.to(F64).view(M, C)
    ln = _ln64(xd, 1.0) @ wln.to(F64).t()
    ref = xd + ln
    e = _err(y, ref)
    # The residual dominates max|ref| on the offset rows, so also compare the LayerNorm term itself per row class: the
    # error beyond half an fp16 ulp of the output (its unavoidable rounding) against that class's max|LN(x) W^T|.
    yd = y.to(F64)
    half_ulp = torch.ldexp(torch.ones_like(ref), torch.floor(torch.log2(torch.maximum(yd.abs(), ref.abs()).clamp_min(2.0 ** -14))).long() - 11)
    excess = ((yd - ref).abs() - half_ulp).clamp_min(0.0)
    ratio = torch.tensor(RATIOS, device=cuda, dtype=F64)[torch.arange(M, device=cuda) % len(RATIOS)]
    errs = {"y": e}
    for r in RATIOS:
        rows = ratio == r
        rows[M // 2] = False
        errs[f"LN term, mean/std {r:g}"] = excess[rows].max().item() / ln[rows].abs().max().item()
    errs["constant row"] = excess[M // 2].max().item() / ln.abs().max().item()
    print(f"ln_fold offset {rows_shape}: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    bad = {k: v for k, v in errs.items() if not v < 2e-3}
    assert not bad, f"errors above 2e-3: {bad}; all: {errs}"
