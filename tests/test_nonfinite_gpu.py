"""Non-finite values through the training path.  Dynamic loss scaling works only if an fp16 overflow anywhere in the
backward reaches a parameter gradient as inf or NaN, so that the optimizer step skips and halves the scale.

D: one +inf, or one NaN, at a seeded position of a kernel's incoming gradient (or of a forward kernel's input): every
output tensor must contain a non-finite value exactly when the float64 reference on the same inputs does.  Where the
value lands and its sign are not checked, only whether a max reduction, clamp or guard dropped it.

E: the same inside a TrainEngine step: an identity autograd node spliced into the backward of a block writes one inf
into the fp16 gradient arriving there when a device flag is set, so one captured graph replays both poisoned and clean
steps.  A poisoned step must be skipped (parameters, Adam moments and EMA bit-identical, scale halved) and the next clean
one taken; an overflowing loss scale is halved replay by replay until a step fits."""
import pytest
import torch
import torch.nn.functional as F

from test_kernels_gpu import _linattn_ref, _tattn_ref, _tattn_scores, _toeplitz_bias
from test_value_ranges_gpu import _mattn_ref64, _rope

pytestmark = pytest.mark.gpu
H16, F64 = torch.float16, torch.float64
EPS = 1e-5


def _poison(t, kind, seed):
    """A copy of `t` with one inf or NaN at a seeded flat position."""
    t = t.clone()
    i = int(torch.randint(0, t.numel(), (1,), generator=torch.Generator().manual_seed(seed)))
    t.view(-1)[i] = float("inf") if kind == "inf" else float("nan")
    return t


def _rn(g, dev, *shape, scale=1.0, dtype=H16):
    return (torch.randn(*shape, device=dev, generator=g) * scale).to(dtype)


# ---- each case: (kind, seed, dev) -> {name: (got, ref)} ---------------------------------------------------------
def _gn_bwd(kind, seed, dev, poison_fwd=False):
    from cesm_emulator_b200 import kernels as K
    g = torch.Generator(device=dev).manual_seed(seed)
    B, P, C, G = 2, 3 * 16 * 16, 64, 8
    x, dout = _rn(g, dev, B, P, C, scale=2.0), _rn(g, dev, B, P, C)
    if poison_fwd:
        x = _poison(x, kind, seed)
    else:
        dout = _poison(dout, kind, seed)
    gamma, beta = torch.randn(C, device=dev, generator=g) + 1, torch.randn(C, device=dev, generator=g)
    film = torch.randn(B, 2 * C, device=dev, generator=g) * 0.3
    sums = K.gn_stats(x, B, G)
    out = K.gn_apply_fwd(x, sums, gamma, beta, film, None, B, G, EPS)
    xr, gr, br, fr = (t.to(F64).requires_grad_(True) for t in (x, gamma, beta, film))
    y = F.group_norm(xr.transpose(1, 2), G, gr, br, EPS) * (fr[:, :C, None] + 1) + fr[:, C:, None]
    y = F.silu(y).transpose(1, 2)
    if poison_fwd:
        return {"sums": (sums, x.to(F64).sum()), "out": (out, y)}
    dx, dg, db, dfl, dcb = K.gn_bwd(x, dout, sums, gamma, beta, film, B, G, EPS, conv_bias_grad=True)
    gx, gg, gb, gf = torch.autograd.grad(y, [xr, gr, br, fr], dout.to(F64))
    return {"dx": (dx, gx), "dgamma": (dg, gg), "dbeta": (db, gb), "dfilm": (dfl, gf), "dconv_bias": (dcb, gx.sum((0, 1)))}


def _ln(kind, seed, dev, poison_fwd=False):
    from cesm_emulator_b200 import kernels as K
    g = torch.Generator(device=dev).manual_seed(seed)
    M, C = 513, 128
    x, dy, dres = _rn(g, dev, M, C, scale=2.0), _rn(g, dev, M, C), _rn(g, dev, M, C)
    gamma = torch.randn(C, device=dev, generator=g) + 1
    xr, gr = x.to(F64).requires_grad_(True), gamma.to(F64).requires_grad_(True)
    if poison_fwd:
        x = _poison(x, kind, seed)
        xr = x.to(F64)
    mean = xr.mean(-1, keepdim=True)
    y = (xr - mean) / (((xr - mean) ** 2).mean(-1, keepdim=True) + EPS).sqrt() * gr
    if poison_fwd:
        return {"out": (K.ln_fwd(x, gamma, EPS), y)}
    dy = _poison(dy, kind, seed)
    dx, dg = K.ln_bwd(x, gamma, dy, dres, EPS)
    gx, gg = torch.autograd.grad(y, [xr, gr], dy.to(F64))
    return {"dx": (dx, gx + dres.to(F64)), "dgamma": (dg, gg)}


def _tattn(Fr):
    def case(kind, seed, dev, poison_fwd=False):
        from cesm_emulator_b200 import kernels as K
        g = torch.Generator(device=dev).manual_seed(seed)
        B, HW, H, D = 2, 40, 8, 32
        rows = B * Fr * HW
        qkv, dout = _rn(g, dev, rows, 3 * H * D), _rn(g, dev, rows, H * D)
        if poison_fwd:
            qkv = _poison(qkv, kind, seed)
        else:
            dout = _poison(dout, kind, seed)
        torch.manual_seed(seed)
        bias = torch.randn(H, Fr, Fr, device=dev) if Fr <= 4 else _toeplitz_bias(H, Fr, dev)[0]
        freqs, cs, sn = _rope(Fr, D, dev)
        out, lse = K.tattn_fwd(qkv, bias, cs, sn, B, Fr, HW, H, D, D ** -0.5)
        qr, br = qkv.to(F64).requires_grad_(True), bias.to(F64).requires_grad_(True)
        ref = _tattn_ref(qr, br, freqs, B, Fr, HW, H, D)
        if poison_fwd:
            res = {"out": (out, ref)}
            if Fr > 4:
                s = _tattn_scores(qkv.to(F64), bias.to(F64), freqs, B, Fr, HW, H, D)
                res["lse"] = (lse, torch.logsumexp(s, dim=-1))
            return res
        dqkv, dbias = K.tattn_bwd(qkv, bias, cs, sn, out, lse, dout, B, Fr, HW, H, D, D ** -0.5)
        gq, gb = torch.autograd.grad(ref, [qr, br], dout.to(F64))
        return {"dqkv": (dqkv, gq), "dbias": (dbias, gb)}
    return case


def _linattn(kind, seed, dev, poison_fwd=False):
    from cesm_emulator_b200 import kernels as K
    g = torch.Generator(device=dev).manual_seed(seed)
    NI, n, H, D = 3, 24 * 36, 8, 32
    qkv, dout = _rn(g, dev, NI * n, 3 * H * D, scale=1.5), _rn(g, dev, NI * n, H * D)
    if poison_fwd:
        qkv = _poison(qkv, kind, seed)
    else:
        dout = _poison(dout, kind, seed)
    out, ws = K.linattn_fwd(qkv, NI, n, H, D, D ** -0.5)
    qr = qkv.to(F64).requires_grad_(True)
    ref = _linattn_ref(qr, NI, n, H, D)
    if poison_fwd:
        return {"out": (out, ref)}
    dqkv = K.linattn_bwd(qkv, ws, dout, NI, n, H, D, D ** -0.5)
    return {"dqkv": (dqkv, torch.autograd.grad(ref, qr, dout.to(F64))[0])}


def _mattn(kind, seed, dev, poison_fwd=False):
    from cesm_emulator_b200 import kernels as K
    g = torch.Generator(device=dev).manual_seed(seed)
    NI, n, H = 2, 216, 8
    qkv, dout = _rn(g, dev, NI * n, 3 * H * 32), _rn(g, dev, NI * n, H * 32)
    if poison_fwd:
        qkv = _poison(qkv, kind, seed)
    else:
        dout = _poison(dout, kind, seed)
    out, lse = K.mattn_fwd(qkv, NI, n, H, 32, 32 ** -0.5)
    o, lse_ref, grads = _mattn_ref64(qkv, dout, NI, n, H)
    if poison_fwd:
        return {"out": (out, o), "lse": (lse, lse_ref)}
    dqkv = K.mattn_bwd(qkv, out, lse, dout, NI, n, H, 32, 32 ** -0.5)
    return {"dqkv": (dqkv, torch.cat(grads, dim=1))}


def _qkv_bwd(kind, seed, dev):
    from cesm_emulator_b200 import kernels as K
    g = torch.Generator(device=dev).manual_seed(seed)
    rows, cin, cout = 2 * 3 * 32 * 32, 64, 768
    x, w = _rn(g, dev, rows, cin), _rn(g, dev, cout, cin, scale=0.1)
    dy = _poison(_rn(g, dev, rows, cout), kind, seed)
    dx, dw = K.qkv_bwd(dy, x, w.t().contiguous())
    xr, wr = x.to(F64).requires_grad_(True), w.to(F64).requires_grad_(True)
    gx, gw = torch.autograd.grad(xr @ wr.t(), [xr, wr], dy.to(F64))
    return {"dx": (dx, gx), "dw": (dw, gw)}


def _wgrad(ks):
    def case(kind, seed, dev):
        from cesm_emulator_b200 import kernels as K
        g = torch.Generator(device=dev).manual_seed(seed)
        n, h, w, c = 2, 32, 32, 64
        stride = 1 if ks == 3 else 2
        x = _rn(g, dev, n, h, w, c)
        dy = _poison(_rn(g, dev, n, h // stride, w // stride, c, scale=0.1), kind, seed)
        taps = K.TAPS_3x3 if ks == 3 else [(kh - 1, kw - 1) for kh in range(4) for kw in range(4)]
        dw = K.wgrad(x, dy, taps=taps, stride=stride)
        wt = torch.zeros(c, c, ks, ks, device=dev, dtype=F64, requires_grad=True)
        y = F.conv2d(x.to(F64).permute(0, 3, 1, 2), wt, stride=stride, padding=1)
        (gw,) = torch.autograd.grad(y, wt, dy.to(F64).permute(0, 3, 1, 2))
        return {"dw": (dw, gw)}
    return case


def _igemm_dgrad(kind, seed, dev):
    """dx = conv_transpose(dy, W) + r through the implicit GEMM with negated taps and the residual in the epilogue."""
    from cesm_emulator_b200 import kernels as K
    g = torch.Generator(device=dev).manual_seed(seed)
    n, h, w, cin, cout = 2, 24, 36, 64, 128
    wt = _rn(g, dev, cout, cin, 3, 3, scale=0.05)
    dy = _poison(_rn(g, dev, n, h, w, cout), kind, seed)
    r = _rn(g, dev, n, h, w, cin)
    wd = wt.permute(1, 2, 3, 0).reshape(cin, 9 * cout).contiguous()
    dx = K.igemm(dy, wd, taps=[(-a, -b) for a, b in K.TAPS_3x3], residual=r)
    ref = F.conv_transpose2d(dy.to(F64).permute(0, 3, 1, 2), wt.to(F64), padding=1).permute(0, 2, 3, 1) + r.to(F64)
    return {"dx": (dx, ref)}


def _colsum(kind, seed, dev):
    from cesm_emulator_b200 import kernels as K
    g = torch.Generator(device=dev).manual_seed(seed)
    x = _poison(_rn(g, dev, 777, 256), kind, seed)
    return {"colsum": (K.colsum(x), x.to(F64).sum(0))}


def _out_conv_bwd(kind, seed, dev):
    from cesm_emulator_b200 import kernels as K
    g = torch.Generator(device=dev).manual_seed(seed)
    B, Fr, H, W = 2, 3, 16, 24
    a = _rn(g, dev, B * Fr, H, W, 64)
    w = torch.randn(1, 64, 1, 1, 1, device=dev, generator=g) * 0.2
    de = _poison(torch.randn(B, 1, H, W, device=dev, generator=g), kind, seed)
    da, dw, db = K.out_conv_bwd(a, w, de, B, Fr, H, W)
    ar, wr, br = a.to(F64).requires_grad_(True), w.to(F64).requires_grad_(True), torch.zeros(1, device=dev, dtype=F64, requires_grad=True)
    ref = ((ar.view(B, Fr, H, W, 64) * wr.view(64)).sum(-1) + br)[:, Fr // 2][:, None]
    ga, gw, gb = torch.autograd.grad(ref, [ar, wr, br], de.to(F64))
    return {"da": (da, ga), "dw": (dw, gw), "db": (db, gb)}


def _input_conv_wgrad(kind, seed, dev):
    from cesm_emulator_b200 import kernels as K
    g = torch.Generator(device=dev).manual_seed(seed)
    B, Fr, H, W = 2, 3, 20, 36
    x = torch.randn(B, 1, 1, H, W, device=dev, generator=g)
    c = torch.randn(B, 1, Fr, H, W, device=dev, generator=g)
    dy = _poison(_rn(g, dev, B * Fr, H, W, 64), kind, seed)
    dw, db = K.input_conv_wgrad(x, c, dy, B, Fr, H, W, 7)
    wr = torch.zeros(64, 2, 1, 7, 7, device=dev, dtype=F64, requires_grad=True)
    br = torch.zeros(64, device=dev, dtype=F64, requires_grad=True)
    xin = torch.cat([x.expand(-1, -1, Fr, -1, -1), c], dim=1).to(F64)
    ref = F.conv3d(xin, wr, br, padding=(0, 3, 3)).permute(0, 2, 3, 4, 1).reshape(B * Fr, H, W, 64)
    gw, gb = torch.autograd.grad(ref, [wr, br], dy.to(F64))
    return {"dw": (dw, gw), "db": (db, gb)}


def _small_linear_bwd(kind, seed, dev):
    from cesm_emulator_b200 import kernels as K
    g = torch.Generator(device=dev).manual_seed(seed)
    x = torch.randn(4, 256, device=dev, generator=g)
    W = torch.randn(512, 256, device=dev, generator=g) * 0.1
    dy = _poison(torch.randn(4, 512, device=dev, generator=g), kind, seed)
    dx, dW, db = K.small_linear_bwd(x, W, dy, True, True)
    xr, Wr = x.to(F64).requires_grad_(True), W.to(F64).requires_grad_(True)
    br = torch.zeros(512, device=dev, dtype=F64, requires_grad=True)
    gx, gW, gb = torch.autograd.grad(F.linear(F.silu(xr), Wr, br), [xr, Wr, br], dy.to(F64))
    return {"dx": (dx, gx), "dW": (dW, gW), "db": (db, gb)}


def _film_all_bwd(kind, seed, dev):
    from cesm_emulator_b200 import ops
    ops.set_grad_sink(None)
    g = torch.Generator(device=dev).manual_seed(seed)
    B, Kd, Ns = 3, 256, [128, 256, 512]
    t = torch.randn(B, Kd, device=dev, generator=g, requires_grad=True)
    Ws = [(torch.randn(n, Kd, device=dev, generator=g) * 0.05).requires_grad_(True) for n in Ns]
    bs = [torch.randn(n, device=dev, generator=g).requires_grad_(True) for n in Ns]
    outs = ops.FilmAllFn.apply(t, *[p for w, b in zip(Ws, bs) for p in (w, b)])
    gs = [torch.randn(B, n, device=dev, generator=g) for n in Ns]
    gs[1] = _poison(gs[1], kind, seed)
    got = torch.autograd.grad(outs, [t] + Ws + bs, gs)
    leaves = [p.detach().to(F64).requires_grad_(True) for p in [t] + Ws + bs]
    refs = [F.linear(F.silu(leaves[0]), w, b) for w, b in zip(leaves[1:1 + len(Ns)], leaves[1 + len(Ns):])]
    want = torch.autograd.grad(refs, leaves, [x.to(F64) for x in gs])
    names = ["dt"] + [f"dW{i}" for i in range(len(Ns))] + [f"db{i}" for i in range(len(Ns))]
    return {n: (a, b) for n, a, b in zip(names, got, want)}


BACKWARD = {"gn_bwd": _gn_bwd, "ln_bwd": _ln, "tattn_bwd_F3": _tattn(3), "tattn_bwd_F12": _tattn(12),
            "linattn_bwd": _linattn, "mattn_bwd": _mattn, "qkv_bwd": _qkv_bwd, "wgrad_3x3": _wgrad(3),
            "wgrad_4x4_s2": _wgrad(4), "igemm_dgrad": _igemm_dgrad, "colsum": _colsum, "out_conv_bwd": _out_conv_bwd,
            "input_conv_wgrad": _input_conv_wgrad, "small_linear_bwd": _small_linear_bwd, "film_all_bwd": _film_all_bwd}
FORWARD = {"gn_fwd": _gn_bwd, "ln_fwd": _ln, "tattn_fwd_F3": _tattn(3), "tattn_fwd_F12": _tattn(12),
           "linattn_fwd": _linattn, "mattn_fwd": _mattn}


def _check(results, what):
    seen = {}
    for name, (got, ref) in results.items():
        seen[name] = (bool(torch.isfinite(got).all()), bool(torch.isfinite(ref).all()))
    bad = {n: f"kernel all-finite {a}, float64 all-finite {b}" for n, (a, b) in seen.items() if a != b}
    assert not bad, f"{what}: {bad}"
    return seen


@pytest.mark.parametrize("kind", ["inf", "nan"])
@pytest.mark.parametrize("case", list(BACKWARD))
def test_nonfinite_incoming_gradient_reaches_outputs(cuda, case, kind):
    for seed in (1, 2):
        seen = _check(BACKWARD[case](kind, seed, cuda), f"{case} with one {kind} in the incoming gradient (seed {seed})")
        assert not all(b for _, b in seen.values())   # the reference itself saw the poisoned value


@pytest.mark.parametrize("kind", ["inf", "nan"])
@pytest.mark.parametrize("case", list(FORWARD))
def test_nonfinite_forward_input_reaches_outputs(cuda, case, kind):
    for seed in (3, 4):
        seen = _check(FORWARD[case](kind, seed, cuda, poison_fwd=True), f"{case} with one {kind} in its input (seed {seed})")
        assert not all(b for _, b in seen.values())


# ------------------------------------------------------------------------------------------------
# E. overflow detection in the training engine
# ------------------------------------------------------------------------------------------------
def _poison_fn(flag):
    """Identity whose backward writes +inf into element 0 of the arriving gradient while `flag` (device) is non-zero."""
    class Poison(torch.autograd.Function):
        @staticmethod
        def forward(ctx, x):
            return x.view_as(x)

        @staticmethod
        def backward(ctx, dy):
            dy = dy.clone()
            first = dy.view(-1)[:1]
            first.copy_(torch.where(flag > 0, torch.full_like(first, float("inf")), first))
            return dy
    return Poison.apply


def _splice(block, flag):
    orig, poison = block.forward_cl, _poison_fn(flag)
    block.forward_cl = lambda x, B, F, **kw: poison(orig(x, B, F, **kw))


@pytest.mark.parametrize("use_graph", [False, True], ids=["eager", "graph"])
def test_engine_skips_steps_with_an_overflow_inside_the_backward(cuda, use_graph):
    from _parity import BASELINE_KW
    from cesm_emulator_b200 import kernels as K, ops
    from cesm_emulator_b200.engine import TrainEngine
    from cesm_emulator_b200.model import Diffusion, UNet
    ops.set_grad_sink(None)
    torch.manual_seed(0)
    d = Diffusion(UNet(**BASELINE_KW)).to(cuda)
    d.train()
    net = d.model.net
    points = {"level-0 spatial attention": net.downs[0][2], "mid temporal attention": net.mid_temporal_attn,
              "ResnetBlock": net.downs[1][0]}
    flags = {name: torch.zeros((), device=cuda) for name in points}
    for name, blk in points.items():
        _splice(blk, flags[name])
    eng = TrainEngine(d, (2, 1, 32, 32), (2, 1, 3, 32, 32), lr=1e-3, ema_decay=0.9, use_graph=use_graph)
    opt, st = eng.opt, eng.opt.state
    gen = torch.Generator().manual_seed(3)
    x0, cond = torch.randn(2, 1, 32, 32, generator=gen), torch.randn(2, 1, 3, 32, 32, generator=gen)
    for _ in range(3):  # graph mode: two eager warm-up steps, then the capture
        eng.step(x0, cond)
    assert (eng.graph is not None) == use_graph
    st[K.OPT_SCALE] = 1024.0

    def snap():
        torch.cuda.synchronize()
        return [t.clone() for t in (opt.p, opt.m, opt.v, opt.ema)], st.clone()

    for name in points:
        (p0, s0) = snap()
        flags[name].fill_(1.0)
        eng.step(x0, cond)
        bufs, s1 = snap()
        assert s1[K.OPT_FOUND_INF].item() == 1, f"{name}: an inf inside the backward was not detected"
        assert s1[K.OPT_SKIPPED].item() == s0[K.OPT_SKIPPED].item() + 1 and s1[K.OPT_STEP].item() == s0[K.OPT_STEP].item()
        assert s1[K.OPT_SCALE].item() == s0[K.OPT_SCALE].item() / 2, (name, s0[K.OPT_SCALE].item(), s1[K.OPT_SCALE].item())
        for what, a, b in zip(("parameters", "exp_avg", "exp_avg_sq", "ema"), bufs, p0):
            assert torch.equal(a, b), f"{name}: a skipped step changed the {what}"
        flags[name].fill_(0.0)
        eng.step(x0, cond)
        bufs, s2 = snap()
        assert s2[K.OPT_FOUND_INF].item() == 0 and s2[K.OPT_STEP].item() == s1[K.OPT_STEP].item() + 1, name
        assert not torch.equal(bufs[0], p0[0]) and not torch.equal(bufs[3], p0[3]), name

    # a loss scale far beyond fp16 range: every step overflows and halves it until one fits
    st[K.OPT_SCALE] = 2.0 ** 40
    skipped = 0
    while True:
        (p0, s0) = snap()
        eng.step(x0, cond)
        bufs, s1 = snap()
        if s1[K.OPT_STEP].item() != s0[K.OPT_STEP].item():
            break
        skipped += 1
        assert s1[K.OPT_FOUND_INF].item() == 1 and s1[K.OPT_SCALE].item() == s0[K.OPT_SCALE].item() / 2
        assert all(torch.equal(a, b) for a, b in zip(bufs, p0)), "a skipped step changed the optimizer buffers"
        assert skipped < 40
    assert skipped >= 10, skipped          # 2^40 / 2^skipped is the first scale whose backward stays in fp16 range
    assert not torch.equal(bufs[0], p0[0])
    ops.set_grad_sink(None)
