"""GPU tests of use_mid_attn=True: the flash softmax attention kernels over the bottleneck pixels
(csrc/mid_attn.cu) against fp32 torch on the same fp16 inputs, and the whole model / engines with the block
switched on against the fp32 CPU oracle (same bars as test_model_gpu.py: forward and EVERY gradient tensor
within 1e-2 of the oracle, loss within 1 %)."""
import numpy as np
import pytest
import torch

from _parity import BASELINE_KW, LOSS_SCALE, make_inputs, module_loss_and_grads, oracle_loss_and_grads, rel_err

pytestmark = pytest.mark.gpu

MID_KW = dict(BASELINE_KW, use_mid_attn=True)
FWD_TOL = 1e-2
GRAD_TOL = 1e-2
SEEDS = (5, 6, 7)
SHAPES = [(2, 3, 128, 128), (1, 3, 48, 72), (2, 3, 32, 32), (2, 1, 16, 16)]
# (NI, n, heads): the config/baseline crop, the bench step, 48x72 / 16x16 / 20x36 bottleneck tails, ch_mults=(1, 2)
CORE_SHAPES = [(6, 1024, 8), (6, 3456, 8), (2, 216, 8), (1, 16, 8), (3, 45, 4), (1, 13824, 8)]


def _core_ref(qkv, dout, NI, n, H):
    """fp32 torch on the same fp16 inputs -> (o, lse, dqkv) in the kernels' layouts."""
    t = qkv.float().view(NI, n, 3, H, 32).permute(2, 0, 3, 1, 4)   # [3, NI, H, n, 32]
    q, k, v = (t[i].clone().requires_grad_(True) for i in range(3))
    s = (q * 32 ** -0.5) @ k.transpose(-1, -2)
    lse = torch.logsumexp(s, dim=-1)
    o = torch.softmax(s, dim=-1) @ v
    do = dout.float().view(NI, n, H, 32).permute(0, 2, 1, 3)
    o.backward(do)
    o_l = o.detach().permute(0, 2, 1, 3).reshape(NI * n, H * 32)
    lse_l = lse.detach().permute(0, 2, 1).reshape(NI * n, H)
    grads = [g.permute(0, 2, 1, 3).reshape(NI * n, H * 32) for g in (q.grad, k.grad, v.grad)]
    return o_l, lse_l, grads


@pytest.mark.parametrize("NI,n,H", CORE_SHAPES)
def test_core_matches_fp32_torch(cuda, NI, n, H):
    from cesm_emulator_b200 import kernels as K
    g = torch.Generator(device=cuda).manual_seed(n + H)
    qkv = torch.randn(NI * n, 3 * H * 32, device=cuda, generator=g).half()
    dout = torch.randn(NI * n, H * 32, device=cuda, generator=g).half()
    out, lse = K.mattn_fwd(qkv, NI, n, H, 32, 32 ** -0.5)
    dqkv = K.mattn_bwd(qkv, out, lse, dout, NI, n, H, 32, 32 ** -0.5)
    o_r, lse_r, (dq_r, dk_r, dv_r) = _core_ref(qkv, dout, NI, n, H)
    hid = H * 32
    errs = {"o": rel_err(out, o_r), "lse": rel_err(lse, lse_r), "dq": rel_err(dqkv[:, :hid], dq_r),
            "dk": rel_err(dqkv[:, hid:2 * hid], dk_r), "dv": rel_err(dqkv[:, 2 * hid:], dv_r)}
    assert errs["o"] < 2e-3 and errs["lse"] < 2e-3, errs
    assert max(errs["dq"], errs["dk"], errs["dv"]) < 3e-3, errs
    assert torch.isfinite(dqkv).all()


def test_backward_is_bitwise_deterministic(cuda):
    from cesm_emulator_b200 import kernels as K
    NI, n, H = 2, 3456, 8
    g = torch.Generator(device=cuda).manual_seed(1)
    qkv = torch.randn(NI * n, 3 * H * 32, device=cuda, generator=g).half()
    dout = torch.randn(NI * n, H * 32, device=cuda, generator=g).half()
    out, lse = K.mattn_fwd(qkv, NI, n, H, 32, 32 ** -0.5)
    a = K.mattn_bwd(qkv, out, lse, dout, NI, n, H, 32, 32 ** -0.5)
    b = K.mattn_bwd(qkv, out, lse, dout, NI, n, H, 32, 32 ** -0.5)
    assert torch.equal(a, b)


def test_c_abi_rejects_other_head_dims(cuda):
    from cesm_emulator_b200 import _lib
    from cesm_emulator_b200 import kernels as K
    qkv = torch.zeros(64, 3 * 8 * 64, dtype=torch.float16, device=cuda)
    with pytest.raises(_lib.CesmError, match="dim_head == 32"):
        K.mattn_fwd(qkv, 1, 64, 8, 64, 64 ** -0.5)
    out, lse = torch.zeros(64, 512, dtype=torch.float16, device=cuda), torch.zeros(64, 8, device=cuda)
    with pytest.raises(_lib.CesmError, match="dim_head == 32"):
        K.mattn_bwd(qkv, out, lse, out, 1, 64, 8, 64, 64 ** -0.5)


def _fresh(cuda, kw):
    from cesm_emulator_b200 import ops
    from cesm_emulator_b200.model import Diffusion, UNet
    ops.set_grad_sink(None)
    torch.manual_seed(0)
    diff = Diffusion(UNet(**kw), timesteps=1000).to(cuda)
    diff.train()
    return diff


def _check_against_oracle(diff, kw, B, K, H, W, seed, cuda):
    x0, cond, t, noise = make_inputs(B, K, H, W, seed=seed, device=cuda)
    eps, loss, grads = module_loss_and_grads(diff, x0, cond, t, noise)
    ref_eps, ref_loss, ref_grads = oracle_loss_and_grads(diff.model, kw, x0, cond, t, noise)
    assert rel_err(eps, ref_eps) < FWD_TOL, (seed, rel_err(eps, ref_eps))
    assert abs(loss.item() - ref_loss.item()) < 1e-2 * abs(ref_loss.item())
    assert set(grads) == set(ref_grads)
    assert {k for k in grads if "mid_spatial_attn" in k} == {
        "net.mid_spatial_attn.fn.norm.gamma", "net.mid_spatial_attn.fn.fn.fn.to_qkv.weight",
        "net.mid_spatial_attn.fn.fn.fn.to_out.weight"}
    errs = {k: rel_err(grads[k], ref_grads[k]) for k in grads}
    worst = max(errs, key=errs.get)
    assert errs[worst] < GRAD_TOL, (seed, worst, errs[worst], float(np.median(list(errs.values()))))


@pytest.fixture(scope="module")
def mid(cuda):
    return _fresh(cuda, MID_KW)


@pytest.mark.parametrize("B,K,H,W", SHAPES)
def test_every_gradient_against_oracle(cuda, mid, B, K, H, W):
    for seed in SEEDS:
        _check_against_oracle(mid, MID_KW, B, K, H, W, seed, cuda)


def test_more_blocks_with_mid_attention_against_oracle(cuda):
    kw = dict(in_channels=2, out_channels=1, base_ch=64, ch_mults=(1, 2, 4, 8), num_res_blocks=6, time_dim=124,
              groups=8, dropout=0.0, use_checkpoint=True, use_mid_attn=True)
    diff = _fresh(cuda, kw)
    _check_against_oracle(diff, kw, 2, 3, 64, 64, 8, cuda)


def test_inference_calls_against_oracle(cuda, mid):
    """The one-frame call (every step of the sampling chain: the mid block runs the full attention), p_sample, and
    the reference-style NCDHW / [b, f, n, c] module calls."""
    from oracle import cesm_oracle as O
    sd = {k: v.detach().float().cpu() for k, v in mid.model.state_dict().items()}
    cfg, buf = O.OracleConfig.from_unet_kwargs(**MID_KW), O.diffusion_buffers(1000)
    x0, cond, t, noise = make_inputs(2, 1, 48, 72, seed=11, device=cuda)
    mid.eval()
    try:
        with torch.no_grad():
            got = mid.model(x0, cond, t)
            ref = O.unet_forward(sd, cfg, x0.cpu(), cond.cpu(), t.cpu())
            assert rel_err(got, ref) < FWD_TOL, rel_err(got, ref)
            c4, tt = cond[:, :, 0], torch.tensor([0, 617], device=cuda)
            got = mid.p_sample(x0, c4, tt, noise=noise)
            ref = O.p_sample(sd, cfg, buf, x0.cpu(), c4.cpu(), tt.cpu(), noise.cpu())
            assert rel_err(got, ref) < FWD_TOL, rel_err(got, ref)
            net = mid.model.net
            nsd = {k[len("net."):]: v for k, v in sd.items() if k.startswith("net.")}
            torch.manual_seed(2)
            x = torch.randn(2, 256, 3, 12, 18, device=cuda)
            got = net.mid_spatial_attn(x)
            ref = O.mid_spatial_attention_block(nsd, "mid_spatial_attn.", x.cpu(), 8)
            assert got.shape == x.shape and rel_err(got, ref) < 3e-3, rel_err(got, ref)
            xb = torch.randn(2, 3, 216, 256, device=cuda)          # [b, f, (h w), c]
            got = net.mid_spatial_attn.fn.fn.fn(xb)
            ref = O.attention(nsd, "mid_spatial_attn.fn.fn.fn.", xb.cpu(), 8, None, rotary=False)
            assert got.shape == xb.shape and rel_err(got, ref) < 3e-3, rel_err(got, ref)
    finally:
        mid.train()


def test_train_engine_gradients_and_graph_replay(cuda):
    """TrainEngine (flat gradient buffer, direct delivery, side stream) with the block on: eager engine gradients
    against plain autograd and the oracle, then graph replay against eager over 5 steps."""
    from cesm_emulator_b200 import ops
    from cesm_emulator_b200.engine import TrainEngine
    B, K, H, W = 2, 3, 32, 48
    d = _fresh(cuda, MID_KW)
    g = torch.Generator().manual_seed(3)
    x0, cond = torch.randn(B, 1, H, W, generator=g).to(cuda), torch.randn(B, 1, K, H, W, generator=g).to(cuda)
    t, noise = torch.tensor([100, 700], device=cuda), torch.randn(B, 1, H, W, generator=g).to(cuda)
    d.zero_grad(set_to_none=True)
    loss_ref = d.loss(x0, cond, t=t, noise=noise)
    (loss_ref * LOSS_SCALE).backward()
    ref = {k: p.grad / LOSS_SCALE for k, p in d.named_parameters() if p.grad is not None}
    _, loss_o, og = oracle_loss_and_grads(d.model, MID_KW, x0, cond, t, noise)
    og = {"model." + k: v for k, v in og.items()}
    eng = TrainEngine(d, (B, 1, H, W), (B, 1, K, H, W), lr=0.0, weight_decay=0.0, max_grad_norm=None, use_graph=False)
    plain_loss = d.loss
    d.loss = lambda x, c: plain_loss(x, c, t=t, noise=noise)
    for rep in range(2):
        loss = eng.step(x0, cond)
        assert abs(loss.item() - loss_ref.item()) < 1e-3 * abs(loss_ref.item()), (loss.item(), loss_ref.item())
        assert abs(loss.item() - loss_o.item()) < 1e-2 * abs(loss_o.item())
        got = {k: p.grad / LOSS_SCALE for k, p in d.named_parameters() if p.requires_grad}
        assert set(got) == set(ref) == set(og)
        vs_auto = np.array([rel_err(got[k], ref[k]) for k in ref])
        vs_orac = np.array([rel_err(got[k], og[k]) for k in ref])
        assert np.median(vs_auto) < 1.5e-3 and vs_auto.max() < 1e-2, (rep, np.median(vs_auto), vs_auto.max())
        assert vs_orac.max() < 1e-2, (rep, np.median(vs_orac), vs_orac.max())
    del d.loss
    ops.set_grad_sink(None)

    B, K, H, W = 1, 3, 32, 32
    g = torch.Generator().manual_seed(5)
    batches = [(torch.randn(B, 1, H, W, generator=g), torch.randn(B, 1, K, H, W, generator=g)) for _ in range(5)]
    losses = {}
    for use_graph in (False, True):
        d = _fresh(cuda, MID_KW)
        eng = TrainEngine(d, (B, 1, H, W), (B, 1, K, H, W), use_graph=use_graph)
        torch.manual_seed(77)
        losses[use_graph] = [eng.step(x0, c).item() for x0, c in batches]
        if use_graph:
            assert eng.graph is not None
        ops.set_grad_sink(None)
    for a, b in zip(losses[False], losses[True]):
        assert abs(a - b) < 5e-3 * abs(a), (losses[False], losses[True])


def test_sample_engine_against_oracle_chain(cuda):
    from oracle import cesm_oracle as O
    from cesm_emulator_b200.engine import SampleEngine
    d = _fresh(cuda, MID_KW)
    d.eval()
    eng = SampleEngine(d, (2, 1, 32, 32))
    cond = torch.randn(2, 1, 32, 32, device=cuda)
    eng.sample(cond, steps=2)
    assert eng.graph is not None
    sd = {k: v.detach().float().cpu() for k, v in d.model.state_dict().items()}
    cfg, buf = O.OracleConfig.from_unet_kwargs(**MID_KW), O.diffusion_buffers(1000)
    torch.manual_seed(9)
    x = torch.randn(2, 1, 32, 32, device=cuda)
    t = torch.tensor([500, 37], device=cuda, dtype=torch.long)
    eng.x.copy_(x); eng.cond.copy_(cond); eng.t.copy_(t)
    eng.step()
    with torch.no_grad():
        ref = O.p_sample(sd, cfg, buf, x.cpu(), cond.cpu(), t.cpu(), eng.z.cpu())
    assert rel_err(eng.x, ref) < 1e-2, rel_err(eng.x, ref)
    eng.x.copy_(x); eng.t.fill_(5)
    xs = x.cpu().clone()
    for tt in range(5, -1, -1):
        eng.step()
        with torch.no_grad():
            xs = O.p_sample(sd, cfg, buf, xs, cond.cpu(), torch.full((2,), tt, dtype=torch.long), eng.z.cpu())
    assert rel_err(eng.x, xs) < 1e-2, rel_err(eng.x, xs)


def test_weights_stay_fresh_across_train_sample_train(cuda):
    """Graph-replayed optimizer steps rewrite the weights behind torch's back; the mid block's packed operands must
    follow, for the eager module call and for a SampleEngine graph captured before the second round of training."""
    from cesm_emulator_b200 import ops
    from cesm_emulator_b200.engine import SampleEngine, TrainEngine
    from cesm_emulator_b200.model import Diffusion, UNet
    B, K, H, W = 1, 3, 32, 32
    kw = dict(MID_KW, ch_mults=(1, 2))
    torch.manual_seed(0)
    d = Diffusion(UNet(**kw)).to(cuda)
    eng = TrainEngine(d, (B, 1, H, W), (B, 1, K, H, W), lr=1e-2)
    g = torch.Generator().manual_seed(1)
    x = torch.randn(2, 1, H, W, generator=g).to(cuda)
    c = torch.randn(2, 1, H, W, generator=g).to(cuda)
    t = torch.tensor([400, 3], device=cuda)
    samp = None

    def fresh_eps():
        torch.manual_seed(0)
        f = Diffusion(UNet(**kw)).to(cuda)
        f.load_state_dict(d.state_dict())
        f.eval()
        with torch.no_grad():
            return f.model(x, c, t)

    outs = []
    for rnd in range(2):
        d.train()
        for _ in range(4):
            eng.step(torch.randn(B, 1, H, W, generator=g), torch.randn(B, 1, K, H, W, generator=g))
        assert eng.graph is not None
        d.eval()
        with torch.no_grad():
            got = d.model(x, c, t)
        assert rel_err(got, fresh_eps()) < 1e-2, rnd
        outs.append(got)
        if samp is None:
            samp = SampleEngine(d, (2, 1, H, W))
            samp.sample(c, steps=2)
        samp.refresh_operands()
        samp.x.copy_(x); samp.cond.copy_(c); samp.t.copy_(t)
        samp.step()
        with torch.no_grad():
            y_ref = d.p_sample(x, c, t, noise=samp.z)
        assert rel_err(samp.x, y_ref) < 1e-2, (rnd, rel_err(samp.x, y_ref))
    assert rel_err(outs[1], outs[0]) > 5e-2
    ops.set_grad_sink(None)
