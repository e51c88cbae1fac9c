"""Input gradients and emission saliency on the GPU: the input-convolution data-gradient kernel against float64
conv_transpose2d, the q_sample backward against torch autograd, d loss / d (cond, x0, noise) of the module against
the fp32 oracle with trainable and frozen weights (and which kernels a frozen backward launches), SaliencyEngine
against an eager loop, seeded row / batch invariance, and saliency.py end to end."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from _parity import BASELINE_KW, LOSS_SCALE, make_inputs, rel_err

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# Two evaluations of the same backward differ: its fp32 atomic reductions (GroupNorm and linear-attention sums) add in
# a different order on every run, and the fp16 gradient stream rounds accordingly.  On a B200, two replays of one
# captured saliency graph on the same inputs differed by 1.7e-3 (max-rel) at 2 x 48x72, so comparisons between two
# runs of this backward use REPEAT_BAR rather than 1e-3.
REPEAT_BAR = 3e-3


# ---- kernel 1: input-convolution data gradient -------------------------------------------------------------------
def _dgrad_ref(dy, w, B, F, f0, f1):
    """float64 conv_transpose2d of the same fp16 dy, summed over frames for a broadcast side."""
    n, H, W, C = dy.shape
    d = dy.double().permute(0, 3, 1, 2)
    outs = []
    for p, fp in ((0, f0), (1, f1)):
        r = torch.nn.functional.conv_transpose2d(d, w[:, p:p + 1, 0].double(), padding=w.shape[-1] // 2)
        r = r.view(B, F, H, W)
        if fp == 1 and F > 1:
            r = r.sum(dim=1, keepdim=True)
        outs.append(r.view(B, 1, fp, H, W))
    return outs


@pytest.mark.parametrize("HW", [(24, 40), (48, 72), (23, 37)])
@pytest.mark.parametrize("F,f0,f1", [(1, 1, 1), (3, 1, 3), (3, 3, 1), (3, 3, 3), (3, 1, 1), (8, 1, 8), (8, 8, 8),
                                     (8, 8, 1)])
def test_input_conv_dgrad_matches_conv_transpose(cuda, F, f0, f1, HW):
    from cesm_emulator_b200 import kernels as K
    H, W = HW
    B = 2
    g = torch.Generator().manual_seed(F * 100 + f0 * 10 + f1 + H)
    dy = torch.randn(B * F, H, W, 64, generator=g).half().to(cuda)
    w = (0.05 * torch.randn(64, 2, 1, 7, 7, generator=g)).to(cuda)
    dx, dc = K.input_conv_dgrad(dy, w, B, F, H, W, 7, f0, f1)
    rx, rc = _dgrad_ref(dy, w, B, F, f0, f1)
    assert dx.shape == rx.shape and dc.shape == rc.shape
    assert rel_err(dx, rx) <= 1e-5 and rel_err(dc, rc) <= 1e-5, (rel_err(dx, rx), rel_err(dc, rc))
    # one side only: the same values, the other output not written
    only_c = K.input_conv_dgrad(dy, w, B, F, H, W, 7, f0, f1, need_x=False)
    assert only_c[0] is None and torch.equal(only_c[1], dc)
    only_x = K.input_conv_dgrad(dy, w, B, F, H, W, 7, f0, f1, need_cond=False)
    assert only_x[1] is None and torch.equal(only_x[0], dx)


@pytest.mark.parametrize("F,f0,f1", [(3, 1, 3), (1, 1, 1)])
def test_input_conv_dgrad_accumulate_and_scale(cuda, F, f0, f1):
    from cesm_emulator_b200 import kernels as K
    B, H, W = 3, 48, 72
    g = torch.Generator().manual_seed(7)
    dy = torch.randn(B * F, H, W, 64, generator=g).half().to(cuda)
    w = (0.05 * torch.randn(64, 2, 1, 7, 7, generator=g)).to(cuda)
    rx, rc = _dgrad_ref(dy, w, B, F, f0, f1)
    bx = torch.randn(B, 1, f0, H, W, generator=g).to(cuda)
    bc = torch.randn(B, 1, f1, H, W, generator=g).to(cuda)
    ax, ac = bx.clone(), bc.clone()
    K.input_conv_dgrad(dy, w, B, F, H, W, 7, f0, f1, dx_out=ax, dcond_out=ac, scale=0.375, accumulate=True)
    assert rel_err(ax, bx.double() + 0.375 * rx) <= 1e-5 and rel_err(ac, bc.double() + 0.375 * rc) <= 1e-5
    ox, oc = bx.clone(), bc.clone()  # overwrite mode ignores what was there
    K.input_conv_dgrad(dy, w, B, F, H, W, 7, f0, f1, dx_out=ox, dcond_out=oc, scale=-2.0)
    assert rel_err(ox, -2.0 * rx) <= 1e-5 and rel_err(oc, -2.0 * rc) <= 1e-5


def test_input_conv_dgrad_rejects_bad_calls(cuda):
    from cesm_emulator_b200 import _lib
    dy = torch.zeros(6, 8, 8, 64, dtype=torch.float16, device=cuda)
    w = torch.zeros(64, 2, 1, 7, 7, device=cuda)
    out = torch.zeros(2, 1, 3, 8, 8, device=cuda)
    for args in [(dy.data_ptr(), w.data_ptr(), 0, 0, 1, 3, 2, 3, 8, 8, 7, 64),          # no output
                 (dy.data_ptr(), w.data_ptr(), 0, out.data_ptr(), 1, 2, 2, 3, 8, 8, 7, 64),  # f1 neither 1 nor F
                 (dy.data_ptr(), w.data_ptr(), 0, out.data_ptr(), 1, 3, 2, 3, 8, 8, 5, 64)]:  # 5x5
        with pytest.raises(_lib.CesmError):
            _lib.call("cesm_input_conv_dgrad", *args, 1.0, 0, None)


# ---- kernel 2: q_sample backward ---------------------------------------------------------------------------------
def test_q_sample_backward_matches_autograd(cuda):
    from cesm_emulator_b200.model import Diffusion
    d = Diffusion(torch.nn.Linear(1, 1)).to(cuda)
    g = torch.Generator().manual_seed(3)
    x0 = torch.randn(4, 1, 24, 40, generator=g).to(cuda).requires_grad_()
    noise = torch.randn(4, 1, 24, 40, generator=g).to(cuda).requires_grad_()
    t = torch.tensor([0, 17, 500, 999], device=cuda)
    up = torch.randn(4, 1, 24, 40, generator=g).to(cuda)
    x_t, _ = d.q_sample(x0, t, noise)
    (x_t * up).sum().backward()
    x0r, nr = x0.detach().clone().requires_grad_(), noise.detach().clone().requires_grad_()
    ref = d.sqrt_alphas_cumprod[t].view(-1, 1, 1, 1) * x0r + d.sqrt_one_minus_alphas_cumprod[t].view(-1, 1, 1, 1) * nr
    assert torch.allclose(x_t.detach(), ref.detach(), rtol=1e-6, atol=1e-7)
    (ref * up).sum().backward()
    assert torch.allclose(x0.grad, x0r.grad, rtol=1e-6, atol=0) and torch.allclose(noise.grad, nr.grad, rtol=1e-6, atol=0)
    x0.grad = None  # one side only
    x_t, _ = d.q_sample(x0, t, noise.detach())
    (x_t * up).sum().backward()
    assert torch.allclose(x0.grad, x0r.grad, rtol=1e-6, atol=0)


# ---- model level -------------------------------------------------------------------------------------------------
def _model(cuda, **kw):
    from cesm_emulator_b200.model import Diffusion, UNet
    torch.manual_seed(0)
    unet = UNet(**BASELINE_KW, **kw)
    return Diffusion(unet).to(cuda), dict(BASELINE_KW, **kw)


def _module_input_grads(diffusion, x0, cond, t, noise):
    """d loss / d (cond, x0, noise) through the module, the loss scaled like a training step (fp16 gradients)."""
    x0, cond, noise = (v.detach().clone().requires_grad_() for v in (x0, cond, noise))
    diffusion.zero_grad(set_to_none=True)
    (diffusion.loss(x0, cond, t, noise) * LOSS_SCALE).backward()
    return {k: v.grad / LOSS_SCALE for k, v in (("cond", cond), ("x0", x0), ("noise", noise))}


def _oracle_input_grads(diffusion, kw, x0, cond, t, noise):
    from oracle import cesm_oracle as O
    cfg = O.OracleConfig.from_unet_kwargs(**kw)
    sd = {k: v.detach().float().cpu() for k, v in diffusion.model.state_dict().items()}
    x0, cond, noise = (v.detach().cpu().clone().requires_grad_() for v in (x0, cond, noise))
    loss = O.diffusion_loss(sd, cfg, O.diffusion_buffers(1000), x0, cond, t.cpu(), noise)
    gc, gx, gn = torch.autograd.grad(loss, [cond, x0, noise])
    return {"cond": gc, "x0": gx, "noise": gn}


@pytest.mark.parametrize("HW", [(64, 64), (48, 72)])
def test_input_gradients_match_oracle_trainable_and_frozen(cuda, HW):
    from cesm_emulator_b200 import _lib
    diffusion, kw = _model(cuda)
    trainable = [p for p in diffusion.parameters() if p.requires_grad]  # all but the rotary frequencies
    for seed in (11, 12):
        x0, cond, t, noise = make_inputs(2, 3, *HW, seed=seed, device=cuda)
        ref = _oracle_input_grads(diffusion, kw, x0, cond, t, noise)
        for p in trainable:
            p.requires_grad_(True)
        got = _module_input_grads(diffusion, x0, cond, t, noise)
        errs = {k: rel_err(got[k], ref[k]) for k in ref}
        assert max(errs.values()) <= 1e-2, errs
        # every parameter frozen: the same input gradients, and no weight-gradient kernel in the backward
        diffusion.requires_grad_(False)
        diffusion.zero_grad(set_to_none=True)
        x0f, condf, noisef = (v.detach().clone().requires_grad_() for v in (x0, cond, noise))
        loss = diffusion.loss(x0f, condf, t, noisef) * LOSS_SCALE
        _lib.PROFILER = prof = _lib.KernelProfiler()
        try:
            loss.backward()
        finally:
            _lib.PROFILER = None
        names = set(prof.summary())
        assert names and not [n for n in names if "wgrad" in n or "colsum" in n or "qkv_bwd" in n], sorted(names)
        assert "cesm_input_conv_dgrad" in names and "cesm_q_sample_bwd" in names
        assert rel_err(condf.grad / LOSS_SCALE, got["cond"]) <= REPEAT_BAR
        assert rel_err(x0f.grad / LOSS_SCALE, ref["x0"]) <= 1e-2 and rel_err(noisef.grad / LOSS_SCALE, ref["noise"]) <= 1e-2
        assert all(p.grad is None for p in diffusion.parameters())


@pytest.mark.parametrize("mid_attn,K", [(False, 1), (True, 3), (True, 1)])
def test_input_gradients_one_frame_and_mid_attention(cuda, mid_attn, K):
    """F = 1 is the sampling shape (4-D x_t and cond): with an input that needs grad the temporal attention takes
    the unfused forward / backward instead of the one-frame fold."""
    diffusion, kw = _model(cuda, use_mid_attn=mid_attn)
    diffusion.requires_grad_(False)
    x0, cond, t, noise = make_inputs(2, K, 48, 72, seed=21, device=cuda)
    if K == 1:
        cond = cond[:, :, 0]
    got = _module_input_grads(diffusion, x0, cond, t, noise)
    ref = _oracle_input_grads(diffusion, kw, x0, cond, t, noise)
    assert got["cond"].shape == cond.shape
    errs = {k: rel_err(got[k], ref[k]) for k in ref}
    assert max(errs.values()) <= 1e-2, errs


def test_training_step_launches_unchanged(cuda):
    """A trainable model issues exactly the launches it did before frozen-weight backward existed: the bench
    training step (B = 2, K = 3, 192x288, config/baseline's UNet) captures 438 library launches, as it did at the parent commit."""
    from cesm_emulator_b200 import ops
    from cesm_emulator_b200.engine import TrainEngine
    cfg = json.load(open(os.path.join(ROOT, "config", "baseline")))
    import train as train_entry
    from cesm_emulator_b200.model import Diffusion
    torch.manual_seed(0)
    d = Diffusion(train_entry.build_model_from_config(cfg["unet"])).to(cuda)
    eng = TrainEngine(d, (2, 1, 192, 288), (2, 1, 3, 192, 288))
    g = torch.Generator().manual_seed(0)
    x0, cond = torch.randn(2, 1, 192, 288, generator=g), torch.randn(2, 1, 3, 192, 288, generator=g)
    for _ in range(3):
        eng.step(x0.to(cuda), cond.to(cuda))
    torch.cuda.synchronize()
    ops.set_grad_sink(None)
    assert eng.launches_per_step == TRAIN_STEP_LAUNCHES, eng.launches_per_step


TRAIN_STEP_LAUNCHES = 438


# ---- SaliencyEngine ----------------------------------------------------------------------------------------------
def _eager_saliency(diffusion, x0, cond, ts, noises):
    """The definition: (1/D) sum_d B * d/d cond Diffusion.loss(x0, cond, t_d, eps_d), one eager backward per draw."""
    B = x0.shape[0]
    acc = torch.zeros_like(cond, dtype=torch.float64)
    for t, n in zip(ts, noises):
        c = cond.detach().clone().requires_grad_()
        (diffusion.loss(x0, c, t, n) * LOSS_SCALE).backward()
        acc += c.grad.double() * (B / LOSS_SCALE)
    return acc / len(ts)


@pytest.mark.parametrize("K,use_graph", [(3, True), (1, True), (3, False)])
def test_engine_matches_eager_loop(cuda, K, use_graph):
    from cesm_emulator_b200 import kernels as K_
    from cesm_emulator_b200.engine import SaliencyEngine, saliency_timesteps
    diffusion, _ = _model(cuda)
    diffusion.requires_grad_(False)
    B, H, W, D = 2, 48, 72, 4
    x0, cond, _, _ = make_inputs(B, K, H, W, seed=31, device=cuda)
    if K == 1:
        cond = cond[:, :, 0]
    seed = 99
    eng = SaliencyEngine(diffusion, x0.shape, cond.shape, draws=D, use_graph=use_graph, seed=seed)
    ids = torch.tensor([5, 9])
    s = eng.saliency(x0, cond, field_ids=ids)
    assert s.shape == (B, 1, K, H, W) and eng.launches_per_step > 100
    ts = [torch.full((B,), int(v), device=cuda) for v in saliency_timesteps(1000, D)]
    noises = [K_.field_normal(seed, ids.to(cuda), K_.SALIENCY_DRAW_BASE + d, (B, 1, H, W)) for d in range(D)]
    ref = _eager_saliency(diffusion, x0, cond, ts, noises).view(B, 1, K, H, W)
    assert rel_err(s, ref) <= REPEAT_BAR, rel_err(s, ref)
    s2 = eng.saliency(x0, cond, field_ids=ids)  # a second call starts from zero again
    assert rel_err(s2, s) <= REPEAT_BAR


def test_engine_unseeded_and_explicit_timesteps(cuda):
    from cesm_emulator_b200.engine import SaliencyEngine
    diffusion, _ = _model(cuda)
    diffusion.requires_grad_(False)
    B, H, W = 2, 48, 72
    x0, cond, _, _ = make_inputs(B, 3, H, W, seed=41, device=cuda)
    tt = torch.tensor([[10, 600], [300, 900]])
    eng = SaliencyEngine(diffusion, x0.shape, cond.shape, timesteps=tt)
    torch.manual_seed(5)
    s = eng.saliency(x0, cond)
    assert eng.draws == 2 and torch.isfinite(s).all()
    torch.manual_seed(5)  # the eager draws of the engine come from torch's generator in the same order
    noises = []
    for _ in range(2):
        noises.append(torch.randn(B, 1, H, W, device=cuda))
    ref = _eager_saliency(diffusion, x0, cond, [tt[d].to(cuda) for d in range(2)], noises)
    assert rel_err(s, ref) <= REPEAT_BAR, rel_err(s, ref)


def test_engine_refuses_trainable_weights_and_bad_arguments(cuda):
    from cesm_emulator_b200.engine import SaliencyEngine
    diffusion, _ = _model(cuda)
    with pytest.raises(ValueError, match="requires_grad|require grad"):
        SaliencyEngine(diffusion, (2, 1, 48, 72), (2, 1, 3, 48, 72))
    diffusion.requires_grad_(False)
    for kw in (dict(draws=0), dict(draws=1001), dict(timesteps=torch.tensor([1000])), dict(seed=-1),
               dict(timesteps=torch.zeros(2, 3, dtype=torch.int64))):
        with pytest.raises(ValueError):
            SaliencyEngine(diffusion, (2, 1, 48, 72), (2, 1, 3, 48, 72), **kw)
    eng = SaliencyEngine(diffusion, (2, 1, 48, 72), (2, 1, 3, 48, 72), draws=1)
    with pytest.raises(ValueError):
        eng.saliency(torch.zeros(2, 1, 48, 72, device=cuda), torch.zeros(2, 1, 3, 48, 72, device=cuda), field_ids=[0, 1])


def test_seeded_field_does_not_depend_on_row_or_batch(cuda):
    """The bar of test_seeded_sampling_gpu.py's real-network invariance test: max-rel < 1e-2."""
    from cesm_emulator_b200.engine import SaliencyEngine
    diffusion, _ = _model(cuda)
    diffusion.requires_grad_(False)
    H, W = 48, 72
    x0, cond, _, _ = make_inputs(4, 3, H, W, seed=51, device=cuda)
    seed = 2024
    e4 = SaliencyEngine(diffusion, x0.shape, cond.shape, draws=3, seed=seed)
    s4 = e4.saliency(x0, cond, field_ids=[10, 11, 12, 13])
    perm = [2, 0, 3, 1]
    s4p = e4.saliency(x0[perm], cond[perm], field_ids=[10 + p for p in perm])
    e2 = SaliencyEngine(diffusion, (2, 1, H, W), (2, 1, 3, H, W), draws=3, seed=seed)
    s2 = e2.saliency(x0[2:], cond[2:], field_ids=[12, 13])
    for i, p in enumerate(perm):
        assert rel_err(s4p[i], s4[p]) < 1e-2
    assert rel_err(s2[0], s4[2]) < 1e-2 and rel_err(s2[1], s4[3]) < 1e-2
    # two ids on the same inputs: different noise, clearly different maps
    same = e2.saliency(x0[:1].expand(2, -1, -1, -1), cond[:1].expand(2, -1, -1, -1, -1), field_ids=[1, 2])
    assert rel_err(same[0], same[1]) > 0.1


# ---- saliency.py -------------------------------------------------------------------------------------------------
def _run(args):
    env = dict(os.environ, PYTHONPATH=ROOT)
    return subprocess.run([sys.executable, *args], capture_output=True, text=True, cwd=ROOT, env=env, timeout=600)


def test_saliency_cli_end_to_end(cuda, tmp_path):
    from scipy.io import netcdf_file
    cfg = json.load(open(os.path.join(ROOT, "config", "baseline")))
    cfg["dataset"]["crop_hw"] = [32, 32]
    cfg_path = str(tmp_path / "baseline_small")
    json.dump(cfg, open(cfg_path, "w"))
    run = str(tmp_path / "run")
    sets = ["train.num_epochs=1", "train.max_steps_per_epoch=3", "train.save_every=1", f"train.save_dir={run}",
            "data.synthetic.lat=32", "data.synthetic.lon=48", "data.synthetic.members=2", "data.synthetic.times=8",
            "train.ema_decay=0.5"]
    r = _run([os.path.join(ROOT, "train.py"), "--config", cfg_path, "--set", *sets])
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    ckpt = os.path.join(run, "checkpoints", "final.pt")
    base = [os.path.join(ROOT, "saliency.py"), "--ckpt", ckpt, "--draws", "2", "--batch_size", "3", "--members", "2",
            "--times", "4"]
    npy = str(tmp_path / "sal.npy")
    r = _run([*base, "--seed", "5", "--out", npy])
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    sal = np.load(npy)
    assert sal.shape == (2, 2, 3, 32, 48) and np.isfinite(sal).all() and np.abs(sal).max() > 0
    nc = str(tmp_path / "sal.nc")
    r = _run([*base, "--seed", "5", "--ema", "--out", nc])
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    with netcdf_file(nc, "r", mmap=False) as f:
        v = f.variables["saliency"]
        assert v.dimensions == ("window", "member_id", "frame", "lat", "lon")
        ema_sal = np.array(v[:])
        assert v.ema == 1 and v.draws == 2 and v.seed == b"5"
    assert ema_sal.shape == sal.shape and np.isfinite(ema_sal).all() and not np.array_equal(ema_sal, sal)
    # batch-size invariance with a seed, through the CLI
    npy2 = str(tmp_path / "sal2.npy")
    r = _run([*base[:5], "--batch_size", "2", *base[7:], "--seed", "5", "--out", npy2])
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    assert rel_err(torch.from_numpy(np.load(npy2)), torch.from_numpy(sal)) < 1e-2
