"""GPU tests of the weight EMA fused into the optimizer step (cesm_adamw_ema_step, FusedAdamW / TrainEngine
ema_decay, train.py / inference.py): the AdamW part is bit-identical to cesm_adamw_step, the EMA matches torch's
AveragedModel(get_ema_multi_avg_fn) and a float64 recurrence, skipped steps leave it alone, and the engine, the
checkpoints and the entry points carry it."""
import json
import os
import subprocess
import sys

import pytest
import torch

from _parity import BASELINE_KW

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HP = dict(lr=2e-4, betas=(0.9, 0.999), weight_decay=1e-4, eps=1e-8)
EPS32 = float(torch.finfo(torch.float32).eps)


def _opt_state(cuda, lr, wd, scale=1.0, interval=0):
    from cesm_emulator_b200 import kernels as K
    st = torch.zeros(K.OPT_STATE_FLOATS)
    st[K.OPT_LR], st[K.OPT_WD], st[K.OPT_SCALE], st[K.OPT_INTERVAL] = lr, wd, scale, interval
    return st.to(cuda)


def _partials(cuda):
    from cesm_emulator_b200 import _lib
    return torch.zeros(_lib.load().cesm_adamw_partials(), device=cuda)


def _ema64(e64, p, k, decay, start):
    """One step of the EMA recurrence in float64 from fp32 parameters p after optimizer step k."""
    p64 = p.double()
    return p64.clone() if k <= start else e64 + (1.0 - decay) * (p64 - e64)


@pytest.mark.parametrize("n,max_norm,scale", [(10_001, 1.0, 1.0), (4096, None, 65536.0), (1_234_567, 0.05, 1024.0),
                                              (7, 1.0, 512.0), (65_538, None, 1.0)])
def test_ema_step_leaves_adamw_bit_identical(cuda, n, max_norm, scale):
    """On identical inputs the EMA entry point leaves p, m, v and the state vector exactly as cesm_adamw_step does."""
    from cesm_emulator_b200 import kernels as K
    torch.manual_seed(3)
    p0 = torch.randn(n, device=cuda)
    bufs = {}
    for ema in (False, True):
        p, m, v = p0.clone(), torch.zeros(n, device=cuda), torch.zeros(n, device=cuda)
        e = p0.clone()
        state, partials = _opt_state(cuda, HP["lr"], HP["weight_decay"], scale), _partials(cuda)
        g_gen = torch.Generator(device=cuda).manual_seed(11)
        for step in range(4):
            g = torch.randn(n, device=cuda, generator=g_gen) * (0.5 + step) * scale
            if ema:
                K.adamw_ema_step(p, g, m, v, e, partials, state, *HP["betas"], HP["eps"], max_norm, 0.99, 1)
            else:
                K.adamw_step(p, g, m, v, partials, state, *HP["betas"], HP["eps"], max_norm)
        bufs[ema] = (p, m, v, state)
    for a, b in zip(bufs[False], bufs[True]):
        assert torch.equal(a, b)
    assert bufs[True][3][K.OPT_STEP].item() == 4


@pytest.mark.parametrize("n,decay", [(10_001, 0.9), (1_234_567, 0.999)])
def test_ema_matches_averaged_model_and_float64(cuda, n, decay):
    """12 steps at ema_start = 1 with an lr change in the middle: the kernel's EMA against torch's AveragedModel fed the
    kernel's own parameters after each step (a few ulp), against a float64 recurrence over the same trajectory, and end
    to end against torch AdamW + the same AveragedModel (the 2e-6 bar of the AdamW kernel test)."""
    from torch.optim.swa_utils import AveragedModel, get_ema_multi_avg_fn
    from cesm_emulator_b200 import kernels as K
    torch.manual_seed(4)
    p0 = torch.randn(n, device=cuda)
    p, m, v, e = p0.clone(), torch.zeros(n, device=cuda), torch.zeros(n, device=cuda), torch.zeros(n, device=cuda)
    state, partials = _opt_state(cuda, HP["lr"], HP["weight_decay"]), _partials(cuda)
    mine = torch.nn.Module()
    mine.w = torch.nn.Parameter(p0.clone())
    avg_mine = AveragedModel(mine, multi_avg_fn=get_ema_multi_avg_fn(decay))
    ref = torch.nn.Module()
    ref.w = torch.nn.Parameter(p0.clone())
    opt = torch.optim.AdamW([ref.w], **HP)
    avg_ref = AveragedModel(ref, multi_avg_fn=get_ema_multi_avg_fn(decay))
    e64 = None
    for step in range(12):
        g = torch.randn(n, device=cuda) * (0.5 + step % 3)
        ref.w.grad = g.clone()
        torch.nn.utils.clip_grad_norm_([ref.w], 1.0)
        opt.step()
        avg_ref.update_parameters(ref)
        K.adamw_ema_step(p, g, m, v, e, partials, state, *HP["betas"], HP["eps"], 1.0, decay, 1)
        k = step + 1
        assert state[K.OPT_STEP].item() == k
        if k == 1:
            assert torch.equal(e, p)                                    # the copy phase is exact
        mine.w.data.copy_(p)
        avg_mine.update_parameters(mine)
        e64 = _ema64(e64, p, k, decay, 1)
        scale_e = e.abs().max().item()
        assert (e - avg_mine.module.w).abs().max().item() <= 4 * EPS32 * scale_e, step
        assert (e.double() - e64).abs().max().item() <= 16 * EPS32 * scale_e, step
        assert (e - avg_ref.module.w).abs().max().item() < 2e-6, step
        if step == 5:
            for gr in opt.param_groups:
                gr["lr"] = 5e-4
            state[K.OPT_LR] = 5e-4
    assert not torch.equal(e, p)


def test_ema_copy_phase_and_skipped_steps(cuda):
    """Copy while the step count is <= ema_start, decay after.  An overflowing gradient skips the step: the EMA is
    unchanged bit for bit and, as the step count does not advance, the copy/decay boundary moves with it."""
    from cesm_emulator_b200 import kernels as K
    torch.manual_seed(5)
    n, decay, start = 5003, 0.9, 3
    p = torch.randn(n, device=cuda)
    m, v, e = torch.zeros(n, device=cuda), torch.zeros(n, device=cuda), torch.full((n,), 7.0, device=cuda)
    state, partials = _opt_state(cuda, 1e-3, 1e-2, 65536.0, 3), _partials(cuda)
    overflow_at = {2, 6}   # call 2 would have been the last copy step; call 6 is in the decay phase
    k, e64 = 0, None
    for call in range(10):
        S = state[K.OPT_SCALE].item()
        g = torch.randn(n, device=cuda) * 0.1 * S
        if call in overflow_at:
            g[call] = float("inf")
        e_before = e.clone()
        K.adamw_ema_step(p, g, m, v, e, partials, state, *HP["betas"], HP["eps"], 1.0, decay, start)
        if call in overflow_at:
            assert state[K.OPT_FOUND_INF].item() == 1
            assert torch.equal(e, e_before), call
            continue
        k += 1
        assert state[K.OPT_STEP].item() == k
        e64 = _ema64(e64, p, k, decay, start)
        if k <= start:
            assert torch.equal(e, p), (call, k)
        else:
            assert not torch.equal(e, p)
            assert (e.double() - e64).abs().max().item() <= 16 * EPS32 * e.abs().max().item(), (call, k)
    assert state[K.OPT_SKIPPED].item() == 2 and k == 8


def test_ema_abi_rejects_bad_arguments(cuda):
    from cesm_emulator_b200 import _lib, kernels as K
    n = 64
    p, m, v, e = (torch.zeros(n, device=cuda) for _ in range(4))
    state, partials = _opt_state(cuda, 1e-3, 0.0), _partials(cuda)
    args = lambda ema, d, s: (K._ptr(p), K._ptr(p), K._ptr(m), K._ptr(v), ema, n, K._ptr(partials), K._ptr(state),
                              0.9, 0.999, 1e-8, 1.0, d, s, K._stream())
    for ema, d, s in [(K._ptr(e) + 4, 0.9, 0), (None, 0.9, 0), (K._ptr(e), 1.0, 0), (K._ptr(e), -0.5, 0),
                      (K._ptr(e), float("nan"), 0), (K._ptr(e), 0.9, -1)]:
        with pytest.raises(_lib.CesmError):
            _lib.call("cesm_adamw_ema_step", *args(ema, d, s))
    assert state[K.OPT_STEP].item() == 0


def _engine(cuda, **kw):
    from cesm_emulator_b200.engine import TrainEngine
    from cesm_emulator_b200.model import Diffusion, UNet
    torch.manual_seed(0)
    d = Diffusion(UNet(**BASELINE_KW)).to(cuda)
    d.train()
    return d, TrainEngine(d, (1, 1, 32, 32), (1, 1, 3, 32, 32), lr=1e-3, **kw)


def test_engine_ema_matches_float64_of_parameter_snapshots(cuda):
    """A graph-replayed TrainEngine with the EMA on: after 10 steps (2 eager, the capture, replays) ema_state_dict()
    equals the float64 EMA of the parameters snapshotted after every step; the EMA adds no launch."""
    from cesm_emulator_b200 import kernels as K, ops
    decay, start = 0.9, 3
    d, eng = _engine(cuda, ema_decay=decay, ema_start=start)
    g = torch.Generator().manual_seed(6)
    names = {id(p): n[len("model."):] for n, p in d.named_parameters()}
    e64, k = None, 0
    for s in range(10):
        eng.step(torch.randn(1, 1, 32, 32, generator=g), torch.randn(1, 1, 3, 32, 32, generator=g))
        kk = int(eng.opt.state[K.OPT_STEP].item())
        if kk == k:
            continue  # a skipped step: neither the parameters nor the EMA moved
        k = kk
        e64 = _ema64(e64, eng.opt.p, k, decay, start)
    assert eng.graph is not None and k >= 8
    sd = eng.ema_state_dict()
    model_sd = d.model.state_dict()
    assert list(sd) == list(model_sd) and all(sd[n].shape == model_sd[n].shape for n in sd)
    for p in eng.buckets.params:
        o = eng.buckets.offsets[id(p)]
        ref = e64[o:o + p.numel()].view(p.shape)
        got = sd[names[id(p)]]
        assert (got.double() - ref).abs().max().item() <= 16 * EPS32 * max(ref.abs().max().item(), 1e-30), names[id(p)]
        assert not torch.equal(got, p.detach())
    frozen = [n for n, p in d.model.named_parameters() if not p.requires_grad]
    assert frozen and all(torch.equal(sd[n], model_sd[n]) for n in frozen)
    launches_ema = eng.launches_per_step
    # reset / load round trip; strict keys and shapes
    eng.reset_ema()
    assert torch.equal(eng.opt.ema, eng.opt.p)
    eng.load_ema_state_dict(sd)
    assert all(torch.equal(eng.ema_state_dict()[n], sd[n]) for n in sd)
    with pytest.raises(RuntimeError):
        eng.load_ema_state_dict({n: t for n, t in list(sd.items())[1:]})
    bad = dict(sd)
    first = next(iter(bad))
    bad[first] = bad[first].flatten()[:-1]
    with pytest.raises(RuntimeError):
        eng.load_ema_state_dict(bad)
    ops.set_grad_sink(None)
    d0, eng0 = _engine(cuda)
    for s in range(4):
        eng0.step(torch.randn(1, 1, 32, 32, generator=g), torch.randn(1, 1, 3, 32, 32, generator=g))
    assert eng0.graph is not None and eng0.opt.ema is None and not eng0.has_ema
    assert eng0.launches_per_step == launches_ema > 100
    with pytest.raises(RuntimeError):
        eng0.ema_state_dict()
    ops.set_grad_sink(None)


def _small_config(tmp_path):
    cfg = json.load(open(os.path.join(ROOT, "config", "baseline")))
    cfg["dataset"]["crop_hw"] = [32, 32]
    path = str(tmp_path / "baseline_small")
    json.dump(cfg, open(path, "w"))
    return path, cfg


def _run(args):
    env = dict(os.environ, PYTHONPATH=ROOT)
    return subprocess.run([sys.executable, *args], capture_output=True, text=True, cwd=ROOT, env=env, timeout=600)


def test_train_resume_and_inference_with_ema(cuda, tmp_path, capsys):
    import train as train_entry
    from cesm_emulator_b200 import ops
    from cesm_emulator_b200.engine import TrainEngine
    from cesm_emulator_b200.model import Diffusion
    cfg_path, cfg = _small_config(tmp_path)
    run = str(tmp_path / "run")
    sets = ["train.num_epochs=1", "train.max_steps_per_epoch=6", "train.save_every=1", f"train.save_dir={run}",
            "data.synthetic.lat=32", "data.synthetic.lon=48", "data.synthetic.members=2", "data.synthetic.times=8",
            "train.ema_decay=0.5", "train.ema_start=2"]
    r = _run([os.path.join(ROOT, "train.py"), "--config", cfg_path, "--set", *sets])
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    ckpt_path = os.path.join(run, "checkpoints", "final.pt")
    ckpt = torch.load(ckpt_path, map_location="cpu", weights_only=False)
    assert len(ckpt["model"]) == 233 and list(ckpt["ema"]) == list(ckpt["model"])
    assert all(ckpt["ema"][k].shape == v.shape for k, v in ckpt["model"].items())
    unet = train_entry.build_model_from_config(cfg["unet"])
    unet.load_state_dict(ckpt["ema"], strict=True)
    trainable = {n for n, p in unet.named_parameters() if p.requires_grad}
    frozen = [k for k in ckpt["model"] if k not in trainable]
    assert frozen and all(torch.equal(ckpt["ema"][k], ckpt["model"][k]) for k in frozen)
    assert all(not torch.equal(ckpt["ema"][k], ckpt["model"][k]) for k in trainable)

    # resume: an engine with the EMA restores it bit for bit; from a checkpoint without "ema" it restarts from the
    # loaded weights
    def fresh():
        torch.manual_seed(1)
        d = Diffusion(train_entry.build_model_from_config(cfg["unet"])).to(cuda)
        return d, TrainEngine(d, (2, 1, 32, 32), (2, 1, 3, 32, 32), ema_decay=0.5, ema_start=2)
    d, eng = fresh()
    train_entry.load_checkpoint(ckpt_path, d, eng, cuda)
    got = eng.ema_state_dict()
    assert all(torch.equal(got[k].cpu(), ckpt["ema"][k]) for k in ckpt["ema"])
    ops.set_grad_sink(None)
    plain = dict(ckpt)
    del plain["ema"]
    plain_path = str(tmp_path / "plain.pt")
    torch.save(plain, plain_path)
    d, eng = fresh()
    capsys.readouterr()
    train_entry.load_checkpoint(plain_path, d, eng, cuda)
    assert 'no "ema"' in capsys.readouterr().out
    got = eng.ema_state_dict()
    assert all(torch.equal(got[k].cpu(), ckpt["model"][k]) for k in ckpt["model"])
    ops.set_grad_sink(None)

    # inference from the EMA with the DPM-Solver++(2M) chain; --ema on a checkpoint without one is an error
    out = str(tmp_path / "pred.npy")
    base = [os.path.join(ROOT, "inference.py"), "--batch_size", "2", "--members", "2", "--times", "2", "--out", out]
    r = _run([*base, "--ckpt", ckpt_path, "--ema", "--dpm_steps", "2"])
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    import numpy as np
    pred = np.load(out)
    assert pred.shape == (2, 2, 32, 48) and np.isfinite(pred).all()
    r = _run([*base, "--ckpt", plain_path, "--ema", "--dpm_steps", "2"])
    assert r.returncode != 0 and '"ema"' in r.stderr, r.stderr[-2000:]
