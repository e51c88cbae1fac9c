"""GPU parity of the whole hot path (UNet forward, Diffusion.loss, every parameter gradient,
one-frame inference call, sampling step) against
  (1) outputs of the UNMODIFIED reference stored in tests/golden/baseline_arch_seed0.npz, and
  (2) the fp32 CPU oracle (oracle/cesm_oracle.py, itself pinned to the reference) run on the
      module's own weights with the same inputs.

Tolerances, as max|got-ref|/max|ref| PER TENSOR -- north_star's contract (16-bit activations vs the
fp32 reference: <= 1e-2 on forward outputs and on every gradient tensor; loss within 1 %):
  forward eps, eps_f1, loss : FWD_TOL  = 1e-2   (measured on B200: 0.9-1.2e-3)
  EVERY parameter gradient  : GRAD_TOL = 1e-2   (measured: median 8e-4, worst tensor 2-4e-3)
No tensor is exempted, and every case runs several input seeds (all must pass): the measured values sit
3-10x inside the bars (profiles/r02_parity_matrix.txt), so a pass does not depend on the seed or on the
order in which fp32 atomics happened to land.  Gradients are taken the way the reference takes them under
autocast: scaled loss, unscaled fp32 parameter gradients (_parity.LOSS_SCALE, train.py:862-864).
"""
import numpy as np
import pytest
import torch

from _parity import (BASELINE_KW, load_golden, make_inputs, module_loss_and_grads, oracle_loss_and_grads, rel_err)

pytestmark = pytest.mark.gpu

FWD_TOL = 1e-2
GRAD_TOL = 1e-2
SEEDS = (5, 6, 7)
# (B, K, H, W): config/baseline's training crop, the smoke shape, two tiny grids (deepest level 4x4 / 8x8 pixels)
SHAPES = [(2, 3, 128, 128), (1, 3, 48, 72), (2, 3, 32, 32), (2, 1, 16, 16)]


def _check_against_oracle(diff, unet_kw, B, K, H, W, seed, cuda):
    x0, cond, t, noise = make_inputs(B, K, H, W, seed=seed, device=cuda)
    eps, loss, grads = module_loss_and_grads(diff, x0, cond, t, noise)
    ref_eps, ref_loss, ref_grads = oracle_loss_and_grads(diff.model, unet_kw, x0, cond, t, noise)
    assert rel_err(eps, ref_eps) < FWD_TOL, (seed, rel_err(eps, ref_eps))
    assert abs(loss.item() - ref_loss.item()) < 1e-2 * abs(ref_loss.item())
    assert set(grads) == set(ref_grads)
    errs = {k: rel_err(grads[k], ref_grads[k]) for k in grads}
    worst = max(errs, key=errs.get)
    assert errs[worst] < GRAD_TOL, (seed, worst, errs[worst], float(np.median(list(errs.values()))))
    return rel_err(eps, ref_eps), errs


@pytest.fixture(scope="module")
def baseline(cuda):
    from cesm_emulator_b200.model import Diffusion, UNet
    torch.manual_seed(0)
    unet = UNet(**BASELINE_KW)
    diff = Diffusion(unet, timesteps=1000).to(cuda)
    diff.train()
    return diff


def test_forward_loss_grads_match_reference_golden(cuda, baseline):
    g = load_golden("baseline_arch_seed0.npz")
    x0, cond, t, noise = (torch.from_numpy(g[k]).to(cuda) for k in ("x0", "cond", "t", "noise"))
    x_t, _ = baseline.q_sample(x0, t, noise)
    assert rel_err(x_t, torch.from_numpy(g["x_t"])) < 1e-6
    eps, loss, grads = module_loss_and_grads(baseline, x0, cond, t, noise)
    assert rel_err(eps, torch.from_numpy(g["eps"])) < FWD_TOL
    assert abs(loss.item() - float(g["loss"])) < 1e-2 * abs(float(g["loss"]))
    # the golden file keeps each gradient's norm and first 8 entries
    names = [k[len("gradnorm/"):] for k in g if k.startswith("gradnorm/")]
    assert set(names) == set(grads)
    for k in names:
        ref_norm = float(g["gradnorm/" + k])
        assert abs(grads[k].float().norm().item() - ref_norm) < 1e-2 * ref_norm + 1e-8, k
    # inference-shaped call: 4-D cond, F = 1 (inference.py:221-229)
    baseline.eval()
    with torch.no_grad():
        eps_f1 = baseline.model(x_t, cond[:, :, 1], t)
    baseline.train()
    assert rel_err(eps_f1, torch.from_numpy(g["eps_f1"])) < FWD_TOL


@pytest.mark.parametrize("B,K,H,W", SHAPES)
def test_every_gradient_against_oracle(cuda, baseline, B, K, H, W):
    for seed in SEEDS:
        _check_against_oracle(baseline, BASELINE_KW, B, K, H, W, seed, cuda)


def test_parity_is_reproducible_run_to_run(cuda, baseline):
    """Three runs of the same step: statistics are accumulated with fp32 atomics, so the runs are not bitwise equal
    (a sum that differs in its last bit flips an fp16 rounding somewhere, and the flip spreads), but they must agree
    inside the parity bar so that a pass / fail does not depend on the run (measured: forward 3e-4, worst gradient
    tensor 3e-3 between runs, against 1e-3 / 3e-3 to the oracle)."""
    x0, cond, t, noise = make_inputs(2, 3, 64, 64, seed=5, device=cuda)
    runs = [module_loss_and_grads(baseline, x0, cond, t, noise) for _ in range(3)]
    for eps, loss, grads in runs[1:]:
        assert rel_err(eps, runs[0][0]) < 2e-3
        # worst tensor measured 3-3.6e-3; the bar is the parity bar itself (a race shows as an outlier >> 1e-2)
        assert max(rel_err(grads[k], runs[0][2][k]) for k in grads) < 1e-2


def test_p_sample_step_matches_oracle(cuda, baseline):
    from oracle import cesm_oracle as O
    B, H, W = 2, 32, 32
    x0, cond, t, noise = make_inputs(B, 1, H, W, seed=9, device=cuda)
    cond = cond[:, :, 0]
    t = torch.tensor([0, 617], device=cuda)
    got = baseline.p_sample(x0, cond, t, noise=noise)
    sd = {k: v.detach().float().cpu() for k, v in baseline.model.state_dict().items()}
    cfg = O.OracleConfig.from_unet_kwargs(**BASELINE_KW)
    with torch.no_grad():
        ref = O.p_sample(sd, cfg, O.diffusion_buffers(1000), x0.cpu(), cond.cpu(), t.cpu(), noise.cpu())
    assert rel_err(got, ref) < FWD_TOL


def test_reference_style_module_calls(cuda, baseline):
    """Sub-modules keep the reference's NCDHW call signatures (video_net.py:219, :254, :84)."""
    from oracle import cesm_oracle as O
    net = baseline.model.net
    sd = {k: v.detach().float().cpu() for k, v in net.state_dict().items()}
    torch.manual_seed(1)
    x = torch.randn(2, 64, 3, 16, 16, device=cuda)
    temb = torch.randn(2, 256, device=cuda)
    blk = net.downs[0][0]
    with torch.no_grad():
        got = blk(x, temb)
        ref = O.resnet_block(sd, "downs.0.0.", x.cpu(), temb.cpu(), 8)
        assert rel_err(got, ref) < 3e-3
        got = net.downs[0][2](x)
        ref = O.spatial_attention_block(sd, "downs.0.2.", x.cpu(), 8)
        assert rel_err(got, ref) < 3e-3
        pb = net.time_rel_pos_bias(3, device=cuda)
        got = net.downs[0][3](x, pos_bias=pb)
        ref = O.temporal_attention_block(sd, "downs.0.3.", x.cpu(), 8, pb.cpu())
        assert rel_err(got, ref) < 3e-3
        got = net.downs[0][4](x)
        ref = torch.nn.functional.conv3d(x.cpu(), sd["downs.0.4.weight"], sd["downs.0.4.bias"], stride=(1, 2, 2),
                                         padding=(0, 1, 1))
        assert rel_err(got, ref) < 3e-3
        full = net(x[:, :1], torch.tensor([3, 900], device=cuda), cond_map=x[:, 1:2])
        cfg = O.OracleConfig.from_unet_kwargs(**BASELINE_KW)
        ref = O.unet3d_forward({"net." + k: v for k, v in sd.items()}, cfg, x[:, :1].cpu(), torch.tensor([3, 900]),
                               x[:, 1:2].cpu())
        assert full.shape == ref.shape and rel_err(full, ref) < FWD_TOL


def _fresh(cuda, unet_kw):
    from cesm_emulator_b200 import ops
    from cesm_emulator_b200.model import Diffusion, UNet
    ops.set_grad_sink(None)
    torch.manual_seed(0)
    diff = Diffusion(UNet(**unet_kw), timesteps=1000).to(cuda)
    diff.train()
    return diff


def test_more_blocks_architecture_against_oracle(cuda):
    """config/more_blocks: ch_mults [1,2,4,8] -> a fourth level with 512 channels (and the level-0
    temporal attention going through `temporal_op`, video_net.py:701), at its configured 64x64 crop."""
    kw = dict(in_channels=2, out_channels=1, base_ch=64, ch_mults=(1, 2, 4, 8), num_res_blocks=6, time_dim=124,
              groups=8, dropout=0.0, use_checkpoint=True)
    diff = _fresh(cuda, kw)
    for seed in (8, 9):
        _check_against_oracle(diff, kw, 2, 3, 64, 64, seed, cuda)


def test_long_window_temporal_attention_against_oracle(cuda):
    """BASELINE.json configs[4]: a longer condition window (K = 12 frames > 4 selects the streaming
    online-softmax temporal-attention kernels and the log-bucketed part of the relative-position table)."""
    diff = _fresh(cuda, BASELINE_KW)
    for seed in (8, 9):
        _check_against_oracle(diff, BASELINE_KW, 1, 12, 16, 16, seed, cuda)
