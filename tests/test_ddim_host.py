"""CPU tests of the strided DDIM schedule (`model.ddim_schedule`): timesteps, argument checks, and the coefficient
table's update against the DDPM posterior step and against the independent x0-form reference in ddim_oracle.py."""
import pytest
import torch

import ddim_oracle as DO
from oracle import cesm_oracle as O

T = 1000


def _buf():
    return O.diffusion_buffers(T)


def _sched(steps, eta=0.0):
    from cesm_emulator_b200.model import ddim_schedule
    return ddim_schedule(_buf()["alphas_cumprod"], steps, eta)


def _apply(coef, t, x, e, z):
    A, B, S = coef[t]
    return A * x + B * e + S * z


def test_trailing_timesteps():
    taus, coef, next_t = _sched(T)
    assert taus == list(range(999, -1, -1))
    taus, _, _ = _sched(50)
    assert len(taus) == 50 and taus[0] == 999 and taus[-1] == 19
    assert all(a > b for a, b in zip(taus, taus[1:]))
    assert taus == DO.ddim_timesteps(T, 50)
    assert _sched(30)[0][:3] == [999, 965, 932]
    assert _sched(1)[0] == [999]


@pytest.mark.parametrize("steps", [1, 10, 50, 1000])
def test_next_t_chains_the_schedule(steps):
    taus, coef, next_t = _sched(steps, 0.5)
    assert coef.dtype == torch.float32 and coef.shape == (T, 3)
    assert next_t.dtype == torch.int64 and next_t.shape == (T,)
    chain, t = [], taus[0]
    while t >= 0:
        chain.append(t)
        t = int(next_t[t])
    assert chain == taus
    on = torch.zeros(T, dtype=torch.bool)
    on[taus] = True
    assert torch.isfinite(coef[on]).all() and torch.isnan(coef[~on]).all() and (next_t[~on] == -1).all()


@pytest.mark.parametrize("steps,eta", [(0, 0.0), (T + 1, 0.0), (2.5, 0.0), (True, 0.0), (50, -0.1), (50, float("nan"))])
def test_invalid_arguments_raise(steps, eta):
    with pytest.raises(ValueError):
        _sched(steps, eta)


@pytest.mark.parametrize("steps", [1, 10, 50, 1000])
def test_eta_zero_draws_no_noise(steps):
    taus, coef, _ = _sched(steps, 0.0)
    assert (coef[taus, 2] == 0).all()
    # the last step lands on alpha_bar = 1: x_0 = x0-prediction, A = 1 / sqrt(ab_tau), and sigma = 0 for any eta
    ac = _buf()["alphas_cumprod"].double()
    last = taus[-1]
    assert abs(coef[last, 0].item() - (1 / ac[last].sqrt()).item()) < 1e-6 * coef[last, 0].item()
    assert _sched(steps, 1.0)[1][last, 2].item() == 0.0


def test_full_chain_eta_one_is_the_ddpm_step():
    """N = T, eta = 1: the table's update equals p_sample's formula (model.py:176-183) on the Diffusion buffers at
    every timestep, within 1e-5 of max|x| (the coefficients differ from the fp32 buffers' by rounding only)."""
    b = _buf()
    _, coef, _ = _sched(T, 1.0)
    g = torch.Generator().manual_seed(0)
    worst = 0.0
    for t in range(T):
        x, e, z = (torch.randn(4096, generator=g) for _ in range(3))
        ref = b["sqrt_recip_alphas"][t] * (x - b["betas"][t] / b["sqrt_one_minus_alphas_cumprod"][t] * e)
        ref = ref + torch.sqrt(b["posterior_variance"][t]) * z
        worst = max(worst, ((_apply(coef, t, x, e, z) - ref).abs().max() / x.abs().max()).item())
    assert worst < 1e-5, worst


@pytest.mark.parametrize("steps", [10, 50])
@pytest.mark.parametrize("eta", [0.0, 0.5, 1.0])
def test_table_matches_x0_form_reference(steps, eta):
    b = _buf()
    taus, coef, next_t = _sched(steps, eta)
    g = torch.Generator().manual_seed(steps)
    worst = 0.0
    for i, t in enumerate(taus):
        x, e, z = (torch.randn(2, 1, 16, 24, generator=g) for _ in range(3))
        tv = torch.full((2,), t, dtype=torch.long)
        ref = DO.ddim_update(b, x, e, tv, next_t[tv], eta, z)
        worst = max(worst, ((_apply(coef, t, x, e, z) - ref).abs().max() / ref.abs().max()).item())
    assert worst < 1e-5, worst


@pytest.mark.parametrize("steps,eta", [(0, 0.0), (T + 1, 0.0), (50, -0.1)])
def test_sample_engine_rejects_invalid_ddim_arguments(steps, eta):
    from torch import nn
    from cesm_emulator_b200.engine import SampleEngine
    from cesm_emulator_b200.model import Diffusion
    with pytest.raises(ValueError):
        SampleEngine(Diffusion(nn.Linear(1, 1)), (2, 1, 8, 8), ddim_steps=steps, eta=eta)


def test_inference_rejects_steps_with_ddim_steps(monkeypatch):
    import numpy as np
    import inference
    cond = np.zeros((1, 1, 1, 8, 8), dtype=np.float32)
    with pytest.raises(ValueError):
        inference.predict_temperature_from_emissions(None, cond, steps=5, ddim_steps=5)
    monkeypatch.setattr("sys.argv", ["inference.py", "--ckpt", "none.pt", "--steps", "5", "--ddim_steps", "5"])
    with pytest.raises(SystemExit) as e:
        inference._cli()
    assert e.value.code == 2
