"""CPU tests of the DPM-Solver++(2M) schedule (`model.dpm_schedule`): timesteps, argument checks, its first-order end
rows against DDIM eta = 0, the table-driven chain against the independent reference in dpm_oracle.py, and its
convergence on an exact Gaussian eps-predictor against the closed-form probability-flow ODE solution."""
import numpy as np
import pytest
import torch

import dpm_oracle as PO
from oracle import cesm_oracle as O

T = 1000


def _ac():
    return O.diffusion_buffers(T)["alphas_cumprod"]


def _sched(steps):
    from cesm_emulator_b200.model import dpm_schedule
    return dpm_schedule(_ac(), steps)


def _ddim(steps):
    from cesm_emulator_b200.model import ddim_schedule
    return ddim_schedule(_ac(), steps, 0.0)


def _apply(coef, t, x, e, hist):
    """The kernel's arithmetic on one row: returns (out, x0); hist is not read where K1 == 0."""
    P, Q, R, K0, K1 = coef[t].to(x.dtype)
    x0 = P * x + Q * e
    out = R * x + K0 * x0
    if K1 != 0:
        out = out + K1 * hist
    return out, x0


@pytest.mark.parametrize("steps", [1, 30, 50, 1000])
def test_timesteps_and_next_t_match_ddim(steps):
    taus, coef, next_t = _sched(steps)
    d_taus, _, d_next = _ddim(steps)
    assert taus == d_taus == PO.dpm_timesteps(T, steps)
    assert torch.equal(next_t, d_next)
    assert coef.dtype == torch.float32 and coef.shape == (T, 5)
    assert next_t.dtype == torch.int64 and next_t.shape == (T,)
    chain, t = [], taus[0]
    while t >= 0:
        chain.append(t)
        t = int(next_t[t])
    assert chain == taus
    on = torch.zeros(T, dtype=torch.bool)
    on[taus] = True
    assert torch.isfinite(coef[on]).all() and torch.isnan(coef[~on]).all() and (next_t[~on] == -1).all()


@pytest.mark.parametrize("steps", [0, T + 1, -3, 2.5, True, "10", None])
def test_invalid_arguments_raise(steps):
    with pytest.raises(ValueError):
        _sched(steps)


@pytest.mark.parametrize("steps", [3, 10, 50, 1000])
def test_first_and_last_rows_are_ddim_eta_zero_steps(steps):
    """R + K0 P = sqrt(ab_p / ab_s) and K0 Q = sigma_p - alpha_p sigma_s / alpha_s on the first and the last row
    (K1 = 0 there); every row in between is second order (K1 != 0)."""
    taus, coef, _ = _sched(steps)
    _, d, _ = _ddim(steps)
    c = coef.double()
    for t in (taus[0], taus[-1]):
        P, Q, R, K0, K1 = c[t]
        assert K1 == 0
        assert abs((R + K0 * P) - d[t, 0]) <= 1e-6 * abs(d[t, 0]), t
        assert abs(K0 * Q - d[t, 1]) <= 1e-6 * abs(d[t, 1]), t
    assert c[taus[-1], 2] == 0 and c[taus[-1], 3] == 1
    assert (c[taus[1:-1], 4] != 0).all()


@pytest.mark.parametrize("steps", [1, 2])
def test_one_and_two_step_chains_are_ddim(steps):
    taus, coef, _ = _sched(steps)
    _, d, _ = _ddim(steps)
    g = torch.Generator().manual_seed(steps)
    x = torch.randn(4096, generator=g)
    y, hist = x.clone(), torch.full_like(x, float("nan"))
    for t in taus:
        e = torch.randn(4096, generator=g)
        x, hist = _apply(coef, t, x, e, hist)
        A, B, _ = d[t]
        y = A * y + B * e
    assert torch.isfinite(x).all()
    assert ((x - y).abs().max() / y.abs().max()).item() < 1e-6


@pytest.mark.parametrize("steps", [10, 50])
def test_table_chain_matches_paper_form_reference(steps):
    """Random x / eps fed at every step, each side carrying its own x0 history, at a vector of per-sample t."""
    buf = O.diffusion_buffers(T)
    taus, coef, _ = _sched(steps)
    g = torch.Generator().manual_seed(steps)
    hist = torch.full((2, 1, 16, 24), float("nan"))
    ref_prev = None
    worst = worst_x0 = 0.0
    for t in taus:
        x, e = (torch.randn(2, 1, 16, 24, generator=g) for _ in range(2))
        out, hist_new = _apply(coef, t, x, e, hist)
        ref, ref_x0 = PO.dpm_update(buf, x, e, torch.full((2,), t, dtype=torch.long), steps, ref_prev)
        worst = max(worst, ((out - ref).abs().max() / ref.abs().max()).item())
        worst_x0 = max(worst_x0, ((hist_new - ref_x0).abs().max() / ref_x0.abs().max()).item())
        hist, ref_prev = hist_new, ref_x0
    assert worst < 1e-4, worst
    assert worst_x0 < 1e-6, worst_x0


def _gauss_chain(coef, taus, x, s):
    """float64 chain on the exact eps-predictor of data ~ N(0, s^2), eps*(x, t) = sqrt(1 - ab_t) x / (ab_t s^2 + 1 - ab_t),
    applying fp32 table rows (3 columns: DDIM, 5 columns: 2M)."""
    ac = _ac().double()
    hist = torch.full_like(x, float("nan"))
    for t in taus:
        a = ac[t]
        e = torch.sqrt(1 - a) * x / (a * s * s + 1 - a)
        if coef.shape[1] == 3:
            A, B, _ = coef[t].double()
            x = A * x + B * e
        else:
            x, hist = _apply(coef, t, x, e, hist)
    return x


def _gauss_err(kind, steps, s=2.0):
    """Max error over max |exact| against the closed-form ODE map x_0 = x_T s / sqrt(ab_{T-1} s^2 + 1 - ab_{T-1})."""
    taus, coef, _ = _sched(steps) if kind == "dpm" else _ddim(steps)
    x_T = torch.randn(4096, generator=torch.Generator().manual_seed(0), dtype=torch.float64)
    a = _ac().double()[T - 1]
    exact = x_T * s / torch.sqrt(a * s * s + 1 - a)
    return ((_gauss_chain(coef, taus, x_T, s) - exact).abs().max() / exact.abs().max()).item()


def test_second_order_on_exact_gaussian_predictor():
    assert _gauss_err("dpm", 10) < 1e-2 < 1e-1 < _gauss_err("ddim", 10)
    dpm = _gauss_err("dpm", 100) / _gauss_err("dpm", 50)
    ddim = _gauss_err("ddim", 100) / _gauss_err("ddim", 50)
    assert dpm < 0.35, dpm         # second order: 0.29
    assert ddim > 0.45, ddim       # first order: 0.50


@pytest.mark.parametrize("kw", [dict(dpm_steps=0), dict(dpm_steps=T + 1), dict(dpm_steps=10, ddim_steps=10),
                                dict(dpm_steps=10, eta=0.5)])
def test_sample_engine_rejects_invalid_dpm_arguments(kw):
    from torch import nn
    from cesm_emulator_b200.engine import SampleEngine
    from cesm_emulator_b200.model import Diffusion
    with pytest.raises(ValueError):
        SampleEngine(Diffusion(nn.Linear(1, 1)), (2, 1, 8, 8), **kw)


@pytest.mark.parametrize("kw,argv", [
    (dict(steps=5, dpm_steps=5), ["--steps", "5", "--dpm_steps", "5"]),
    (dict(ddim_steps=5, dpm_steps=5), ["--ddim_steps", "5", "--dpm_steps", "5"]),
    (dict(eta=0.5, dpm_steps=5), ["--eta", "0.5", "--dpm_steps", "5"]),
])
def test_inference_rejects_dpm_steps_combinations(monkeypatch, kw, argv):
    import inference
    cond = np.zeros((1, 1, 1, 8, 8), dtype=np.float32)
    with pytest.raises(ValueError):
        inference.predict_temperature_from_emissions(None, cond, **kw)
    monkeypatch.setattr("sys.argv", ["inference.py", "--ckpt", "none.pt", *argv])
    with pytest.raises(SystemExit) as e:
        inference._cli()
    assert e.value.code == 2
