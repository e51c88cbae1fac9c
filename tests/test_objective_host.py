"""CPU tests of the v-prediction target and Min-SNR-gamma weighting: the folded sampler tables of a v-model against the
eps tables on an exact Gaussian denoiser, the weight tables, argument checks, state-dict layout and the checkpoint
config keys."""
import math

import pytest
import torch

from objective_oracle import weighted_diffusion_loss
from oracle import cesm_oracle as O

T = 1000
S = 2.0  # data ~ N(0, S^2)


def _ac():
    return O.diffusion_buffers(T)["alphas_cumprod"]


def _diffusion(prediction_type="eps"):
    from cesm_emulator_b200.model import Diffusion
    return Diffusion(torch.nn.Linear(1, 1), prediction_type=prediction_type)


def _gauss_eps(x, t):
    """Exact eps-predictor of data ~ N(0, S^2) in float64."""
    a = _ac().double()[t]
    return torch.sqrt(1 - a) * x / (a * S * S + 1 - a)


def _gauss_v(x, t):
    """The same denoiser as a v-predictor: v = (eps - sqrt(1 - ab) x) / sqrt(ab)."""
    a = _ac().double()[t]
    return (_gauss_eps(x, t) - torch.sqrt(1 - a) * x) / torch.sqrt(a)


def _row(coef, t, x, e, z, hist):
    c = coef[t].double()
    if coef.shape[1] == 3:
        return c[0] * x + c[1] * e + c[2] * z, hist
    x0 = c[0] * x + c[1] * e
    return c[2] * x + c[3] * x0 + (c[4] * hist if c[4] != 0 else 0.0), x0


def _chains(kind, steps, eta=0.0):
    """Run the eps-table chain fed eps and the v-table chain fed v from one x_T (and one z per step) in float64.
    -> (worst one-step rel. difference, final rel. difference)."""
    from cesm_emulator_b200.model import ddim_schedule, dpm_schedule
    if kind == "dpm":
        taus, ce, _ = dpm_schedule(_ac(), steps)
        _, cv, _ = dpm_schedule(_ac(), steps, "v")
    else:
        taus, ce, _ = ddim_schedule(_ac(), steps, eta)
        _, cv, _ = ddim_schedule(_ac(), steps, eta, "v")
    g = torch.Generator().manual_seed(steps)
    xe = xv = torch.randn(4096, generator=g, dtype=torch.float64)
    he = hv = torch.full_like(xe, float("nan"))
    worst = 0.0
    for t in taus:
        z = torch.randn(4096, generator=g, dtype=torch.float64)
        # one step from the same point
        se, _ = _row(ce, t, xv, _gauss_eps(xv, t), z, hv)
        sv, _ = _row(cv, t, xv, _gauss_v(xv, t), z, hv)
        worst = max(worst, ((se - sv).abs().max() / se.abs().max()).item())
        xe, he = _row(ce, t, xe, _gauss_eps(xe, t), z, he)
        xv, hv = _row(cv, t, xv, _gauss_v(xv, t), z, hv)
    return worst, ((xe - xv).abs().max() / xe.abs().max()).item()


# Both tables are fp32 roundings of float64 rows; measured: at most 1.4e-7 per step and 5.8e-7 over 1000 steps
@pytest.mark.parametrize("kind,steps,eta", [("ddim", 10, 0.0), ("ddim", 50, 0.0), ("ddim", 10, 1.0), ("ddim", 50, 1.0),
                                            ("ddim", 1000, 1.0), ("dpm", 10, 0.0), ("dpm", 20, 0.0)])
def test_folded_tables_fed_v_equal_eps_tables_fed_eps(kind, steps, eta):
    step, chain = _chains(kind, steps, eta)
    assert step < 2e-6 and chain < 2e-6, (step, chain)


def test_v_tables_keep_the_schedule_shape():
    from cesm_emulator_b200.model import ddim_schedule, dpm_schedule
    for fn, args in ((ddim_schedule, (50, 0.5)), (dpm_schedule, (15,))):
        te, ce, ne = fn(_ac(), *args)
        tv, cv, nv = fn(_ac(), *args, prediction_type="v")
        assert te == tv and torch.equal(ne, nv) and cv.dtype == torch.float32 and cv.shape == ce.shape
        assert torch.equal(torch.isnan(cv), torch.isnan(ce))
    # DPM: x0 = sqrt(ab) x - sqrt(1 - ab) v exactly (no cancellation in the table)
    taus, cv, _ = dpm_schedule(_ac(), 10, "v")
    a = _ac().double()[taus[0]]
    assert cv[taus[0], 0].item() == pytest.approx(math.sqrt(a), rel=1e-7)
    assert cv[taus[0], 1].item() == pytest.approx(-math.sqrt(1 - a), rel=1e-7)


def test_eps_tables_unchanged():
    """The eps rows are the ones the samplers used before prediction_type existed."""
    from cesm_emulator_b200.model import ddim_schedule
    ac = _ac().double()
    taus, coef, _ = ddim_schedule(_ac(), 20, 0.0)
    for i, t in enumerate(taus):
        a_t, a_p = ac[t], (ac[taus[i + 1]] if i + 1 < len(taus) else torch.tensor(1.0, dtype=torch.float64))
        assert coef[t, 0].item() == pytest.approx(torch.sqrt(a_p / a_t).item(), rel=1e-6)
        ref_b = torch.sqrt(1 - a_p) - torch.sqrt(a_p) * torch.sqrt(1 - a_t) / torch.sqrt(a_t)
        assert coef[t, 1].item() == pytest.approx(ref_b.item(), rel=1e-6)


def test_ddpm_table_of_a_v_model_is_the_posterior_step():
    """Diffusion(prediction_type="v").ddpm_coef fed v equals p_sample's posterior formula fed eps, at every t."""
    d = _diffusion("v")
    assert d.ddpm_coef.shape == (T, 3) and d.ddpm_coef.dtype == torch.float32 and torch.isfinite(d.ddpm_coef).all()
    assert _diffusion("eps").ddpm_coef is None and _diffusion("eps").target_coef is None
    g = torch.Generator().manual_seed(1)
    worst = 0.0
    for t in list(range(0, T, 37)) + [1, T - 1]:
        x = torch.randn(2048, generator=g, dtype=torch.float64) * 1.5
        z = torch.randn(2048, generator=g, dtype=torch.float64)
        e = _gauss_eps(x, t)
        mean = d.sqrt_recip_alphas.double()[t] * (x - d.betas.double()[t] / d.sqrt_one_minus_alphas_cumprod.double()[t] * e)
        ref = mean + torch.sqrt(d.posterior_variance.double()[t]) * z
        got, _ = _row(d.ddpm_coef, t, x, _gauss_v(x, t), z, None)
        worst = max(worst, ((got - ref).abs().max() / ref.abs().max()).item())
    assert worst < 1e-4, worst
    assert d.ddpm_coef[0, 2] == 0  # the last step adds no noise, as posterior_variance[0] == 0


def test_v_target_coefficients():
    d = _diffusion("v")
    ac = d.alphas_cumprod.double()
    assert d.target_coef.dtype == torch.float32 and d.target_coef.shape == (T, 2)
    assert torch.allclose(d.target_coef.double(), torch.stack([ac.sqrt(), -(1 - ac).sqrt()], 1), rtol=1e-7, atol=0)


# ---- weights -----------------------------------------------------------------------------------------------------
def test_min_snr_weights_values():
    de, dv = _diffusion("eps"), _diffusion("v")
    ac = de.alphas_cumprod.double()
    snr = ac / (1 - ac)
    we, wv = de.min_snr_weights(5), dv.min_snr_weights(5.0)
    assert we.dtype == wv.dtype == torch.float32 and we.shape == wv.shape == (T,)
    # the smallest weights: v at t = 999 (SNR < gamma there, so w = SNR / (SNR + 1) = ab), eps at t = 0
    assert wv[999].item() == pytest.approx(ac[999].item(), rel=1e-6) and 3.9e-5 < wv[999].item() < 4.1e-5
    assert we[0].item() == pytest.approx(5.0 / snr[0].item(), rel=1e-6) and 4.9e-4 < we[0].item() < 5.1e-4
    assert wv.min() == wv[999] and we.min() == we[0]
    # below gamma: eps weight 1, v weight SNR / (SNR + 1); above: gamma / SNR and gamma / (SNR + 1)
    for t in (0, 100, 300, 700, 999):
        s = snr[t].item()
        assert we[t].item() == pytest.approx(min(s, 5.0) / s, rel=1e-6)
        assert wv[t].item() == pytest.approx(min(s, 5.0) / (s + 1), rel=1e-6)
    # both weight the x0 error by min(SNR, gamma)
    assert torch.allclose(we.double() * snr, wv.double() * (snr + 1), rtol=1e-6)
    assert torch.allclose(de.min_snr_weights(1e9).double(), torch.ones(T, dtype=torch.float64))


def test_alpha_bar_times_v_error_is_the_eps_error():
    """At one x_t, eps_hat - eps = sqrt(ab) (v_hat - v): the saliency of a v-model weights its v-MSE by ab."""
    ac = _ac().double()
    g = torch.Generator().manual_seed(2)
    for t in (0, 250, 999):
        a = ac[t]
        x0, eps, v_hat = (torch.randn(512, generator=g, dtype=torch.float64) for _ in range(3))
        x_t = a.sqrt() * x0 + (1 - a).sqrt() * eps
        v = a.sqrt() * eps - (1 - a).sqrt() * x0
        eps_hat = a.sqrt() * v_hat + (1 - a).sqrt() * x_t
        lhs = a * ((v_hat - v) ** 2).sum()
        assert lhs.item() == pytest.approx(((eps_hat - eps) ** 2).sum().item(), rel=1e-10)


# ---- argument checks ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("bad", ["x0", "V", "", None, 1, "epsilon"])
def test_bad_prediction_type_raises(bad):
    from cesm_emulator_b200.model import ddim_schedule, dpm_schedule
    with pytest.raises(ValueError, match="prediction_type"):
        _diffusion(bad)
    with pytest.raises(ValueError):
        ddim_schedule(_ac(), 10, 0.0, bad)
    with pytest.raises(ValueError):
        dpm_schedule(_ac(), 10, bad)


@pytest.mark.parametrize("bad", [0, 0.0, -1, -5.0, float("nan"), float("inf"), -float("inf"), True, False, "5", None])
def test_bad_gamma_raises(bad):
    for d in (_diffusion("eps"), _diffusion("v")):
        with pytest.raises(ValueError, match="min_snr_gamma"):
            d.min_snr_weights(bad)


def test_bad_weights_raise_before_any_kernel():
    d = _diffusion("v")
    x = torch.zeros(2, 1, 4, 4)
    for w in (torch.ones(T - 1), torch.ones(2, T), [1.0] * T):
        with pytest.raises(ValueError, match="weights"):
            d.loss(x, x, torch.zeros(2, dtype=torch.long), x, weights=w)


def test_prediction_type_is_keyword_only_and_state_dict_unchanged():
    from cesm_emulator_b200.model import Diffusion
    with pytest.raises(TypeError):
        Diffusion(torch.nn.Linear(1, 1), 1, 1000, "linear", "v")
    ke, kv = list(_diffusion("eps").state_dict()), list(_diffusion("v").state_dict())
    assert ke == kv
    assert not [k for k in kv if "coef" in k]
    assert _diffusion().prediction_type == "eps"
    with pytest.raises(ValueError):  # other schedules are still refused
        Diffusion(torch.nn.Linear(1, 1), beta_schedule="cosine", prediction_type="v")


def test_config_keys_and_resume_check(tmp_path):
    import train as train_entry
    assert train_entry.prediction_type_from_config({}) == "eps"
    assert train_entry.prediction_type_from_config(None) == "eps"
    assert train_entry.prediction_type_from_config({"diffusion": {"timesteps": 1000}}) == "eps"
    assert train_entry.prediction_type_from_config({"diffusion": {"prediction_type": "v"}}) == "v"
    dv = _diffusion("v")
    path = str(tmp_path / "v.pt")
    sd = dv.state_dict()
    torch.save({"epoch": 3, "model": {k[len("model."):]: v for k, v in sd.items() if k.startswith("model.")},
                "config": {"diffusion": {"prediction_type": "v"}}}, path)
    assert train_entry.load_checkpoint(path, _diffusion("v"), device="cpu") == 4
    with pytest.raises(ValueError, match="prediction_type"):
        train_entry.load_checkpoint(path, _diffusion("eps"), device="cpu")
    old = str(tmp_path / "old.pt")  # a checkpoint from before the key existed is an eps checkpoint
    torch.save({"epoch": 1, "model": {}, "config": {"diffusion": {"timesteps": 1000}}}, old)
    assert train_entry.load_checkpoint(old, _diffusion("eps"), device="cpu") == 2
    with pytest.raises(ValueError, match="prediction_type"):
        train_entry.load_checkpoint(old, _diffusion("v"), device="cpu")


def test_train_engine_rejects_bad_gamma_before_building():
    from cesm_emulator_b200.engine import TrainEngine
    with pytest.raises(ValueError, match="min_snr_gamma"):
        TrainEngine(_diffusion("v"), (2, 1, 4, 4), (2, 1, 1, 4, 4), min_snr_gamma=0)


def test_objective_oracle_reduces_to_the_reference_loss():
    """The weighted oracle with the eps target and no (or unit) weights is the reference's MSE; with the v target and
    weights it is the batch mean of weights[t_b] times each sample's own MSE against v."""
    cfg = O.OracleConfig(model_dim=16, dim_mults=(1, 2))
    sd = O.random_state_dict(cfg, seed=3)
    buf = O.diffusion_buffers(T)
    g = torch.Generator().manual_seed(4)
    x0, noise = torch.randn(2, 1, 8, 8, generator=g), torch.randn(2, 1, 8, 8, generator=g)
    cond = torch.randn(2, 1, 3, 8, 8, generator=g)
    t = torch.tensor([5, 900])
    with torch.no_grad():
        ref = O.diffusion_loss(sd, cfg, buf, x0, cond, t, noise)
        assert torch.allclose(weighted_diffusion_loss(sd, cfg, buf, x0, cond, t, noise, "eps"), ref, rtol=1e-6)
        assert torch.allclose(weighted_diffusion_loss(sd, cfg, buf, x0, cond, t, noise, "eps", torch.ones(T)), ref,
                              rtol=1e-6)
        w = torch.rand(T, generator=g)
        pred = O.unet_forward(sd, cfg, O.q_sample(buf, x0, t, noise), cond, t)
        a, s = buf["sqrt_alphas_cumprod"][t].view(-1, 1, 1, 1), buf["sqrt_one_minus_alphas_cumprod"][t].view(-1, 1, 1, 1)
        per = ((pred - (a * noise - s * x0)) ** 2).mean(dim=(1, 2, 3))
        got = weighted_diffusion_loss(sd, cfg, buf, x0, cond, t, noise, "v", w)
        assert torch.allclose(got, (w[t] * per).mean(), rtol=1e-6)
