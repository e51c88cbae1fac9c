"""CPU tests of classifier-free guidance: the float64 guided chains at w = 0 against the existing chain references, that
combining v equals combining eps, argument checks of the guidance weight and the dropout probability, the checkpoint
config round trip, and that a reference checkpoint still loads strictly."""
import math
import os

import pytest
import torch

import ddim_oracle as DO
import dpm_oracle as PO
import guidance_oracle as GO
from oracle import cesm_oracle as O

T = 1000
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _tiny():
    cfg = O.OracleConfig(model_dim=16, dim_mults=(1, 2))
    return cfg, O.random_state_dict(cfg, seed=5)


def _inputs(seed=6):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(2, 1, 8, 8, generator=g), torch.randn(2, 1, 8, 8, generator=g), g


def _close(a, b, tol=1e-4):
    a, b = a.double(), b.double()
    return ((a - b).abs().max() / b.abs().max()).item() <= tol


def test_oracle_at_w0_equals_the_existing_chains():
    cfg, sd = _tiny()
    buf = O.diffusion_buffers(T)
    net = GO.oracle_net(sd, cfg)
    cond, x_T, g = _inputs()
    with torch.no_grad():
        assert _close(GO.guided_ddim_sample(net, buf, cond, x_T, 3, 0.0, 0.0), DO.ddim_sample(sd, cfg, buf, cond, x_T, 3, 0.0))
        zs = [torch.randn(2, 1, 8, 8, generator=g) for _ in range(3)]
        assert _close(GO.guided_ddim_sample(net, buf, cond, x_T, 3, 1.0, 0.0, zs),
                      DO.ddim_sample(sd, cfg, buf, cond, x_T, 3, 1.0, zs))
        assert _close(GO.guided_dpm_sample(net, buf, cond, x_T, 4, 0.0), PO.dpm_sample(sd, cfg, buf, cond, x_T, 4))
        x = x_T
        for i, z in enumerate(zs):
            x = O.p_sample(sd, cfg, buf, x, cond, torch.full((2,), T - 1 - i, dtype=torch.long), z)
        assert _close(GO.guided_ddpm_sample(net, buf, cond, x_T, 0.0, zs), x)


def test_guided_output_calls_the_net_with_the_null_condition():
    calls = []

    def net(x, cond, t):
        calls.append(cond.clone())
        return x + cond.mean()

    x, cond = torch.ones(2, 1, 4, 4), torch.full((2, 1, 4, 4), 3.0)
    assert torch.equal(GO.guided_output(net, x, cond, torch.zeros(2, dtype=torch.long), 0.0), x + 3) and len(calls) == 1
    out = GO.guided_output(net, x, cond, torch.zeros(2, dtype=torch.long), 2.0)
    assert len(calls) == 3 and torch.equal(calls[2], torch.zeros_like(cond))
    assert torch.allclose(out, 3 * (x + 3) - 2 * x)


@pytest.mark.parametrize("w", [0.5, 1.0, 4.0])
def test_combining_v_equals_combining_eps(w):
    """The weights (1 + w, -w) sum to 1 and eps = sqrt(ab) v + sqrt(1 - ab) x is affine in v at fixed (x, t): the eps of
    the combined v is the combination of the two eps.  So one kernel formula serves both targets."""
    buf = O.diffusion_buffers(T)
    g = torch.Generator().manual_seed(7)
    x, vc, vu = (torch.randn(4, 1, 6, 6, generator=g, dtype=torch.float64) for _ in range(3))
    t = torch.tensor([0, 250, 750, 999])
    lhs = GO.to_eps(buf, x, GO.combine(vc, vu, w), t, "v")
    rhs = GO.combine(GO.to_eps(buf, x, vc, t, "v"), GO.to_eps(buf, x, vu, t, "v"), w)
    assert torch.allclose(lhs, rhs, rtol=0, atol=1e-12)
    # and through the folded sampler tables of a v-model: a row applied to combined v is the eps row applied to the
    # combined eps
    from cesm_emulator_b200.model import ddim_schedule
    ac = buf["alphas_cumprod"]
    _, ce, _ = ddim_schedule(ac, 10, 0.5, "eps")
    _, cv, _ = ddim_schedule(ac, 10, 0.5, "v")
    taus = DO.ddim_timesteps(T, 10)
    tau = torch.tensor([taus[0], taus[3], taus[7], taus[9]])
    z = torch.randn(4, 1, 6, 6, generator=g, dtype=torch.float64)
    ev, ee = cv.double()[tau], ce.double()[tau]
    col = lambda c: c.view(-1, 1, 1, 1)  # noqa: E731
    out_v = col(ev[:, 0]) * x + col(ev[:, 1]) * GO.combine(vc, vu, w) + col(ev[:, 2]) * z
    eps_c = GO.combine(GO.to_eps(buf, x, vc, tau, "v"), GO.to_eps(buf, x, vu, tau, "v"), w)
    out_e = col(ee[:, 0]) * x + col(ee[:, 1]) * eps_c + col(ee[:, 2]) * z
    assert ((out_v - out_e).abs().max() / out_e.abs().max()).item() <= 1e-5


def test_masked_loss_is_the_loss_on_the_null_condition():
    cfg, sd = _tiny()
    buf = O.diffusion_buffers(T)
    g = torch.Generator().manual_seed(8)
    x0, noise = torch.randn(2, 1, 8, 8, generator=g), torch.randn(2, 1, 8, 8, generator=g)
    cond = torch.randn(2, 1, 3, 8, 8, generator=g)
    t = torch.tensor([40, 700])
    with torch.no_grad():
        full = GO.masked_diffusion_loss(sd, cfg, buf, x0, cond, t, noise, torch.ones(2))
        assert torch.allclose(full, O.diffusion_loss(sd, cfg, buf, x0, cond, t, noise), rtol=1e-6)
        keep = torch.tensor([1.0, 0.0])
        got = GO.masked_diffusion_loss(sd, cfg, buf, x0, cond, t, noise, keep)
        null = cond.clone()
        null[1] = 0
        assert torch.allclose(got, O.diffusion_loss(sd, cfg, buf, x0, null, t, noise), rtol=1e-6)


@pytest.mark.parametrize("bad", [-0.5, -1e-9, float("nan"), float("inf"), True, "2", None])
def test_bad_guidance_raises(bad):
    from cesm_emulator_b200.model import check_guidance
    with pytest.raises(ValueError, match="guidance"):
        check_guidance(bad)


def test_good_guidance_values():
    from cesm_emulator_b200.model import check_guidance
    assert check_guidance(0) == 0.0 and check_guidance(2) == 2.0 and check_guidance(0.75) == 0.75


@pytest.mark.parametrize("bad", [-0.1, 1.0, 1.5, float("nan"), True, "0.1", None])
def test_bad_cond_drop_prob_raises(bad):
    from cesm_emulator_b200.engine import TrainEngine
    from cesm_emulator_b200.model import Diffusion, check_cond_drop_prob
    with pytest.raises(ValueError, match="cond_drop_prob"):
        check_cond_drop_prob(bad)
    with pytest.raises(ValueError, match="cond_drop_prob"):  # before anything is built
        TrainEngine(Diffusion(torch.nn.Linear(1, 1)), (2, 1, 4, 4), (2, 1, 1, 4, 4), cond_drop_prob=bad)


def test_samplers_reject_bad_guidance_before_any_kernel():
    from cesm_emulator_b200.engine import SampleEngine
    from cesm_emulator_b200.model import Diffusion
    d = Diffusion(torch.nn.Linear(1, 1))
    for call in (lambda: d.sample(None, (1, 1, 4, 4), "cpu", guidance=-1),
                 lambda: d.ddim_sample(None, (1, 1, 4, 4), "cpu", guidance=-1),
                 lambda: d.dpm_sample(None, (1, 1, 4, 4), "cpu", guidance=float("nan")),
                 lambda: SampleEngine(d, (1, 1, 4, 4), guidance=-2.0)):
        with pytest.raises(ValueError, match="guidance"):
            call()


def test_guidance_needs_a_checkpoint_trained_with_dropout():
    from inference import check_guidance_for_config
    assert check_guidance_for_config(0.0, {}) == 0.0
    assert check_guidance_for_config(0, {"train": {"cond_drop_prob": 0.0}}) == 0.0
    assert check_guidance_for_config(3, {"train": {"cond_drop_prob": 0.1}}) == 3.0
    for cfg in ({}, None, {"train": {}}, {"train": {"cond_drop_prob": 0.0}}, {"train": {"cond_drop_prob": None}}):
        with pytest.raises(ValueError, match="cond_drop_prob"):
            check_guidance_for_config(1.5, cfg)
    with pytest.raises(ValueError, match="guidance"):
        check_guidance_for_config(-1.0, {"train": {"cond_drop_prob": 0.1}})


@pytest.mark.parametrize("argv", [["--guidance", "-1"], ["--guidance", "nan"], ["--guidance", "inf"]])
def test_inference_cli_rejects_bad_guidance(argv):
    import inference
    with pytest.raises(SystemExit):
        inference._parse_args(["--ckpt", "x.pt", *argv])


def test_inference_cli_takes_guidance_with_every_sampler():
    import inference
    for extra in ([], ["--ddim_steps", "10", "--eta", "1"], ["--dpm_steps", "5"], ["--ema", "--seed", "3"]):
        a = inference._parse_args(["--ckpt", "x.pt", "--guidance", "2.5", *extra])
        assert a.guidance == 2.5
    assert inference._parse_args(["--ckpt", "x.pt"]).guidance == 0.0


def test_cond_drop_prob_round_trips_through_the_checkpoint(tmp_path):
    import train as train_entry
    from cesm_emulator_b200.model import Diffusion

    class _Engine:  # what save_checkpoint reads of a TrainEngine
        has_ema = False

        class opt:
            @staticmethod
            def state_dict():
                return {"state": {}, "param_groups": []}

    cfg = {"train": {"cond_drop_prob": 0.1, "batch_size": 2}, "diffusion": {"prediction_type": "eps"}}
    path = str(tmp_path / "ck" / "c.pt")
    d = Diffusion(torch.nn.Linear(1, 1))
    train_entry.save_checkpoint(path, 2, d, _Engine, cfg)
    ck = torch.load(path, map_location="cpu", weights_only=False)
    assert train_entry.cond_drop_prob_from_config(ck["config"]) == 0.1
    assert train_entry.cond_drop_prob_from_config({}) == 0.0
    assert train_entry.cond_drop_prob_from_config({"train": {"batch_size": 2}}) == 0.0
    assert train_entry.load_checkpoint(path, Diffusion(torch.nn.Linear(1, 1)), device="cpu") == 3
    assert set(ck["model"]) == {k[len("model."):] for k in d.state_dict() if k.startswith("model.")}


def test_reference_checkpoint_still_loads_strictly():
    """Guidance adds no parameter or buffer: the reference's checkpoint loads with strict=True into the UNet that
    train.py builds, and the Diffusion's state-dict keys are unchanged."""
    import train as train_entry
    from cesm_emulator_b200.model import Diffusion
    ck = torch.load(os.path.join(ROOT, "tests", "golden", "ref_ckpt_tiny.pt"), map_location="cpu", weights_only=False)
    unet = train_entry.build_model_from_config(ck["config"].get("unet", {}))
    unet.load_state_dict(ck["model"], strict=True)
    d = Diffusion(unet)
    assert set(d.state_dict()) == {"model." + k for k in ck["model"]} | set(ck.get("diffusion_buffers", {}))
    assert math.isclose(train_entry.cond_drop_prob_from_config(ck["config"]), 0.0)
