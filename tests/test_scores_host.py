"""Host tests of the ensemble scores: the float64 oracle, the synthetic ensemble's known truth, evaluate.py's argument
checks and the NetCDF writers."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import score_oracle  # noqa: E402


def test_oracle_hand_worked_two_members():
    # X = {0, 2}, Y = {1, 3}: mean_j (1/2) sum_i |x_i - y_j| = (1 + 2) / 2, pair term |0 - 2| / (2 * 1) = 1
    s = score_oracle.ensemble_scores(np.array([[[0.0], [2.0]]]), np.array([[[1.0], [3.0]]]))
    assert s["crps"][0, 0] == pytest.approx(0.5)
    assert s["bias"][0, 0] == pytest.approx(-1.0)
    assert s["sd_pred"][0, 0] == pytest.approx(np.sqrt(2)) and s["sd_target"][0, 0] == pytest.approx(np.sqrt(2))
    assert s["mse_mean"][0, 0] == pytest.approx(2.0)  # mean(X) = 1: ((1 - 1)^2 + (1 - 3)^2) / 2
    assert s["rank_hist"].tolist() == [[0, 1, 1]]


def test_oracle_ties_are_not_below():
    s = score_oracle.ensemble_scores(np.array([[[1.0], [1.0], [2.0]]]), np.array([[[1.0], [2.0]]]))
    assert s["rank_hist"].tolist() == [[1, 0, 1, 0]]  # y = 1: nothing below; y = 2: the two ones


def test_oracle_non_finite_column():
    x = np.zeros((1, 3, 2))
    x[0, 1, 0] = np.inf
    s = score_oracle.ensemble_scores(x, np.ones((1, 2, 2)))
    assert all(np.isnan(s[k][0, 0]) and np.isfinite(s[k][0, 1]) for k in ("crps", "bias", "sd_pred", "mse_mean"))
    assert s["rank_hist"].tolist() == [[0, 0, 0, 2]]


def test_oracle_fair_crps_matches_the_gaussian_closed_form():
    # E[fair CRPS of n draws from N(mu, s^2)] = CRPS(N(mu, s^2), y) exactly; over 20000 columns of n = 64 the
    # standard error of the mean difference is ~ 0.4 % of s (per-column spread of the estimator ~ 0.6 s), so 2 % of s
    # is a 5-sigma bar
    rng = np.random.default_rng(0)
    P, n, mu, s = 20000, 64, 1.5, 0.7
    x = mu + s * rng.standard_normal((1, n, P))
    y = mu + 2 * s * rng.standard_normal((1, 1, P))
    got = score_oracle.ensemble_scores(x, np.repeat(y, 2, axis=1))["crps"].mean()
    want = score_oracle.gaussian_crps(mu, s, y).mean()
    assert abs(got - want) < 0.02 * s, (got, want)


def test_synthetic_known_truth_reproduces_the_targets():
    from cesm_emulator_b200.synthetic import SyntheticEnsemble
    ds = SyntheticEnsemble(members=6, times=10, lat=24, lon=36, seed=3)
    assert ds.target_mean.shape == (10, 24, 36) and ds.target_mean.dtype == np.float32
    resid = (ds.tgt[:, :, 0].astype(np.float64) - ds.target_mean[:, None]) / ds.target_noise_std
    assert abs(resid.mean()) < 0.02 and abs(resid.std() - 1) < 0.02, (resid.mean(), resid.std())
    fa = SyntheticEnsemble.from_arrays(ds.cond, ds.tgt)
    assert fa.target_mean is None and fa.target_noise_std is None


def _tiny_checkpoint(tmp_path, with_ema):
    from cesm_emulator_b200.model import Diffusion
    from train import build_model_from_config
    ucfg = {"base_ch": 16, "ch_mults": [1, 2], "groups": 4, "num_res_blocks": 1, "time_dim": 16,
            "in_channels": 2, "out_channels": 1}
    cfg = {"unet": ucfg, "diffusion": {"timesteps": 20},
           "data": {"synthetic": {"members": 3, "times": 4, "lat": 16, "lon": 16, "seed": 5}}}
    torch.manual_seed(0)
    diff = Diffusion(build_model_from_config(ucfg), timesteps=20)
    ckpt = {"model": diff.model.state_dict(), "config": cfg, "epoch": 1}
    if with_ema:
        ckpt["ema"] = diff.model.state_dict()
    path = str(tmp_path / "tiny.pt")
    torch.save(ckpt, path)
    return path


@pytest.mark.parametrize("argv", [
    ["--years", "3"], ["--years", "a:4"], ["--years", "4:2"], ["--years", "-1:2"], ["--years", "0:4:0"],
    ["--years", "0:1:2:3"], ["--steps", "10", "--ddim_steps", "5"], ["--dpm_steps", "5", "--steps", "10"],
    ["--dpm_steps", "5", "--ddim_steps", "5"], ["--dpm_steps", "5", "--eta", "1"], ["--seed", "-1"],
    ["--seed", str(1 << 64)], ["--guidance", "-1"], ["--guidance", "nan"], ["--batch_size", "0"],
    ["--out", "scores.npy"]])
def test_evaluate_argument_errors(argv, capsys):
    import evaluate
    with pytest.raises(SystemExit) as e:
        evaluate._parse_args(["--ckpt", "x.pt", *argv])
    assert e.value.code == 2
    assert "error" in capsys.readouterr().err


def test_evaluate_argument_defaults():
    import evaluate
    a = evaluate._parse_args(["--ckpt", "x.pt"])
    assert (a.batch_size, a.years, a.out, a.seed, a.ema, a.guidance) == (16, None, "scores.npz", None, False, 0.0)
    assert evaluate._parse_args(["--ckpt", "x.pt", "--years", "2:10:4"]).years == slice(2, 10, 4)
    assert evaluate._parse_args(["--ckpt", "x.pt", "--ddim_steps", "5", "--eta", "1"]).eta == 1.0


def test_evaluate_ema_on_a_checkpoint_without_one(tmp_path):
    import evaluate
    path = _tiny_checkpoint(tmp_path, with_ema=False)
    with pytest.raises(SystemExit) as e:
        evaluate.main(["--ckpt", path, "--ema", "--out", str(tmp_path / "s.npz")])
    assert '"ema"' in str(e.value.code)
    assert not os.path.exists(tmp_path / "s.npz")


def test_evaluate_guidance_without_condition_dropout(tmp_path):
    import evaluate
    path = _tiny_checkpoint(tmp_path, with_ema=True)
    with pytest.raises(SystemExit) as e:
        evaluate.main(["--ckpt", path, "--guidance", "1", "--out", str(tmp_path / "s.npz")])
    assert "cond_drop_prob" in str(e.value.code)


def test_evaluate_years_outside_the_checkpoint_ensemble(tmp_path):
    import evaluate
    path = _tiny_checkpoint(tmp_path, with_ema=True)  # times = 4
    with pytest.raises(SystemExit) as e:
        evaluate.main(["--ckpt", path, "--years", "2:5", "--out", str(tmp_path / "s.npz")])
    assert "outside the 4 years" in str(e.value.code)


def test_inference_and_evaluate_share_the_sampler_flags():
    import evaluate
    import inference
    flags = ("--steps", "--ddim_steps", "--eta", "--dpm_steps", "--ema", "--seed", "--guidance")
    for mod in (inference, evaluate):
        a = mod._parse_args(["--ckpt", "x.pt", "--dpm_steps", "7", "--ema", "--seed", "3", "--guidance", "0.5"])
        assert (a.dpm_steps, a.ema, a.seed, a.guidance, a.steps, a.ddim_steps, a.eta) == (7, True, 3, 0.5, None, None,
                                                                                          0.0)
    assert all(f.lstrip("-") in vars(evaluate._parse_args(["--ckpt", "x.pt"])) for f in flags)


def test_multi_variable_netcdf_round_trip(tmp_path):
    from scipy.io import netcdf_file
    import inference
    rng = np.random.default_rng(0)
    a, h = rng.standard_normal((3, 4, 5)).astype(np.float32), rng.integers(0, 9, (3, 6))
    s = rng.standard_normal(3)
    path = str(tmp_path / "sub" / "multi.nc")
    inference.write_netcdf_variables(
        path, [("year", [4, 6, 8], 3), ("lat", None, 4), ("lon", np.linspace(0, 1, 5), 5), ("rank", None, 6)],
        [("crps", a, ("year", "lat", "lon"), {"units": "standardized"}), ("rank_hist", h, ("year", "rank"), {}),
         ("crps_year", s, ("year",), {})],
        {"checkpoint": "/x/final.pt", "seed": "0", "ema": 1, "eta": 0.5})
    with netcdf_file(path, "r", mmap=False) as f:
        assert f.variables["crps"].dimensions == ("year", "lat", "lon")
        assert np.array_equal(np.array(f.variables["crps"][:]), a) and f.variables["crps"].units == b"standardized"
        assert f.variables["rank_hist"].dimensions == ("year", "rank") and f.variables["rank_hist"][:].dtype.kind == "i"
        assert np.array_equal(np.array(f.variables["rank_hist"][:]), h)
        assert np.array_equal(np.array(f.variables["crps_year"][:]), s.astype(np.float32))
        assert list(f.variables["year"][:]) == [4, 6, 8] and list(f.variables["rank"][:]) == list(range(6))
        assert np.allclose(f.variables["lon"][:], np.linspace(0, 1, 5))
        assert (f.checkpoint, f.seed, f.ema, f.eta) == (b"/x/final.pt", b"0", 1, 0.5)


def _parent_write_netcdf_variable(path, name, data, coords, attrs):
    """write_netcdf_variable as it was before it became a front of write_netcdf_variables."""
    from scipy.io import netcdf_file
    d = os.path.dirname(path)
    if d:
        os.makedirs(d, exist_ok=True)
    with netcdf_file(path, "w", version=2) as f:
        for dim, vals, n in coords:
            f.createDimension(dim, n)
            vals = np.arange(n) if vals is None else np.asarray(vals)
            if vals.shape != (n,):
                raise ValueError(f"coordinate {dim} has shape {vals.shape}, expected ({n},)")
            vals = vals.astype(np.float64 if vals.dtype.kind == "f" else np.int32)
            v = f.createVariable(dim, vals.dtype, (dim,))
            v[:] = vals
        v = f.createVariable(name, np.float32, tuple(dim for dim, _, _ in coords))
        v[:] = np.asarray(data, dtype=np.float32)
        for k, val in attrs.items():
            setattr(v, k, val)


def test_single_variable_netcdf_is_byte_identical_to_before(tmp_path):
    import inference
    pred = np.random.default_rng(1).standard_normal((2, 3, 4, 5)).astype(np.float32)
    attrs = {"description": "d", "units": "standardized", "checkpoint": "/x/final.pt", "draws": 16}
    for coords in ([("year", None, 2), ("member_id", [1, 2, 3], 3), ("lat", np.linspace(-1, 1, 4), 4),
                    ("lon", None, 5)],):
        inference.write_netcdf_variable(str(tmp_path / "new.nc"), "TREFHT_pred", pred, coords, attrs)
        _parent_write_netcdf_variable(str(tmp_path / "old.nc"), "TREFHT_pred", pred, coords, attrs)
        assert (tmp_path / "new.nc").read_bytes() == (tmp_path / "old.nc").read_bytes()
    inference.write_prediction_netcdf(str(tmp_path / "p_new.nc"), pred, attrs={"checkpoint": "/c.pt"})
    T, M, H, W = pred.shape
    _parent_write_netcdf_variable(
        str(tmp_path / "p_old.nc"), "TREFHT_pred", pred,
        [("year", None, T), ("member_id", None, M), ("lat", None, H), ("lon", None, W)],
        {"description": "Predicted near-surface air temperature from emissions via diffusion model",
         "units": "standardized", "checkpoint": "/c.pt"})
    assert (tmp_path / "p_new.nc").read_bytes() == (tmp_path / "p_old.nc").read_bytes()


def test_summaries_on_hand_made_maps():
    import evaluate
    n = 3
    crps = torch.tensor([[1.0, 3.0, float("nan")], [2.0, 2.0, 2.0]])
    scores = {"crps": crps, "bias": torch.tensor([[1.0, -1.0, float("nan")], [0.5, 0.5, 0.5]]),
              "sd_pred": torch.tensor([[1.0, 1.0, float("nan")], [2.0, 2.0, 2.0]]),
              "sd_target": torch.ones(2, 3),
              "mse_mean": torch.tensor([[4.0, 4.0, float("nan")], [1.0, 1.0, 1.0]]),
              "rank_hist": torch.tensor([[2, 2, 0, 0], [1, 1, 1, 3]])}
    s = evaluate.summarize_scores(scores, n)
    y, o = s["year"], s["overall"]
    assert y["crps"].tolist() == [2.0, 2.0] and y["nonfinite"].tolist() == [1, 0]
    assert y["rmse"].tolist() == [2.0, 1.0] and y["spread"].tolist() == [1.0, 2.0]
    assert y["ssr"].tolist() == pytest.approx([np.sqrt(4 / 3) / 2, np.sqrt(4 / 3) * 2])
    assert np.allclose(y["rank_freq"].numpy(), [[0.5, 0.5, 0, 0], [1 / 6, 1 / 6, 1 / 6, 0.5]])
    assert o["crps"] == pytest.approx(2.0) and o["bias"] == pytest.approx(0.3) and o["nonfinite"] == 1
    assert o["rmse"] == pytest.approx(np.sqrt(11 / 5)) and o["spread"] == pytest.approx(np.sqrt(14 / 5))
    assert o["rank_freq"].tolist() == pytest.approx([0.3, 0.3, 0.1, 0.3])
    assert o["chi2"] == pytest.approx(sum((c - 2.5) ** 2 / 2.5 for c in (3, 3, 1, 3)))
