"""Ensemble scores on the GPU: cesm_ensemble_scores against the float64 oracle (sizes, tiles, offsets, ties, non-finite
columns), its argument checks, launch count and reproducibility, its statistics on two draws of one Gaussian, and
evaluate.py end to end."""
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import score_oracle

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MAPS = ("crps", "bias", "sd_pred", "sd_target", "mse_mean")
BAR = 2e-5  # of each map's max |value|


def _data(T, n, m, HW, seed, scale="unit"):
    g = torch.Generator().manual_seed(seed)
    x, y = torch.randn((T, n, HW), generator=g), torch.randn((T, m, HW), generator=g) * 1.2 + 0.3
    if scale == "offset":
        x, y = x + 1000.0, y + 1000.0
    elif scale == "tiny":
        x, y = x * 1e-3, y * 1e-3
    return x.float(), y.float()


def _check(got, ref):
    for k in MAPS:
        a, b = got[k].double().cpu().numpy(), ref[k]
        assert np.array_equal(np.isnan(a), np.isnan(b)), k
        fin = ~np.isnan(b)
        if fin.any():
            err = np.abs(a[fin] - b[fin]).max() / max(np.abs(b[fin]).max(), 1e-30)
            assert err <= BAR, (k, err)
    assert np.array_equal(got["rank_hist"].cpu().numpy(), ref["rank_hist"])


CASES = ([(n, m, HW, T) for n in (2, 3, 31, 50, 257, 1024) for m in (2, 7, 50) for HW in (1, 33) for T in (1, 3)]
         + [(n, m, 192 * 288, 1) for n, m in ((2, 2), (3, 7), (31, 50), (50, 50))] + [(50, 7, 192 * 288, 3)])


@pytest.mark.parametrize("n,m,HW,T", CASES)
def test_scores_match_the_oracle(cuda, n, m, HW, T):
    from cesm_emulator_b200 import kernels as K
    x, y = _data(T, n, m, HW, seed=n * 7919 + m * 31 + HW + T)
    got = K.ensemble_scores(x.to(cuda), y.to(cuda))
    assert got["rank_hist"].dtype == torch.int64 and got["rank_hist"].shape == (T, n + 1)
    assert all(got[k].shape == (T, HW) and got[k].dtype == torch.float32 for k in MAPS)
    _check(got, score_oracle.ensemble_scores(x.numpy(), y.numpy()))
    assert int(got["rank_hist"].sum()) == T * m * HW


@pytest.mark.parametrize("scale", ["unit", "offset", "tiny"])
@pytest.mark.parametrize("n,m,HW,T", [(50, 50, 33, 3), (1024, 7, 33, 1), (31, 50, 192 * 288, 1)])
def test_accuracy_does_not_depend_on_the_offset(cuda, n, m, HW, T, scale):
    from cesm_emulator_b200 import kernels as K
    x, y = _data(T, n, m, HW, seed=11, scale=scale)
    _check(K.ensemble_scores(x.to(cuda), y.to(cuda)), score_oracle.ensemble_scores(x.numpy(), y.numpy()))


def test_ties_are_not_below(cuda):
    from cesm_emulator_b200 import kernels as K
    # one column by hand: X = {1, 1, 2}, Y = {1, 2, 3}: ranks 0, 2, 3
    x = torch.tensor([[[1.0], [1.0], [2.0]]], device=cuda)
    y = torch.tensor([[[1.0], [2.0], [3.0]]], device=cuda)
    assert K.ensemble_scores(x, y)["rank_hist"].tolist() == [[1, 0, 1, 1]]
    # many ties: values on a coarse grid, compared with the oracle's strict "<"
    g = torch.Generator().manual_seed(3)
    x = torch.randint(0, 4, (3, 37, 70), generator=g).float()
    y = torch.randint(0, 4, (3, 9, 70), generator=g).float()
    _check(K.ensemble_scores(x.to(cuda), y.to(cuda)), score_oracle.ensemble_scores(x.numpy(), y.numpy()))


@pytest.mark.parametrize("bad", [float("nan"), float("inf"), -float("inf")])
def test_non_finite_columns(cuda, bad):
    from cesm_emulator_b200 import kernels as K
    T, n, m, HW = 2, 13, 6, 70
    x, y = _data(T, n, m, HW, seed=5)
    clean = K.ensemble_scores(x.to(cuda), y.to(cuda))
    x[1, 4, 40] = bad   # one pred value
    y[0, 2, 3] = bad    # one target value
    got = K.ensemble_scores(x.to(cuda), y.to(cuda))
    ref = score_oracle.ensemble_scores(x.numpy(), y.numpy())
    _check(got, ref)
    keep = torch.ones((T, HW), dtype=torch.bool)
    keep[1, 40] = keep[0, 3] = False
    for k in MAPS:
        assert torch.isnan(got[k][1, 40]) and torch.isnan(got[k][0, 3])
        assert torch.equal(got[k].cpu()[keep], clean[k].cpu()[keep]), k
    assert got["rank_hist"].sum(1).tolist() == [m * (HW - 1), m * (HW - 1)]


def test_argument_errors_launch_nothing(cuda):
    from cesm_emulator_b200 import _lib
    from cesm_emulator_b200 import kernels as K
    ok = torch.zeros((2, 4, 33), device=cuda)
    bad = [(torch.zeros((2, 1, 33), device=cuda), ok), (ok, torch.zeros((2, 1, 33), device=cuda)),
           (torch.zeros((2, 1025, 1), device=cuda), torch.zeros((2, 4, 1), device=cuda)),
           (ok, torch.zeros((2, 1025, 33), device=cuda)),
           (ok, torch.zeros((3, 4, 33), device=cuda)), (ok, torch.zeros((2, 4, 32), device=cuda)),
           (ok.cpu(), ok), (ok, ok.cpu()), (ok.half(), ok), (ok, ok.double()),
           (torch.zeros((2, 33, 4), device=cuda).transpose(1, 2), ok), (ok, ok[:, :, :32].contiguous()[:, :, :31]),
           (ok[0], ok[0]), (ok, ok.view(2, 4, 33, 1))]
    torch.cuda.synchronize()
    before = _lib.launch_count()
    for p, t in bad:
        with pytest.raises(ValueError):
            K.ensemble_scores(p, t)
    assert _lib.launch_count() == before


def test_one_launch_and_bitwise_reproducible(cuda):
    from cesm_emulator_b200 import _lib
    from cesm_emulator_b200 import kernels as K
    x, y = _data(3, 50, 50, 192 * 288, seed=1)
    x, y = x.to(cuda), y.to(cuda)
    before = _lib.launch_count()
    a = K.ensemble_scores(x, y)
    assert _lib.launch_count() == before + 1
    b = K.ensemble_scores(x, y)
    for k in (*MAPS, "rank_hist"):
        assert torch.equal(a[k], b[k]), k
    # the tile of 16 pixels used when 32 do not fit in shared memory (n and m near 1024)
    x, y = _data(1, 1024, 1024, 40, seed=2)
    a, b = K.ensemble_scores(x.to(cuda), y.to(cuda)), K.ensemble_scores(x.to(cuda), y.to(cuda))
    assert all(torch.equal(a[k], b[k]) for k in (*MAPS, "rank_hist"))
    _check(a, score_oracle.ensemble_scores(x.numpy(), y.numpy()))


def test_two_draws_of_one_gaussian_are_calibrated(cuda):
    """Two independent 8-member ensembles from the same per-column N(mu, sigma^2): SSR = 1, a flat rank histogram and
    mean CRPS = sigma / sqrt(pi), the expected CRPS of a perfect Gaussian forecast.  Fixed seeds; the bars are ~ 10x
    the sampling error (the m values of a column share X, so the bins are not independent counts)."""
    import evaluate
    from cesm_emulator_b200 import kernels as K
    T, n, HW, sigma = 2, 8, 192 * 288, 1.3
    g = torch.Generator(device=cuda).manual_seed(1234)
    mu = 5.0 * torch.randn((T, 1, HW), generator=g, device=cuda)
    x = mu + sigma * torch.randn((T, n, HW), generator=g, device=cuda)
    y = mu + sigma * torch.randn((T, n, HW), generator=g, device=cuda)
    o = evaluate.summarize_scores(K.ensemble_scores(x, y), n)["overall"]
    assert abs(o["ssr"] - 1) < 0.02, o["ssr"]
    freq = o["rank_freq"].cpu().numpy()
    assert np.all(np.abs(freq * (n + 1) - 1) < 0.05), freq
    assert abs(o["crps"] / (sigma / math.sqrt(math.pi)) - 1) < 0.01, o["crps"]
    assert o["nonfinite"] == 0 and abs(o["bias"]) < 0.01


# ---- evaluate.py --------------------------------------------------------------------------------------------------
def _run(args):
    env = dict(os.environ, PYTHONPATH=ROOT)
    return subprocess.run([sys.executable, *args], capture_output=True, text=True, cwd=ROOT, env=env, timeout=900)


def test_evaluate_cli_end_to_end(cuda, tmp_path):
    from scipy.io import netcdf_file
    from cesm_emulator_b200 import kernels as K
    from cesm_emulator_b200.model import Diffusion
    from cesm_emulator_b200.synthetic import SyntheticEnsemble
    from inference import load_diffusion_from_checkpoint, predict_temperature_from_emissions
    from train import build_model_from_config
    cfg = json.load(open(os.path.join(ROOT, "config", "baseline")))
    cfg["data"]["synthetic"] = {"members": 3, "times": 5, "lat": 32, "lon": 48, "seed": 7}
    torch.manual_seed(0)
    diff = Diffusion(build_model_from_config(cfg["unet"]), timesteps=cfg["diffusion"]["timesteps"])
    ckpt = str(tmp_path / "tiny.pt")
    torch.save({"model": diff.model.state_dict(), "config": cfg, "epoch": 1}, ckpt)
    base = [os.path.join(ROOT, "evaluate.py"), "--ckpt", ckpt, "--dpm_steps", "2", "--seed", "0", "--batch_size", "4",
            "--years", "1:5:2"]
    npz, nc = str(tmp_path / "s.npz"), str(tmp_path / "s.nc")
    r = _run([*base, "--out", npz])
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    assert "ideal" in r.stdout and "model" in r.stdout, r.stdout
    r = _run([*base, "--out", nc])
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    Ty, n, H, W = 2, 3, 32, 48
    z = np.load(npz)
    assert z["year"].tolist() == [1, 3]
    assert all(z[k].shape == (Ty, H, W) for k in MAPS) and z["rank_hist"].shape == (Ty, n + 1)
    assert all(z[f"{k}_year"].shape == (Ty,) for k in ("crps", "bias", "rmse", "spread", "ssr", "nonfinite"))
    assert z["rank_freq_year"].shape == (Ty, n + 1) and z["rank_hist"].sum() == Ty * n * H * W
    assert json.loads(str(z["attrs"]))["dpm_steps"] == 2
    with netcdf_file(nc, "r", mmap=False) as f:
        for k in MAPS:
            assert f.variables[k].dimensions == ("year", "lat", "lon")
            assert np.allclose(np.array(f.variables[k][:]), z[k], rtol=0, atol=1e-3 * np.abs(z[k]).max())
        assert f.variables["rank_hist"].dimensions == ("year", "rank")
        assert f.variables["crps_year"].dimensions == ("year",) and f.seed == b"0" and f.sampler == b"dpm"
        assert list(f.variables["year"][:]) == [1, 3]
    # the maps are kernels.ensemble_scores of predict_temperature_from_emissions with the same seed
    diffusion, cfg2 = load_diffusion_from_checkpoint(ckpt, cuda)
    ds = SyntheticEnsemble(**cfg["data"]["synthetic"])
    pred = predict_temperature_from_emissions(diffusion, np.ascontiguousarray(ds.cond[1:5:2]), 4, device=cuda,
                                              dpm_steps=2, seed=0)
    ref = K.ensemble_scores(torch.from_numpy(pred.reshape(Ty, n, H * W)).to(cuda),
                            torch.from_numpy(ds.tgt[1:5:2].reshape(Ty, n, H * W)).to(cuda))
    for k in MAPS:
        a = ref[k].reshape(Ty, H, W).cpu().numpy()
        assert np.abs(a - z[k]).max() <= 1e-3 * np.abs(a).max(), k
