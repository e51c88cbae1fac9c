#!/usr/bin/env python
"""Score a trained emulator's ensembles against the target ensemble of the synthetic data it was trained on.

    python evaluate.py --ckpt runs/exp/checkpoints/final.pt [--ema] [--ddim_steps N [--eta E] | --dpm_steps N |
                       --steps S] [--seed S] [--guidance w] [--batch_size 16] [--years START:STOP[:STEP]]
                       [--out scores.nc | scores.npz]
    torchrun --standalone --nproc_per_node=8 evaluate.py --ckpt ...

The synthetic ensemble is rebuilt exactly as train.py built it, from the checkpoint's data.synthetic block (members,
times, lat, lon, seed).  For the selected years the emulator generates one field per (year, member) -- so the
generated and the target ensembles both have n = m = members -- through `predict_temperature_from_emissions` (sharded
over ranks under torchrun; with --seed, field (t, m) of the selected years draws from the id (t << 32) | m, t counted
from the first selected year).  Rank 0 then scores it against the targets in one kernel pass
(`kernels.ensemble_scores`): per (year, pixel) the fair CRPS, bias, the two spreads and the ensemble-mean squared
error, and per year the rank histogram.  It also scores an ideal ensemble, n members drawn from the known truth
N(target_mean, target_noise_std^2), against the same targets, and prints both rows.

Output: the five maps over (year, lat, lon), `rank_hist` over (year, rank) and the per-year summaries over (year),
as NetCDF-3 (`.nc`, the sampler flags, checkpoint and seed as global attributes) or as `.npz`.
"""
import argparse
import json
import math
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

from cesm_emulator_b200 import kernels as K
from cesm_emulator_b200.synthetic import SyntheticEnsemble
from inference import (add_sampler_args, check_guidance_for_config, check_sampler_args, load_diffusion_from_checkpoint,
                       predict_temperature_from_emissions, write_netcdf_variables)

SUMMARY_KEYS = ("crps", "bias", "rmse", "spread", "ssr", "nonfinite")


def summarize_scores(scores: dict, n: int) -> dict:
    """Per-year and overall summaries of `kernels.ensemble_scores` output for n predicted members: plain means over
    the finite pixels (no area weighting) of the CRPS and the bias; the RMSE of the ensemble mean, sqrt(mean mse_mean);
    the spread, sqrt(mean sd_pred^2); the spread-skill ratio sqrt((n+1)/n) * spread / RMSE (1 for a calibrated
    ensemble); the rank histogram normalised to frequencies; the number of non-finite columns; and, overall, the chi^2
    statistic of the rank histogram against a flat one (descriptive only: the counts of one column share its X, so
    they are not independent and the statistic has no p-value).
    -> {"year": {key: [T] tensor, "rank_freq": [T, n+1]}, "overall": {key: float, "rank_freq": [n+1], "chi2": float}}"""
    finite = torch.isfinite(scores["crps"])  # a non-finite column is NaN in every map

    def means(x):
        x = torch.where(finite, x.double(), 0.0)
        return x.sum(1) / finite.sum(1), x.sum() / finite.sum()

    def group(crps, bias, mse, var, nonfinite, hist):
        rmse, spread = mse.sqrt(), var.sqrt()
        return {"crps": crps, "bias": bias, "rmse": rmse, "spread": spread,
                "ssr": math.sqrt((n + 1) / n) * spread / rmse, "nonfinite": nonfinite,
                "rank_freq": hist.double() / hist.sum(-1, keepdim=True)}

    (crps_t, crps), (bias_t, bias) = means(scores["crps"]), means(scores["bias"])
    (mse_t, mse), (var_t, var) = means(scores["mse_mean"]), means(scores["sd_pred"].double() ** 2)
    hist = scores["rank_hist"]
    year = group(crps_t, bias_t, mse_t, var_t, (~finite).sum(1), hist)
    total = hist.sum(0)
    overall = {k: float(v) for k, v in group(crps, bias, mse, var, (~finite).sum(), total).items() if k != "rank_freq"}
    overall["rank_freq"] = total.double() / total.sum()
    expect = total.sum().double() / (n + 1)
    overall["chi2"] = float(((total.double() - expect) ** 2 / expect).sum())
    return {"year": year, "overall": overall}


def parse_years(text: str) -> slice:
    """START:STOP[:STEP] with integers, STOP > START >= 0 and STEP >= 1 -> slice."""
    parts = text.split(":")
    if len(parts) not in (2, 3):
        raise ValueError(f"--years must be START:STOP[:STEP], got {text!r}")
    try:
        start, stop, step = int(parts[0]), int(parts[1]), int(parts[2]) if len(parts) == 3 else 1
    except ValueError:
        raise ValueError(f"--years must hold integers, got {text!r}") from None
    if not (0 <= start < stop and step >= 1):
        raise ValueError(f"--years needs 0 <= START < STOP and STEP >= 1, got {text!r}")
    return slice(start, stop, step)


def _parse_args(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--ckpt", required=True)
    ap.add_argument("--batch_size", type=int, default=16)
    add_sampler_args(ap)
    ap.add_argument("--years", default=None,
                    help="START:STOP[:STEP]: the years of the synthetic ensemble to score (default: all)")
    ap.add_argument("--out", default="scores.npz", help="scores.nc (NetCDF-3) or scores.npz")
    a = ap.parse_args(argv)
    check_sampler_args(ap, a)
    if a.batch_size < 1:
        ap.error(f"--batch_size must be >= 1, got {a.batch_size}")
    if a.years is not None:
        try:
            a.years = parse_years(a.years)
        except ValueError as e:
            ap.error(str(e))
    if not (a.out.endswith(".nc") or a.out.endswith(".npz")):
        ap.error(f"--out must end in .nc or .npz, got {a.out!r}")
    return a


def _row(name, o):
    return (f"{name:<8}{o['crps']:>10.5f}{o['bias']:>+11.5f}{o['rmse']:>10.5f}{o['spread']:>10.5f}{o['ssr']:>8.4f}"
            f"{o['chi2']:>14.1f}{int(o['nonfinite']):>11d}")


def main(argv=None):
    a = _parse_args(argv)
    try:  # on the host first: a missing EMA or an unusable guidance weight is reported before any device work
        diffusion, cfg = load_diffusion_from_checkpoint(a.ckpt, "cpu", ema=a.ema)
        guidance = check_guidance_for_config(a.guidance, cfg)
    except (KeyError, ValueError) as e:
        raise SystemExit(f"evaluate.py: error: {e.args[0]}")
    syn = cfg.get("data", {}).get("synthetic", {})
    # train.py's defaults: another `times` is another synthetic world, so nothing here may differ from training
    members, times = syn.get("members", 34), syn.get("times", 251)
    years = a.years or slice(0, times)
    sel = np.arange(times)[years]
    if years.stop > times or sel.size == 0:
        raise SystemExit(f"evaluate.py: error: --years {years.start}:{years.stop}:{years.step} is outside the "
                         f"{times} years of the checkpoint's synthetic ensemble")
    if not torch.cuda.is_available():
        raise SystemExit("evaluate.py: error: generation and scoring need a CUDA device")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank, local = int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    diffusion = diffusion.to(dev)
    ds = SyntheticEnsemble(members=members, times=times, lat=syn.get("lat", 192), lon=syn.get("lon", 288),
                           seed=syn.get("seed", 1234))
    pred = predict_temperature_from_emissions(diffusion, np.ascontiguousarray(ds.cond[sel]), a.batch_size, a.steps,
                                              rank, world, dev, ddim_steps=a.ddim_steps, eta=a.eta,
                                              dpm_steps=a.dpm_steps, seed=a.seed, guidance=guidance)
    if rank == 0:
        Ty, n, H, W = pred.shape
        tgt = torch.from_numpy(ds.tgt[sel].reshape(Ty, n, H * W)).to(dev)
        scores = K.ensemble_scores(torch.from_numpy(pred.reshape(Ty, n, H * W)).to(dev), tgt)
        summary = summarize_scores(scores, n)
        g = torch.Generator().manual_seed(0 if a.seed is None else a.seed)
        ideal = (torch.from_numpy(ds.target_mean[sel]).reshape(Ty, 1, H * W)
                 + ds.target_noise_std * torch.randn((Ty, n, H * W), generator=g))
        ideal_summary = summarize_scores(K.ensemble_scores(ideal.to(dev), tgt), n)["overall"]
        print(f"{Ty} years x {n} members, {H}x{W}, scored against the {n} target members")
        print(f"{'':<8}{'CRPS':>10}{'bias':>11}{'RMSE':>10}{'spread':>10}{'SSR':>8}{'rank chi2':>14}{'non-finite':>11}")
        print(_row("model", summary["overall"]))
        print(_row("ideal", ideal_summary))
        sampler = ("dpm" if a.dpm_steps is not None else "ddim" if a.ddim_steps is not None else "ddpm")
        attrs = {"checkpoint": os.path.abspath(a.ckpt), "ema": int(a.ema), "sampler": sampler,
                 "steps": -1 if a.steps is None else a.steps, "ddim_steps": -1 if a.ddim_steps is None else a.ddim_steps,
                 "eta": float(a.eta), "dpm_steps": -1 if a.dpm_steps is None else a.dpm_steps,
                 "guidance": float(guidance), "seed": "none" if a.seed is None else str(a.seed),
                 **{f"overall_{k}": float(summary["overall"][k]) for k in (*SUMMARY_KEYS, "chi2")},
                 **{f"ideal_{k}": float(ideal_summary[k]) for k in (*SUMMARY_KEYS, "chi2")}}
        maps = {k: scores[k].reshape(Ty, H, W).cpu().numpy() for k in K.SCORE_MAPS}
        arrays = {**maps, "rank_hist": scores["rank_hist"].cpu().numpy().astype(np.int32),
                  **{f"{k}_year": summary["year"][k].cpu().numpy() for k in (*SUMMARY_KEYS, "rank_freq")}}
        if a.out.endswith(".nc"):
            dims = [("year", sel, Ty), ("lat", None, H), ("lon", None, W), ("rank", None, n + 1)]
            variables = [(k, v, ("year", "lat", "lon"), {}) for k, v in maps.items()]
            variables += [("rank_hist", arrays["rank_hist"], ("year", "rank"), {})]
            variables += [(f"{k}_year", arrays[f"{k}_year"], ("year",), {}) for k in SUMMARY_KEYS]
            variables += [("rank_freq_year", arrays["rank_freq_year"], ("year", "rank"), {})]
            write_netcdf_variables(a.out, dims, variables, attrs)
        else:
            d = os.path.dirname(a.out)
            if d:
                os.makedirs(d, exist_ok=True)
            np.savez(a.out, year=sel, **arrays, attrs=json.dumps(attrs))
        print(f"wrote {a.out}")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main(sys.argv[1:])
