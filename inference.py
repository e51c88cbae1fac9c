#!/usr/bin/env python
"""Ensemble generation entry point (reference: inference.py:174-284).

    python inference.py --ckpt runs/exp/checkpoints/final.pt [--batch_size 16] [--steps 1000] [--out pred.npy | pred.nc]
    python inference.py --ckpt ... --ddim_steps 50 [--eta 0.0]     # strided DDIM chain: 50 UNet calls per field
    python inference.py --ckpt ... --dpm_steps 15                  # DPM-Solver++(2M) chain: 15 UNet calls per field
    python inference.py --ckpt ... --ema [--dpm_steps 15]          # sample from the weight EMA (ckpt["ema"])
    python inference.py --ckpt ... --seed 7                        # counter-based noise: same fields on any world size
    torchrun --standalone --nproc_per_node=8 inference.py --ckpt ...

`predict_temperature_from_emissions` keeps the reference's flow: rebuild UNet/Diffusion from
ckpt["config"], flatten the condition (T, M, 1, H, W) -> (N, 1, H, W), and run the full reverse chain
per batch of independent fields (inference.py:217-232).  Here each chain step is one CUDA-graph replay
(cesm_emulator_b200.engine.SampleEngine) and, under torchrun, the N fields are sharded over ranks.
Condition data comes from the synthetic ensemble; output is a (T, M, H, W) float32 array, written as .npy or
-- `--out x.nc` -- as the reference's NetCDF product (`TREFHT_pred`, inference.py:260-281) in classic NetCDF-3
through scipy (xarray / netCDF4 are not in this image).
"""
import argparse
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

from cesm_emulator_b200.engine import SampleEngine
from cesm_emulator_b200.model import Diffusion
from cesm_emulator_b200.synthetic import SyntheticEnsemble
from train import build_model_from_config, prediction_type_from_config


def load_diffusion_from_checkpoint(path, device, ema=False):
    """inference.py:47-75.  With `ema=True` the UNet gets the checkpoint's weight EMA (ckpt["ema"], written by a run
    with train.ema_decay set) instead of its raw weights (ckpt["model"]); a checkpoint without one is an error.  The
    Diffusion predicts the target the run trained (diffusion.prediction_type in ckpt["config"], eps when absent)."""
    ckpt = torch.load(path, map_location=device)
    if ema and "ema" not in ckpt:
        raise KeyError(f'{path} has no "ema" entry: it was not trained with train.ema_decay set '
                       f'(load it without ema=True / --ema to sample from its raw weights)')
    cfg = ckpt["config"]
    diffusion = Diffusion(build_model_from_config(cfg.get("unet", {})),
                          timesteps=cfg.get("diffusion", {}).get("timesteps", 1000),
                          prediction_type=prediction_type_from_config(cfg)).to(device)
    missing, unexpected = diffusion.model.load_state_dict(ckpt["ema" if ema else "model"], strict=False)
    if missing or unexpected:
        print(f"[load] missing={list(missing)} unexpected={list(unexpected)}")
    diffusion.eval()
    for p in diffusion.parameters():
        p.requires_grad_(False)
    return diffusion, cfg


@torch.no_grad()
def predict_temperature_from_emissions(diffusion, cond_tm1hw: np.ndarray, batch_size=16, steps=None, rank=0, world=1,
                                       device="cuda", ddim_steps=None, eta=0.0, dpm_steps=None, seed=None):
    """cond (T, M, 1, H, W) -> prediction (T, M, H, W); fields are independent and sharded over ranks.
    `ddim_steps=N` generates with the strided DDIM chain (N UNet calls per field, noise scaled by `eta`) instead of
    the full DDPM chain; it cannot be combined with `steps`.  `dpm_steps=N` generates with the deterministic
    DPM-Solver++(2M) chain (N UNet calls per field); it cannot be combined with `steps`, `ddim_steps` or eta != 0.

    With `seed` (an int in [0, 2^64)) the noise of (year index t, member m) is drawn from the field id (t << 32) | m,
    so the prediction does not depend on `batch_size`, on the number of ranks or on --times / --members, up to
    run-to-run rounding.  Without it every rank draws from torch's CUDA generator, whose default seed is the same on
    every process."""
    if ddim_steps is not None and steps is not None:
        raise ValueError("steps and ddim_steps are mutually exclusive")
    if dpm_steps is not None and (steps is not None or ddim_steps is not None):
        raise ValueError("dpm_steps cannot be combined with steps or ddim_steps")
    if dpm_steps is not None and eta != 0:
        raise ValueError(f"eta applies to DDIM only; dpm_steps is deterministic (got eta={eta})")
    T, M, _, H, W = cond_tm1hw.shape
    if seed is None and world > 1 and rank == 0:
        print(f"inference: the {world} ranks share one noise stream, so members can coincide; --seed gives every "
              "field its own noise", file=sys.stderr)
    flat = torch.from_numpy(cond_tm1hw.reshape(T * M, 1, H, W))
    mine = list(range(rank, T * M, world))
    out = torch.zeros((T * M, 1, H, W), dtype=torch.float32)
    eng = None
    for i in range(0, len(mine), batch_size):
        sel = mine[i:i + batch_size]
        c = flat[sel]
        if c.shape[0] < batch_size:  # keep the captured graph's static shape
            c = torch.cat([c, c[-1:].expand(batch_size - c.shape[0], -1, -1, -1)], 0)
        if eng is None:
            eng = SampleEngine(diffusion, (batch_size, 1, H, W), ddim_steps=ddim_steps, eta=eta, dpm_steps=dpm_steps,
                               seed=seed)
        ids = None
        if seed is not None:  # padding rows repeat the last real field
            ids = [((k // M) << 32) | (k % M) for k in sel]
            ids = torch.tensor(ids + ids[-1:] * (batch_size - len(sel)), dtype=torch.int64)
        y = eng.sample(c.to(device), steps=steps, field_ids=ids)
        out[sel] = y[: len(sel)].cpu()
    if world > 1:
        out = out.to(device)
        dist.all_reduce(out)  # disjoint shards: sum == gather
        out = out.cpu()
    return out.reshape(T, M, H, W).numpy()


def write_prediction_netcdf(path, pred_tmhw: np.ndarray, stack_coord=None, member_coord=None, lat=None, lon=None,
                            stack_dim="year", member_dim="member_id", lat_name="lat", lon_name="lon", attrs=None):
    """The reference's output product (inference.py:239-281): variable `TREFHT_pred` with dims
    (year, member_id, lat, lon), coordinate variables and the description / units attributes.  xarray and
    netCDF4 are not in this image, so the file is written as classic NetCDF-3 by scipy
    (`xr.open_dataset` reads it with its scipy engine)."""
    T, M, H, W = pred_tmhw.shape
    coords = [(stack_dim, stack_coord, T), (member_dim, member_coord, M), (lat_name, lat, H), (lon_name, lon, W)]
    write_netcdf_variable(path, "TREFHT_pred", pred_tmhw, coords, {
        "description": "Predicted near-surface air temperature from emissions via diffusion model",
        "units": "standardized", **(attrs or {})})


def write_netcdf_variable(path, name, data, coords, attrs):
    """One float32 variable `name` over the dimensions `coords` = [(dim name, coordinate values or None for
    arange, length), ...] with its coordinate variables and attributes, as classic NetCDF-3 through scipy."""
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


def _parse_args(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--ckpt", required=True)
    ap.add_argument("--batch_size", type=int, default=16)
    ap.add_argument("--steps", type=int, default=None, help="reverse steps (default: all T)")
    ap.add_argument("--ddim_steps", type=int, default=None,
                    help="generate with a strided DDIM chain of this many UNet calls instead of the T-step DDPM chain")
    ap.add_argument("--eta", type=float, default=0.0, help="DDIM noise scale (0 = deterministic, 1 = DDPM-like)")
    ap.add_argument("--dpm_steps", type=int, default=None,
                    help="generate with a deterministic DPM-Solver++(2M) chain of this many UNet calls")
    ap.add_argument("--ema", action="store_true",
                    help='generate from the weight EMA stored in the checkpoint ("ema") instead of its raw weights')
    ap.add_argument("--seed", type=int, default=None,
                    help="draw every field's noise from (seed, year, member), in [0, 2**64): the output then does not "
                         "depend on --batch_size or the number of GPUs")
    ap.add_argument("--members", type=int, default=2)
    ap.add_argument("--times", type=int, default=4)
    ap.add_argument("--out", default="pred.npy")
    a = ap.parse_args(argv)
    if a.steps is not None and a.ddim_steps is not None:
        ap.error("--steps and --ddim_steps are mutually exclusive")
    if a.dpm_steps is not None and (a.steps is not None or a.ddim_steps is not None):
        ap.error("--dpm_steps cannot be combined with --steps or --ddim_steps")
    if a.dpm_steps is not None and a.eta != 0:
        ap.error("--eta applies to --ddim_steps only; --dpm_steps is deterministic")
    if a.seed is not None and not 0 <= a.seed < 1 << 64:
        ap.error(f"--seed must be in [0, 2**64), got {a.seed}")
    return a


def _cli():
    a = _parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank, local = int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    try:
        diffusion, cfg = load_diffusion_from_checkpoint(a.ckpt, dev, ema=a.ema)
    except KeyError as e:
        raise SystemExit(f"inference.py: error: {e.args[0]}")
    syn = cfg.get("data", {}).get("synthetic", {})
    ds = SyntheticEnsemble(members=a.members, times=a.times, lat=syn.get("lat", 192), lon=syn.get("lon", 288),
                           seed=syn.get("seed", 1234))
    pred = predict_temperature_from_emissions(diffusion, ds.cond, a.batch_size, a.steps, rank, world, dev,
                                              ddim_steps=a.ddim_steps, eta=a.eta, dpm_steps=a.dpm_steps, seed=a.seed)
    if rank == 0:
        if a.out.endswith(".nc"):
            write_prediction_netcdf(a.out, pred, attrs={"checkpoint": os.path.abspath(a.ckpt), "cond_var": "synthetic"})
        else:
            np.save(a.out, pred)
        print(f"wrote {a.out} {pred.shape}")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    _cli()
