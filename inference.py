#!/usr/bin/env python
"""Ensemble generation entry point (reference: inference.py:174-284).

    python inference.py --ckpt runs/exp/checkpoints/final.pt [--batch_size 16] [--steps 1000] [--out pred.npy | pred.nc]
    python inference.py --ckpt ... --ddim_steps 50 [--eta 0.0]     # strided DDIM chain: 50 UNet calls per field
    python inference.py --ckpt ... --dpm_steps 15                  # DPM-Solver++(2M) chain: 15 UNet calls per field
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

import numpy as np
import torch
import torch.distributed as dist

from cesm_emulator_b200.engine import SampleEngine
from cesm_emulator_b200.model import Diffusion
from cesm_emulator_b200.synthetic import SyntheticEnsemble
from train import build_model_from_config


def load_diffusion_from_checkpoint(path, device):
    """inference.py:47-75."""
    ckpt = torch.load(path, map_location=device)
    cfg = ckpt["config"]
    diffusion = Diffusion(build_model_from_config(cfg.get("unet", {})),
                          timesteps=cfg.get("diffusion", {}).get("timesteps", 1000)).to(device)
    missing, unexpected = diffusion.model.load_state_dict(ckpt["model"], strict=False)
    if missing or unexpected:
        print(f"[load] missing={list(missing)} unexpected={list(unexpected)}")
    diffusion.eval()
    for p in diffusion.parameters():
        p.requires_grad_(False)
    return diffusion, cfg


@torch.no_grad()
def predict_temperature_from_emissions(diffusion, cond_tm1hw: np.ndarray, batch_size=16, steps=None, rank=0, world=1,
                                       device="cuda", ddim_steps=None, eta=0.0, dpm_steps=None):
    """cond (T, M, 1, H, W) -> prediction (T, M, H, W); fields are independent and sharded over ranks.
    `ddim_steps=N` generates with the strided DDIM chain (N UNet calls per field, noise scaled by `eta`) instead of
    the full DDPM chain; it cannot be combined with `steps`.  `dpm_steps=N` generates with the deterministic
    DPM-Solver++(2M) chain (N UNet calls per field); it cannot be combined with `steps`, `ddim_steps` or eta != 0."""
    if ddim_steps is not None and steps is not None:
        raise ValueError("steps and ddim_steps are mutually exclusive")
    if dpm_steps is not None and (steps is not None or ddim_steps is not None):
        raise ValueError("dpm_steps cannot be combined with steps or ddim_steps")
    if dpm_steps is not None and eta != 0:
        raise ValueError(f"eta applies to DDIM only; dpm_steps is deterministic (got eta={eta})")
    T, M, _, H, W = cond_tm1hw.shape
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
            eng = SampleEngine(diffusion, (batch_size, 1, H, W), ddim_steps=ddim_steps, eta=eta, dpm_steps=dpm_steps)
        y = eng.sample(c.to(device), steps=steps)
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
    from scipy.io import netcdf_file
    T, M, H, W = pred_tmhw.shape
    coords = [(stack_dim, stack_coord, T), (member_dim, member_coord, M), (lat_name, lat, H), (lon_name, lon, W)]
    d = os.path.dirname(path)
    if d:
        os.makedirs(d, exist_ok=True)
    with netcdf_file(path, "w", version=2) as f:
        for name, vals, n in coords:
            f.createDimension(name, n)
            vals = np.arange(n) if vals is None else np.asarray(vals)
            if vals.shape != (n,):
                raise ValueError(f"coordinate {name} has shape {vals.shape}, expected ({n},)")
            vals = vals.astype(np.float64 if vals.dtype.kind == "f" else np.int32)
            v = f.createVariable(name, vals.dtype, (name,))
            v[:] = vals
        v = f.createVariable("TREFHT_pred", np.float32, (stack_dim, member_dim, lat_name, lon_name))
        v[:] = np.asarray(pred_tmhw, dtype=np.float32)
        v.description = "Predicted near-surface air temperature from emissions via diffusion model"
        v.units = "standardized"
        for k, val in (attrs or {}).items():
            setattr(v, k, val)


def _cli():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ckpt", required=True)
    ap.add_argument("--batch_size", type=int, default=16)
    ap.add_argument("--steps", type=int, default=None, help="reverse steps (default: all T)")
    ap.add_argument("--ddim_steps", type=int, default=None,
                    help="generate with a strided DDIM chain of this many UNet calls instead of the T-step DDPM chain")
    ap.add_argument("--eta", type=float, default=0.0, help="DDIM noise scale (0 = deterministic, 1 = DDPM-like)")
    ap.add_argument("--dpm_steps", type=int, default=None,
                    help="generate with a deterministic DPM-Solver++(2M) chain of this many UNet calls")
    ap.add_argument("--members", type=int, default=2)
    ap.add_argument("--times", type=int, default=4)
    ap.add_argument("--out", default="pred.npy")
    a = ap.parse_args()
    if a.steps is not None and a.ddim_steps is not None:
        ap.error("--steps and --ddim_steps are mutually exclusive")
    if a.dpm_steps is not None and (a.steps is not None or a.ddim_steps is not None):
        ap.error("--dpm_steps cannot be combined with --steps or --ddim_steps")
    if a.dpm_steps is not None and a.eta != 0:
        ap.error("--eta applies to --ddim_steps only; --dpm_steps is deterministic")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank, local = int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    diffusion, cfg = load_diffusion_from_checkpoint(a.ckpt, dev)
    syn = cfg.get("data", {}).get("synthetic", {})
    ds = SyntheticEnsemble(members=a.members, times=a.times, lat=syn.get("lat", 192), lon=syn.get("lon", 288),
                           seed=syn.get("seed", 1234))
    pred = predict_temperature_from_emissions(diffusion, ds.cond, a.batch_size, a.steps, rank, world, dev,
                                              ddim_steps=a.ddim_steps, eta=a.eta, dpm_steps=a.dpm_steps)
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
