#!/usr/bin/env python
"""Emission saliency entry point: how sensitive a trained emulator's denoising loss is to each pixel and frame of
the CO2-emission window (the reference's XAI helpers, which take d loss / d cond through q_sample and the UNet).

    python saliency.py --ckpt runs/exp/checkpoints/final.pt [--ema] [--draws 16] [--seed S] [--batch_size 8]
                       [--members 2] [--times 8] --out sal.npy | sal.nc
    torchrun --standalone --nproc_per_node=8 saliency.py --ckpt ...

For every (window t0, member m) of the synthetic ensemble -- sample index t0 * M + m, the target field and its
K-frame emission window -- the map is `SaliencyEngine`'s: the gradient of the field's own denoising MSE with
respect to its condition, averaged over `--draws` stratified timesteps with fresh noise each.  With `--seed` the
noise of (t0, m) comes from the field id (t0 << 32) | m, so a map does not depend on --batch_size or the number of
ranks.  Output: (windows, M, K, H, W) float32 as .npy, or -- `--out x.nc` -- the NetCDF variable `saliency`.
"""
import argparse
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

from cesm_emulator_b200.engine import SaliencyEngine
from cesm_emulator_b200.synthetic import SyntheticEnsemble
from inference import load_diffusion_from_checkpoint, write_netcdf_variable


def compute_saliency(diffusion, ds: SyntheticEnsemble, batch_size=8, draws=16, seed=None, rank=0, world=1,
                     device="cuda") -> np.ndarray:
    """Saliency of every (window, member) of `ds` -> (windows, M, K, H, W); indices are sharded over ranks."""
    M, Kf, H, W = ds.M, ds.K, ds.H, ds.W
    windows = ds.T - Kf + 1
    if windows < 1:
        raise ValueError(f"the ensemble has {ds.T} times, fewer than the window length K={Kf}")
    N = windows * M
    mine = list(range(rank, N, world))
    out = torch.zeros((N, Kf, H, W), dtype=torch.float32)
    eng = None
    for i in range(0, len(mine), batch_size):
        sel = mine[i:i + batch_size]
        cond, x0 = ds.batch(sel, augment=False)
        pad = batch_size - len(sel)
        if pad:  # keep the captured graph's static shape: padding rows repeat the last real field
            cond = torch.cat([cond, cond[-1:].expand(pad, -1, -1, -1, -1)], 0)
            x0 = torch.cat([x0, x0[-1:].expand(pad, -1, -1, -1)], 0)
        if eng is None:
            eng = SaliencyEngine(diffusion, tuple(x0.shape), tuple(cond.shape), draws=draws, seed=seed)
        ids = None
        if seed is not None:
            ids = [((k // M) << 32) | (k % M) for k in sel]
            ids = torch.tensor(ids + ids[-1:] * pad, dtype=torch.int64)
        s = eng.saliency(x0.to(device), cond.to(device), field_ids=ids)
        out[sel] = s[:len(sel), 0].cpu()
    if world > 1:
        out = out.to(device)
        dist.all_reduce(out)  # disjoint shards: sum == gather
        out = out.cpu()
    return out.reshape(windows, M, Kf, H, W).numpy()


def write_saliency_netcdf(path, sal_wmkhw: np.ndarray, window_coord=None, member_coord=None, lat=None, lon=None,
                          attrs=None):
    """Variable `saliency` with dims (window, member_id, frame, lat, lon) and coordinate variables, as classic
    NetCDF-3 (see inference.write_prediction_netcdf)."""
    Wn, M, Kf, H, W = sal_wmkhw.shape
    coords = [("window", window_coord, Wn), ("member_id", member_coord, M), ("frame", None, Kf), ("lat", lat, H),
              ("lon", lon, W)]
    write_netcdf_variable(path, "saliency", sal_wmkhw, coords, {
        "description": "d(denoising MSE of the field)/d(emission condition), averaged over diffusion draws",
        "units": "per standardized condition unit", **(attrs or {})})


def _parse_args(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--ckpt", required=True)
    ap.add_argument("--ema", action="store_true",
                    help='use the weight EMA stored in the checkpoint ("ema") instead of its raw weights')
    ap.add_argument("--draws", type=int, default=16, help="stratified timesteps (with fresh noise) averaged per map")
    ap.add_argument("--seed", type=int, default=None,
                    help="draw every field's noise from (seed, window, member), in [0, 2**64): the maps then do not "
                         "depend on --batch_size or the number of GPUs")
    ap.add_argument("--batch_size", type=int, default=8)
    ap.add_argument("--members", type=int, default=2)
    ap.add_argument("--times", type=int, default=8)
    ap.add_argument("--out", default="sal.npy")
    a = ap.parse_args(argv)
    if a.draws < 1:
        ap.error(f"--draws must be >= 1, got {a.draws}")
    if a.seed is not None and not 0 <= a.seed < 1 << 64:
        ap.error(f"--seed must be in [0, 2**64), got {a.seed}")
    if a.batch_size < 1:
        ap.error(f"--batch_size must be >= 1, got {a.batch_size}")
    return a


def main(argv=None):
    a = _parse_args(argv)
    try:  # on the host first: a missing EMA is reported before any device work
        diffusion, cfg = load_diffusion_from_checkpoint(a.ckpt, "cpu", ema=a.ema)
    except KeyError as e:
        raise SystemExit(f"saliency.py: error: {e.args[0]}")
    if not torch.cuda.is_available():
        raise SystemExit("saliency.py: error: the saliency kernels need a CUDA device")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank, local = int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    diffusion = diffusion.to(dev)
    syn = cfg.get("data", {}).get("synthetic", {})
    ds = SyntheticEnsemble(members=a.members, times=a.times, lat=syn.get("lat", 192), lon=syn.get("lon", 288),
                           seed=syn.get("seed", 1234), K=cfg.get("dataset", {}).get("K", 3))
    try:
        sal = compute_saliency(diffusion, ds, a.batch_size, a.draws, a.seed, rank, world, dev)
    except ValueError as e:
        raise SystemExit(f"saliency.py: error: {e}")
    if rank == 0:
        if a.out.endswith(".nc"):
            write_saliency_netcdf(a.out, sal, attrs={
                "checkpoint": os.path.abspath(a.ckpt), "cond_var": "synthetic",
                "draws": int(a.draws), "seed": "none" if a.seed is None else str(a.seed), "ema": int(a.ema)})
        else:
            np.save(a.out, sal)
        print(f"wrote {a.out} {sal.shape}")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main(sys.argv[1:])
