#!/usr/bin/env python
"""Training entry point with the reference's CLI (train.py:1204-1215):

    python train.py --config config/baseline [--set train.batch_size=4 ...]
    torchrun --standalone --nproc_per_node=8 train.py --config config/baseline

It builds the same `UNet` / `Diffusion` from the same config keys (train.py:669-680, 1021-1030), but
every step runs in cesm_emulator_b200.engine.TrainEngine: the sm_100a kernels, a CUDA graph per
step, and -- under torchrun -- a real bucketed NCCL gradient all-reduce overlapped with backward
(the reference's DDP wrapper is bypassed by its own `.module.loss` call; see DESIGN.md).
Data: the synthetic (member, time, lat, lon, channel) ensemble replaces the NetCDF files
(cesm_emulator_b200/synthetic.py).  Checkpoints use the reference's layout (train.py:1154-1165).
"""
import argparse
import os
import time

import torch
import torch.distributed as dist

from cesm_emulator_b200.engine import TrainEngine
from cesm_emulator_b200.model import Diffusion, UNet
from cesm_emulator_b200.synthetic import SyntheticEnsemble
from utils_conf import apply_overrides, load_config

UNET_KEYS = ("in_channels", "out_channels", "base_ch", "ch_mults", "num_res_blocks", "time_dim", "groups", "dropout",
             "use_checkpoint")


def build_model_from_config(ucfg: dict) -> UNet:
    """train.py:669-680: only these nine keys are forwarded; everything else takes UNet's default."""
    defaults = dict(in_channels=2, out_channels=1, base_ch=64, ch_mults=(1, 2, 4), num_res_blocks=2, time_dim=256,
                    groups=8, dropout=0.0, use_checkpoint=False)
    kw = {k: ucfg.get(k, defaults[k]) for k in UNET_KEYS}
    kw["ch_mults"] = tuple(kw["ch_mults"])
    return UNet(**kw)


def setup_distributed():
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    return int(os.environ.get("RANK", "0")), world, torch.device("cuda", local_rank)


def save_checkpoint(path, epoch, diffusion, engine, cfg):
    sd = diffusion.state_dict()
    ckpt = {
        "epoch": epoch,
        "model": {k[len("model."):]: v for k, v in sd.items() if k.startswith("model.")},
        "diffusion_buffers": {k: v for k, v in sd.items() if not k.startswith("model.")},
        "optimizer": engine.opt.state_dict(),
        "config": cfg,
    }
    if engine.has_ema:
        ckpt["ema"] = engine.ema_state_dict()  # UNet state-dict layout, like "model"
    if "grad_scaler" in ckpt["optimizer"]:  # GradScaler.state_dict() layout; the reference loads "scaler" if present (train.py:940-944)
        ckpt["scaler"] = dict(ckpt["optimizer"]["grad_scaler"])
    os.makedirs(os.path.dirname(path), exist_ok=True)
    torch.save(ckpt, path)


def prediction_type_from_config(cfg: dict) -> str:
    """diffusion.prediction_type of a run's config (or a checkpoint's "config"); absent means the reference's eps."""
    return (cfg or {}).get("diffusion", {}).get("prediction_type", "eps")


def load_checkpoint(path, diffusion, engine=None, device="cuda"):
    """train.py:915-946 semantics: strict=False on the UNet, buffers merged, start_epoch = epoch + 1.  An engine with a
    weight EMA loads the checkpoint's "ema", or restarts the EMA from the loaded weights if it has none.  A checkpoint
    whose config names another prediction_type than `diffusion`'s is an error: its weights predict another target."""
    ckpt = torch.load(path, map_location=device)
    saved = prediction_type_from_config(ckpt.get("config"))
    if saved != diffusion.prediction_type:
        raise ValueError(f"{path} was trained with diffusion.prediction_type={saved!r}; this run uses "
                         f"{diffusion.prediction_type!r}")
    missing, unexpected = diffusion.model.load_state_dict(ckpt["model"], strict=False)
    if missing or unexpected:
        print(f"[resume] missing={list(missing)} unexpected={list(unexpected)}")
    for k, v in ckpt.get("diffusion_buffers", {}).items():
        if hasattr(diffusion, k):
            getattr(diffusion, k).copy_(v.to(device))
    if engine is not None and "optimizer" in ckpt:
        engine.opt.load_state_dict(ckpt["optimizer"])
    if engine is not None and engine.has_ema:
        if "ema" in ckpt:
            engine.load_ema_state_dict(ckpt["ema"])
        else:
            engine.reset_ema()
            print(f"[resume] {path} has no \"ema\": the weight EMA starts from the loaded weights")
    return int(ckpt.get("epoch", 0)) + 1


def main(cfg):
    rank, world, dev = setup_distributed()
    tcfg, dcfg = cfg.get("train", {}), cfg.get("dataset", {})
    syn = cfg.get("data", {}).get("synthetic", {})
    K = int(dcfg.get("K", 3))
    crop = dcfg.get("crop_hw")
    ds = SyntheticEnsemble(members=syn.get("members", 34), times=syn.get("times", 251), lat=syn.get("lat", 192),
                           lon=syn.get("lon", 288), seed=syn.get("seed", 1234), K=K,
                           crop_hw=tuple(crop) if crop else None, time_reverse_p=float(dcfg.get("time_reverse_p", 0.5)))
    B = int(tcfg.get("batch_size", 2))
    h, w = (crop if crop else (ds.H, ds.W))
    torch.manual_seed(0)
    diffusion = Diffusion(build_model_from_config(cfg.get("unet", {})),
                          timesteps=cfg.get("diffusion", {}).get("timesteps", 1000),
                          beta_schedule=cfg.get("diffusion", {}).get("beta_schedule", "linear"),
                          prediction_type=prediction_type_from_config(cfg)).to(dev)
    diffusion.train()
    opt = tcfg.get("optimizer", {})
    engine = TrainEngine(diffusion, (B, 1, h, w), (B, 1, K, h, w), lr=opt.get("lr", 2e-4),
                         betas=tuple(opt.get("betas", (0.9, 0.999))), weight_decay=opt.get("weight_decay", 1e-4),
                         max_grad_norm=tcfg.get("max_grad_norm", 1.0), ema_decay=tcfg.get("ema_decay"),
                         ema_start=tcfg.get("ema_start", 0), min_snr_gamma=tcfg.get("min_snr_gamma"))
    start = 1
    if tcfg.get("resume") and os.path.exists(tcfg["resume"]):
        start = load_checkpoint(tcfg["resume"], diffusion, engine, dev)
    save_dir = tcfg.get("save_dir", "runs/exp")
    max_steps = int(tcfg.get("max_steps_per_epoch", 0))
    # data.on_device (default on): both arrays resident in HBM, batches gathered by one kernel
    dev_ds = ds.to_device(dev) if cfg.get("data", {}).get("on_device", True) else None
    for epoch in range(start, int(tcfg.get("num_epochs", 1)) + 1):
        idx = ds.shard_indices(epoch, rank, world)
        n_steps = len(idx) // B if not max_steps else min(max_steps, len(idx) // B)
        t0, total = time.time(), torch.zeros((), device=dev)
        for s in range(n_steps):
            if dev_ds is not None:
                loss = engine.step_indices(dev_ds, idx[s * B:(s + 1) * B])
            else:
                cond, x0 = ds.batch(idx[s * B:(s + 1) * B], pin=True)
                loss = engine.step(x0, cond)
            total += loss
        mean = (total / max(1, n_steps)).item()  # one host sync per epoch, not per step
        if not (mean == mean and abs(mean) != float("inf")):
            raise RuntimeError(f"Non-finite loss at epoch {epoch}: {mean}")  # train.py:860-861
        if rank == 0:
            dt = time.time() - t0
            st = engine.opt.state.tolist()
            print(f"epoch {epoch}: loss {mean:.5f}  {n_steps * B * world / dt:.1f} samples/s ({world} GPU)  "
                  f"loss scale {st[2]:.0f}, {int(st[5])} skipped step(s)")
            if epoch % int(tcfg.get("save_every", 10)) == 0:
                save_checkpoint(os.path.join(save_dir, "checkpoints", f"ckpt_epoch_{epoch}.pt"), epoch, diffusion,
                                engine, cfg)
    if rank == 0:
        save_checkpoint(os.path.join(save_dir, "checkpoints", "final.pt"), epoch, diffusion, engine, cfg)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", required=True)
    ap.add_argument("--set", nargs="*", default=[])
    a = ap.parse_args()
    cfg = load_config(a.config)
    apply_overrides(cfg, a.set)
    main(cfg)
