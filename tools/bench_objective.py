#!/usr/bin/env python
"""Cost of the training objectives and of v-prediction sampling, on config/baseline's UNet over the 192x288 grid.

Training: one TrainEngine step at bench.py's shape (B = 2, K = 3) for the eps target (the reference's MSE), the v
target, and the v target with Min-SNR-gamma weights (gamma = 5).  Sampling: one DDPM SampleEngine step for 16
one-frame fields, eps (p_sample) against v (ddim_step with the folded N = T, eta = 1 table).  Each step is a CUDA-graph
replay timed with CUDA events; the modes of a group are alternated segment by segment in the same process, and every
engine's `launches_per_step` is recorded.  The card's name, power limit and max SM clock are read in the same run.

    python tools/bench_objective.py [--segments 5] [--steps 20] [--out profiles/x.json]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def _diffusion(cfg, prediction_type):
    import train as train_entry
    from cesm_emulator_b200.model import Diffusion
    torch.manual_seed(0)
    return Diffusion(train_entry.build_model_from_config(cfg["unet"]), prediction_type=prediction_type).cuda()


def _ms(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def train_modes(cfg, segments, steps):
    from cesm_emulator_b200 import ops
    from cesm_emulator_b200.engine import TrainEngine
    B, K, H, W = 2, 3, 192, 288
    g = torch.Generator().manual_seed(0)
    x0, cond = torch.randn(B, 1, H, W, generator=g).cuda(), torch.randn(B, 1, K, H, W, generator=g).cuda()
    engines = {}
    for name, pt, gamma in (("eps", "eps", None), ("v", "v", None), ("v_minsnr5", "v", 5.0)):
        d = _diffusion(cfg, pt)
        d.train()
        engines[name] = TrainEngine(d, x0.shape, cond.shape, min_snr_gamma=gamma)
    # every model runs its eager warm-up steps before the first capture, so that all three graphs record the same
    # weight-pack plan (ops.prepack_all) and none is rebuilt under a captured graph
    for _ in range(3):  # two eager warm-up steps, then the capture
        for eng in engines.values():
            eng.step(x0, cond)
    torch.cuda.synchronize()
    ms = {n: [] for n in engines}
    for _ in range(segments):
        for n, eng in engines.items():
            ms[n].append(_ms(eng.step_resident, steps))
    ops.set_grad_sink(None)
    return {"B": B, "frames": K, "H": H, "W": W, "ms_per_step": ms,
            "launches_per_step": {n: e.launches_per_step for n, e in engines.items()},
            "loss": {n: float(e.loss) for n, e in engines.items()}}


def sample_modes(cfg, segments, steps):
    from cesm_emulator_b200.engine import SampleEngine
    shape = (16, 1, 192, 288)
    cond = torch.randn(shape, generator=torch.Generator().manual_seed(1)).cuda()
    engines = {}
    for pt in ("eps", "v"):
        d = _diffusion(cfg, pt).eval()
        d.requires_grad_(False)
        eng = SampleEngine(d, shape)
        eng.refresh_operands()
        eng.cond.copy_(cond)
        eng.x.normal_()
        eng.t.fill_(d.T - 1)
        eng.step()  # capture
        engines[pt] = eng
    torch.cuda.synchronize()
    ms = {n: [] for n in engines}
    for _ in range(segments):
        for n, eng in engines.items():
            eng.x.normal_()
            eng.t.fill_(eng.diffusion.T - 1)
            ms[n].append(_ms(eng.step, steps))
    return {"fields": shape[0], "H": shape[2], "W": shape[3], "ms_per_step": ms,
            "launches_per_step": {n: e.launches_per_step for n, e in engines.items()}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--segments", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    cfg = json.load(open(os.path.join(ROOT, "config", "baseline")))
    res = {"card": _card(), "train": train_modes(cfg, a.segments, a.steps),
           "sample_ddpm": sample_modes(cfg, a.segments, a.steps)}
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        open(a.out, "w").write(text)


if __name__ == "__main__":
    main()
