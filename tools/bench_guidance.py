#!/usr/bin/env python
"""Cost of classifier-free guidance on config/baseline's UNet over the 192x288 grid.

Sampling: fields/s of a whole SampleEngine chain for 16 one-frame fields, unguided (w = 0) against guided (w = 2), for
DDIM with N = 50 (eta = 0) and DPM-Solver++(2M) with N = 15.  A guided step is one UNet call on 32 rows and one guided
update launch.  Training: one TrainEngine step at bench.py's shape (B = 2, K = 3) with condition dropout off against
p = 0.1.  Every step is a CUDA-graph replay timed with CUDA events; the modes of a group are alternated segment by
segment in the same process, and every engine's `launches_per_step` is recorded.  The card's name, power limit and max
SM clock are read in the same run.

    python tools/bench_guidance.py [--segments 3] [--steps 20] [--out profiles/x.json]
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


def _diffusion(cfg):
    import train as train_entry
    from cesm_emulator_b200.model import Diffusion
    torch.manual_seed(0)
    return Diffusion(train_entry.build_model_from_config(cfg["unet"])).cuda()


def _ms(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def sample_modes(cfg, segments):
    from cesm_emulator_b200.engine import SampleEngine
    shape = (16, 1, 192, 288)
    cond = torch.randn(shape, generator=torch.Generator().manual_seed(1)).cuda()
    d = _diffusion(cfg).eval()
    d.requires_grad_(False)
    res = {}
    for chain, kw in (("ddim50", dict(ddim_steps=50)), ("dpm15", dict(dpm_steps=15))):
        engines = {w: SampleEngine(d, shape, guidance=w, seed=7, **kw) for w in (0.0, 2.0)}
        for eng in engines.values():
            eng.sample(cond)  # capture and warm up
        torch.cuda.synchronize()
        ms = {w: [] for w in engines}
        for _ in range(segments):
            for w, eng in engines.items():
                ms[w].append(_ms(lambda: eng.sample(cond), 1))
        res[chain] = {"fields": shape[0], "H": shape[2], "W": shape[3],
                      "ms_per_chain": {str(w): v for w, v in ms.items()},
                      "fields_per_s": {str(w): shape[0] * 1000.0 / min(v) for w, v in ms.items()},
                      "launches_per_step": {str(w): e.launches_per_step for w, e in engines.items()}}
    return res


def train_modes(cfg, segments, steps):
    from cesm_emulator_b200 import ops
    from cesm_emulator_b200.engine import TrainEngine
    B, K, H, W = 2, 3, 192, 288
    g = torch.Generator().manual_seed(0)
    x0, cond = torch.randn(B, 1, H, W, generator=g).cuda(), torch.randn(B, 1, K, H, W, generator=g).cuda()
    engines = {}
    for p in (0.0, 0.1):
        d = _diffusion(cfg)
        d.train()
        engines[p] = TrainEngine(d, x0.shape, cond.shape, cond_drop_prob=p)
    for _ in range(3):  # two eager warm-up steps, then the capture
        for eng in engines.values():
            eng.step(x0, cond)
    torch.cuda.synchronize()
    ms = {p: [] for p in engines}
    for _ in range(segments):
        for p, eng in engines.items():
            ms[p].append(_ms(eng.step_resident, steps))
    ops.set_grad_sink(None)
    return {"B": B, "frames": K, "H": H, "W": W, "ms_per_step": {str(p): v for p, v in ms.items()},
            "launches_per_step": {str(p): e.launches_per_step for p, e in engines.items()}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--segments", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    cfg = json.load(open(os.path.join(ROOT, "config", "baseline")))
    res = {"card": _card(), "sample": sample_modes(cfg, a.segments), "train": train_modes(cfg, a.segments, a.steps)}
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        open(a.out, "w").write(text)


if __name__ == "__main__":
    main()
