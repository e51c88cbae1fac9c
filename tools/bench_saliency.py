#!/usr/bin/env python
"""Cost of emission saliency against a training step, on config/baseline's UNet over the full 192x288 grid.

For each shape -- B = 2, K = 3 (the bench training shape) and B = 16, F = 1 (the sampling shape) -- a SaliencyEngine
draw (forward + frozen-weight backward, one CUDA-graph replay plus the noise draw) and a TrainEngine step are timed
with CUDA events, alternated segment by segment in the same process.  Then one eager, instrumented draw gives the
per-call time of cesm_input_conv_dgrad (kernels.KernelProfiler).  The card's name, power limit and max SM clock are
read in the same run.

    python tools/bench_saliency.py [--draws 8] [--segments 5] [--steps 10] [--out profiles/x.json]
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


def _model(cfg, frozen):
    import train as train_entry
    from cesm_emulator_b200.model import Diffusion
    torch.manual_seed(0)
    d = Diffusion(train_entry.build_model_from_config(cfg["unet"])).cuda()
    if frozen:
        d.requires_grad_(False)
    return d


def _ms(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def measure(cfg, B, K, draws, segments, steps):
    from cesm_emulator_b200 import _lib, ops
    from cesm_emulator_b200.engine import SaliencyEngine, TrainEngine
    H, W = 192, 288
    g = torch.Generator().manual_seed(0)
    x0 = torch.randn(B, 1, H, W, generator=g).cuda()
    cond = torch.randn(*((B, 1, K, H, W) if K > 1 else (B, 1, H, W)), generator=g).cuda()
    sal = SaliencyEngine(_model(cfg, True), x0.shape, cond.shape, draws=draws, seed=1)
    train = TrainEngine(_model(cfg, False), x0.shape, cond.shape)
    for _ in range(3):
        train.step(x0, cond)
    sal.saliency(x0, cond)
    ops.set_grad_sink(None)
    torch.cuda.synchronize()
    per_draw, per_step = [], []
    for _ in range(segments):
        per_draw.append(_ms(lambda: sal.saliency(x0, cond), 1) / draws)
        per_step.append(_ms(lambda: train.step_resident(), steps))
    ops.set_grad_sink(None)
    eager = SaliencyEngine(sal.diffusion, x0.shape, cond.shape, draws=1, use_graph=False, seed=1)
    eager.saliency(x0, cond)
    _lib.PROFILER = prof = _lib.KernelProfiler()
    try:
        eager.saliency(x0, cond)
    finally:
        _lib.PROFILER = None
    summ = prof.summary()
    dg = summ["cesm_input_conv_dgrad"]
    return {"B": B, "frames": K, "H": H, "W": W, "draws": draws,
            "saliency_ms_per_draw": per_draw, "train_ms_per_step": per_step,
            "saliency_launches_per_draw": sal.launches_per_step, "train_launches_per_step": train.launches_per_step,
            "input_conv_dgrad_ms": dg["ms"] / dg["calls"], "input_conv_dgrad_gflop": dg["flops"] / dg["calls"] / 1e9,
            "input_conv_dgrad_mb": dg["bytes"] / dg["calls"] / 1e6,
            "eager_draw_kernel_ms": sum(v["ms"] for v in summ.values())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--draws", type=int, default=8)
    ap.add_argument("--segments", type=int, default=5)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    cfg = json.load(open(os.path.join(ROOT, "config", "baseline")))
    res = {"card": _card(), "shapes": [measure(cfg, 2, 3, a.draws, a.segments, a.steps),
                                       measure(cfg, 16, 1, a.draws, a.segments, a.steps)]}
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        open(a.out, "w").write(text)


if __name__ == "__main__":
    main()
