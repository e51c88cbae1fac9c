#!/usr/bin/env python
"""Benchmark of the hot path: data-parallel training of the config/baseline space-time U-Net.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's B200 path
    python bench.py --impl reference [--gpus N] [--steps K] ...    # the reference algorithm on host cores
    python bench.py ... --dump-outputs DIR                          # also write the last timed step's outputs

A "step" is one training step (Diffusion.loss forward + backward, gradient all-reduce when N > 1,
global-norm clip, AdamW) on one synthetic batch.  Workload (BASELINE.json configs[1]): the
config/baseline model, K=3 condition frames, full 192x288 grid, per-GPU batch 2 (train.batch_size),
fp16 activations / gradients (the reference's autocast dtype, train.py:853) with dynamic loss scaling, fp32
accumulation and fp32 master weights.  One JSON line is printed by rank 0.

  value    : samples/s over all N GPUs, inputs already resident in HBM (CUDA events, max over ranks)
  e2e      : the same metric through the public API (TrainEngine.step) with pinned HOST batches
             copied in and the loss read back every step
  roofline : the dominant kernel (the tcgen05 implicit GEMM, all its launches in one step):
             algorithmic FLOPs / summed CUDA-event durations from an untimed instrumented step,
             against the measured bf16 peak in MEASURED_PEAKS.json; `step_frac` does the same
             for the whole step (algorithmic FLOPs per sample from SURVEY.md section 8(d))
  cpu_baseline : the CPU oracle (a port of the reference's fp32 algorithm) timed on this box's
             host cores on a bounded sample, N=1 only
  gpu_comparator : the same port run on THIS GPU by stock PyTorch (cuDNN / cuBLAS / aten) under
             torch.autocast(fp16), same shape, CUDA-event timed, N=1 only (SURVEY.md section 8(d))
  extra    : BASELINE.json's other two numbers, measured the same way at this N: ensemble-generation
             fields/s (SampleEngine, fields sharded over ranks) and config/more_blocks training
  ranks_in_sync : N > 1: every rank holds bit-identical parameters after the timed steps
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

BASELINE_KW = dict(in_channels=2, out_channels=1, base_ch=64, ch_mults=(1, 2, 4), num_res_blocks=2, time_dim=124,
                   groups=8, dropout=0.0, use_checkpoint=False)          # config/baseline "unet"
MORE_BLOCKS_KW = dict(in_channels=2, out_channels=1, base_ch=64, ch_mults=(1, 2, 4, 8), num_res_blocks=6,
                      time_dim=124, groups=8, dropout=0.0, use_checkpoint=False)  # config/more_blocks "unet"
# algorithmic GFLOP per sample, forward + backward, K = 3 (SURVEY.md section 8(d); linear in pixels)
GFLOP_PER_PIXEL = {"baseline": 476.45 / (128 * 128), "more_blocks": 137.5 / (64 * 64)}
METRIC = "train samples/s (baseline cfg)"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--arch", default="baseline", choices=["baseline", "more_blocks"])
    ap.add_argument("--batch", type=int, default=2, help="per-GPU batch (config/baseline train.batch_size = 2)")
    ap.add_argument("--hw", default="192x288", help="grid (lat x lon); 192x288 = full CESM2 f09 grid")
    ap.add_argument("--frames", type=int, default=3, help="dataset.K condition frames")
    ap.add_argument("--workload", default="train", choices=["train", "sample"],
                    help="train: the headline training step; sample: reverse-diffusion steps of ensemble generation")
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of a CUDA graph")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-kernel-pass", action="store_true")
    ap.add_argument("--no-gpu-comparator", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the ensemble-generation and more_blocks side measurements")
    ap.add_argument("--kernel-table", default="", help="write the per-kernel breakdown to this file")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (float32, "
                         "64 MB at most); the inputs are seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the B200 path (--impl b200)")
    return args


DUMP_BUDGET = 63_000_000  # bytes of array data over all files: the .npy headers keep the total under 64 MB


def dump_outputs(out_dir, outputs):
    """Write every tensor of `outputs` as out_dir/<name>.npy in float32, smallest first.  One larger than its share of
    what is left of DUMP_BUDGET is written flattened, as the elements at a fixed sample of positions (sorted, drawn
    by a generator seeded with 0: the same positions in every run and every build)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = sorted(((k, v.detach().float().cpu().numpy()) for k, v in outputs.items()), key=lambda kv: kv[1].size)
    left = DUMP_BUDGET
    for i, (name, a) in enumerate(arrays):
        share = left // (len(arrays) - i) // a.itemsize
        if a.size > share:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, share, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)
        left -= a.nbytes


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"],
                "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi sampled every 200 ms during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.idx)], stdout=f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                c = [x.strip() for x in line.split(",")]
                if len(c) < 9:
                    continue
                try:
                    sm.append(float(c[1]))
                    mx.append(float(c[2]))
                except ValueError:
                    continue
                for n, v in zip(names, c[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            sm_sorted = sorted(sm)
            out.update(sm_mhz=sm_sorted[len(sm_sorted) // 2], sm_max_mhz=max(mx), reasons=sorted(reasons),
                       samples=len(sm))
        return out


# ------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port of the reference algorithm on host cores
# ------------------------------------------------------------------------------------------------
def _oracle_setup(arch_kw, threads):
    import torch
    from oracle import cesm_oracle as O
    torch.set_num_threads(threads)
    cfg = O.OracleConfig.from_unet_kwargs(**arch_kw)
    sd = O.random_state_dict(cfg, seed=0)   # reference key/shape layout; the product package is not imported here
    return O, cfg, sd, O.diffusion_buffers(1000)


def _oracle_inputs(B, frames, H, W, seed=1234):
    import torch
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(B, 1, H, W, generator=g), torch.randn(B, 1, frames, H, W, generator=g),
            torch.randint(0, 1000, (B,), generator=g), torch.randn(B, 1, H, W, generator=g))


def cpu_reference_step_time(arch_kw, frames, B, H, W, threads, steps, warmup):
    """Seconds per training step (loss fwd + bwd, global-norm clip, AdamW: train.py:858-867 in fp32) of a batch of B
    samples at H x W on `threads` host threads."""
    import torch
    O, cfg, sd, buf = _oracle_setup(arch_kw, threads)
    names = [k for k, v in sd.items() if v.is_floating_point() and not k.endswith("rotary_emb.freqs")]
    leaves = [sd[k].requires_grad_(True) for k in names]
    opt = torch.optim.AdamW(leaves, lr=2e-4, weight_decay=1e-4)
    x0, cond, t, noise = _oracle_inputs(B, frames, H, W)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        _, grads = O.loss_and_grads(sd, cfg, buf, x0, cond, t, noise)
        for k, p in zip(names, leaves):
            p.grad = grads[k]
        torch.nn.utils.clip_grad_norm_(leaves, 1.0)
        opt.step()
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    return sum(times) / len(times)


def pick_cpu_sample(B, H, W, budget_s, n_steps, arch_kw, frames, threads):
    """The largest per-step sample of the workload whose n_steps fit the budget: the full batch on the full grid,
    else one sample on the full grid, else one sample on a power-of-two fraction of the grid.  -> (b, h, w, frac)"""
    probe_h, probe_w = max(16, H // 4), max(16, W // 4)   # small grids overestimate the per-pixel cost: probe at 1/16
    t_probe = cpu_reference_step_time(arch_kw, frames, 1, probe_h, probe_w, threads, steps=1, warmup=1)
    per_pixel = t_probe / (probe_h * probe_w)
    for b, frac in ((B, 1), (1, 1), (1, 2), (1, 4), (1, 8)):
        if per_pixel * b * (H // frac) * (W // frac) * n_steps <= budget_s or frac == 8:
            return b, H // frac, W // frac, frac


def run_reference(args, H, W, arch_kw):
    """The reference arm: the reference's algorithm for the same step on this box's host cores (the reference is
    pure PyTorch and cannot travel to the GPU box, so this is the oracle port -- pinned to the reference's outputs
    by tests/golden).  `config` states what actually ran; nothing is extrapolated when the full batch fits."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    n_steps = args.steps + args.warmup
    B = args.batch
    b, h, w, frac = pick_cpu_sample(B, H, W, budget_s=330.0, n_steps=n_steps, arch_kw=arch_kw, frames=args.frames,
                                    threads=threads)
    sec = cpu_reference_step_time(arch_kw, args.frames, b, h, w, threads, steps=args.steps, warmup=args.warmup)
    full = (b, h, w) == (B, H, W)
    value = b / (sec * (H * W) / (h * w))     # samples/s; frac > 1: scaled by pixel count (cost is linear in pixels)
    sample = (f"oracle port of the reference fp32 step (loss fwd+bwd, clip, AdamW), {b} sample(s) at {h}x{w} per step"
              + ("" if frac == 1 else f" (1/{frac * frac} of the {H}x{W} grid; samples/s scaled by pixel count)")
              + f", {args.steps} timed steps after {args.warmup} warm-up, {threads} threads")
    cfg = workload_config(args, H, W, b)
    cfg["parallelism"] = "host cores (1 process)" if not full else cfg["parallelism"]
    if not full:
        cfg["sample"] = {"per_step_batch": b, "grid": [h, w], "scaled_by_pixels": frac > 1}
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {**cfg, "cuda_graph": False, "l2": "host arm: caches as the host leaves them"},
        "cpu_baseline": {"value": value, "unit": "samples/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def gpu_comparator(arch_kw, frames, B, H, W, dev, steps=5, warmup=3):
    """SURVEY.md section 8(d) "GPU comparator": the reference's algorithm (oracle port = the same torch calls the
    reference modules make) executed by STOCK PyTorch on this GPU -- cuDNN convolutions, cuBLAS matmuls, aten
    normalisation / softmax / elementwise kernels -- under torch.autocast(fp16) as the reference trains
    (train.py:853), plus clip_grad_norm_ and fused torch AdamW.  None of this repo's kernels run here."""
    import torch
    O, cfg, sd, buf = _oracle_setup(arch_kw, os.cpu_count() or 1)
    sd = {k: v.to(dev) for k, v in sd.items()}
    buf = {k: v.to(dev) for k, v in buf.items()}
    names = [k for k, v in sd.items() if v.is_floating_point() and not k.endswith("rotary_emb.freqs")]
    leaves = [sd[k].requires_grad_(True) for k in names]
    opt = torch.optim.AdamW(leaves, lr=2e-4, weight_decay=1e-4, fused=True)
    x0, cond, t, noise = (v.to(dev) for v in _oracle_inputs(B, frames, H, W))
    torch.backends.cudnn.benchmark = True
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def step():
        with torch.autocast("cuda", dtype=torch.float16):
            loss = O.diffusion_loss(sd, cfg, buf, x0, cond, t, noise)
        (loss * 65536.0).backward()
        for p in leaves:
            p.grad.mul_(1.0 / 65536.0)
        torch.nn.utils.clip_grad_norm_(leaves, 1.0)
        opt.step()
        opt.zero_grad(set_to_none=True)

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = 0.0
    for _ in range(steps):
        flush.zero_()
        e0.record()
        step()
        e1.record()
        torch.cuda.synchronize()
        ms += e0.elapsed_time(e1)
    ms /= steps
    mem = torch.cuda.max_memory_allocated(dev) / 2**30
    del sd, leaves, opt
    torch.cuda.empty_cache()
    return {"value": B / (ms * 1e-3), "unit": "samples/s", "ms_per_step": ms, "steps": steps, "warmup": warmup,
            "what": "oracle port of the reference step on this GPU through stock PyTorch "
                    f"{torch.__version__} (cuDNN/cuBLAS/aten) under torch.autocast(float16), eager, B={B} K={frames} {H}x{W}",
            "peak_mem_gib": round(mem, 1)}


def workload_config(args, H, W, per_gpu_batch):
    return {"workload": f"config/{args.arch} training step (Diffusion.loss fwd+bwd + grad all-reduce + clip + AdamW), "
                        f"K={args.frames} frames, {H}x{W} grid",
            "per_gpu_batch": per_gpu_batch, "global_batch": per_gpu_batch * args.gpus, "frames": args.frames,
            "grid": [H, W], "parallelism": f"dp{args.gpus}"}


# ------------------------------------------------------------------------------------------------
# the B200 arm
# ------------------------------------------------------------------------------------------------
def run_b200(args, H, W, arch_kw):
    import torch
    import torch.distributed as dist
    from cesm_emulator_b200 import _lib
    from cesm_emulator_b200.engine import TrainEngine
    from cesm_emulator_b200.model import Diffusion, UNet
    from cesm_emulator_b200.synthetic import SyntheticEnsemble

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit(f"--gpus {args.gpus} needs `python -m torch.distributed.run --nproc-per-node {args.gpus} bench.py ...`")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the B200 path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # stdout carries the one JSON line only
        dist.init_process_group("nccl", device_id=dev)
    peaks = load_peaks()
    B, Kf = args.batch, args.frames

    torch.manual_seed(0)
    diff = Diffusion(UNet(**arch_kw), timesteps=1000).to(dev)
    diff.train()
    eng = TrainEngine(diff, (B, 1, H, W), (B, 1, Kf, H, W), use_graph=not args.no_graph)
    # the seeded starting state (weights, AdamW moments, step count and loss scale) for --dump-outputs
    start = [t.clone() for t in (eng.opt.p, eng.opt.m, eng.opt.v, eng.opt.state)] if args.dump_outputs else None

    # synthetic (member, time, lat, lon, channel) ensemble; a small pool of pinned host batches
    ds = SyntheticEnsemble(members=4, times=max(8, Kf + 5), lat=H, lon=W, seed=1234 + rank, K=Kf)
    idx = ds.shard_indices(0, rank, world)
    pool = [ds.batch(idx[(i * B + torch.arange(B).numpy()) % len(idx)], pin=True) for i in range(4)]
    torch.manual_seed(1234 + rank)
    eng.x0.copy_(pool[0][1])
    eng.cond.copy_(pool[0][0])

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # warm-up: engine-internal eager steps + capture, then W replays
    for _ in range(3 + args.warmup):
        eng.step_resident()
    barrier()

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        n0 = _lib.launch_count()
        e0.record()
        for i in range(args.steps):
            flush.zero_()
            fn(i)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms, _lib.launch_count() - n0

    sampler = ClockSampler(local_rank)
    if rank == 0 and not os.environ.get("CESM_BENCH_NO_SAMPLER"):
        sampler.start()
    ms_res, eager_launches = timed(lambda i: eng.step_resident())
    losses = []

    def e2e_step(i):
        cond, x0 = pool[i % len(pool)]
        losses.append(eng.step(x0, cond).item())  # D2H read of the loss: syncs every step, as train.py:898 does

    for i in range(2):   # untimed: first pinned H2D copy / first blocking D2H read have one-off driver costs
        e2e_step(i)
    losses.clear()
    ms_e2e, _ = timed(e2e_step)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        # What is written is the last timed step (the e2e pass's last TrainEngine.step: same graph, same batch, the
        # RNG where the timed steps left it) repeated once, untimed, from the seeded starting state.  The timed step
        # itself starts from weights that differ from run to run by more than rounding: fp32 atomics add in a
        # different order each time, and AdamW's normalised update turns a last-bit difference in a near-zero
        # gradient into a full step of either sign, so the weights drift apart over the timed steps.  From the seeded
        # state, two runs and two builds start from the same inputs.  The weights the repeated step leaves are not
        # written: its update already flips sign where the gradient is near zero (1e-4 of max|w| between two runs, 10x
        # the gradient's difference; profiles/r03_dump_reproducibility.txt), and they follow elementwise from the
        # gradient and the seeded state.  The state the timed run reached and the RNG are put back afterwards, so
        # every reported field still describes the timed run.
        live = (eng.opt.p, eng.opt.m, eng.opt.v, eng.opt.state)
        reached, rng = [t.clone() for t in live], torch.cuda.get_rng_state(dev)
        for dst, src in zip(live, start):
            dst.copy_(src)
        scale = eng.opt.loss_scale.clone()
        cond, x0 = pool[(args.steps - 1) % len(pool)]
        eng.step(x0, cond)
        # p.grad views the flat gradient buffer, which holds the loss-scaled gradient before clipping (module order)
        outputs = {"loss": eng.loss, "grad_norm": eng.grad_norm, "loss_scale": eng.opt.loss_scale,
                   "gradient": torch.cat([p.grad.reshape(-1) for p in diff.parameters() if p.requires_grad]) / scale}
        if rank == 0:
            dump_outputs(args.dump_outputs, outputs)
        del outputs
        for dst, src in zip(live, reached):
            dst.copy_(src)
        torch.cuda.set_rng_state(rng, dev)

    in_sync = None
    if world > 1:
        # every rank must hold bit-identical parameters after the same all-reduced updates (train.py:1076)
        bits = eng.opt.p.view(torch.int32).to(torch.int64)
        sig = torch.stack([bits.sum(), (bits * (torch.arange(bits.numel(), device=dev) % 8191 + 1)).sum()])
        sigs = [torch.zeros_like(sig) for _ in range(world)]
        dist.all_gather(sigs, sig)
        in_sync = all(torch.equal(sigs[0], x) for x in sigs)

    samples = B * world * args.steps
    value = samples / (ms_res * 1e-3)
    e2e_value = samples / (ms_e2e * 1e-3)
    launches = eng.launches_per_step * args.steps  # graph replays re-issue the captured kernels
    h2d = pool[0][0].numel() * 4 + pool[0][1].numel() * 4

    # ---- untimed instrumented step: per-kernel breakdown and the dominant kernel's roofline --------
    roofline, table = None, None
    gflop_sample = GFLOP_PER_PIXEL[args.arch] * H * W if Kf == 3 else None
    step_tf = (gflop_sample * B / (ms_res / args.steps)) if gflop_sample else None  # GFLOP/ms == TFLOP/s
    if not args.no_kernel_pass:
        # every rank runs the step (it contains the all-reduce); rank 0 reports
        for h in eng.buckets._hooks:
            h.remove()
        prof_eng = TrainEngine(diff, (B, 1, H, W), (B, 1, Kf, H, W), use_graph=False)
        prof_eng.side_stream = None   # per-call event timing wants one stream: no overlap between bracketed calls
        prof_eng.x0.copy_(eng.x0)
        prof_eng.cond.copy_(eng.cond)
        prof_eng.step_resident()
        torch.cuda.synchronize()
        _lib.PROFILER = _lib.KernelProfiler()
        prof_eng.step_resident()
        table = _lib.PROFILER.summary()
        _lib.PROFILER = None
    if rank == 0 and table is not None:
        ig = [v for k, v in table.items() if k.startswith("cesm_igemm")]
        ig_ms, ig_fl, ig_calls = sum(v["ms"] for v in ig), sum(v["flops"] for v in ig), sum(v["calls"] for v in ig)
        total_ms = sum(v["ms"] for v in table.values())
        peak = peaks["bf16_tflops_sustained"]
        ach = ig_fl / (ig_ms * 1e-3) / 1e12
        traffic = None  # DRAM bytes per launch of the same kernels, from the committed ncu pass of this workload
        tj = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "r02_step_traffic.json")
        if args.arch == "baseline" and (B, Kf, H, W) == (2, 3, 192, 288) and os.path.exists(tj):
            tk = [v for k, v in json.load(open(tj)).items() if "igemm2_kernel" in k]
            traffic = sum(v["dram_bytes_per_launch"] * v["launches"] for v in tk) / max(1, sum(v["launches"] for v in tk))
        roofline = {"bound": "tensor", "kernel": "igemm2_kernel (tcgen05 implicit GEMM: conv fwd + dgrad + projections)",
                    "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                    "peak_source": f"{peaks['source']} bf16_tflops_sustained (kernel timed inside a long step)",
                    "launches_per_step": ig_calls, "share_of_kernel_time": ig_ms / total_ms, "traffic": traffic,
                    "traffic_source": "profiles/r02_step_traffic.txt (ncu dram__bytes_read+write, mean per launch)",
                    "algorithmic_bytes_per_launch": sum(v["bytes"] for v in ig) / max(1, ig_calls),
                    "step_achieved": step_tf, "step_frac": (step_tf / peak) if step_tf else None}
        lines = [f"{'kernel':40s} {'calls':>6s} {'ms':>9s} {'share':>7s} {'TFLOP/s':>9s} {'GB/s':>9s}"]
        for k, v in sorted(table.items(), key=lambda kv: -kv[1]["ms"]):
            tf = v["flops"] / (v["ms"] * 1e-3) / 1e12 if v["flops"] else 0.0
            gb = v["bytes"] / (v["ms"] * 1e-3) / 1e9 if v["bytes"] else 0.0
            lines.append(f"{k:40s} {v['calls']:6d} {v['ms']:9.3f} {v['ms'] / total_ms:7.1%} {tf:9.1f} {gb:9.1f}")
        lines.append(f"{'total (instrumented eager step)':40s} {sum(v['calls'] for v in table.values()):6d} {total_ms:9.3f}")
        text = "\n".join(lines)
        sys.stderr.write(text + "\n")
        if args.kernel_table:
            with open(args.kernel_table, "w") as f:
                f.write(f"# bench.py kernel pass: arch={args.arch} B={B} K={Kf} grid={H}x{W}\n" + text + "\n")

    cpu_baseline = comparator = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        b, h, w, frac = pick_cpu_sample(1, H, W, budget_s=40.0, n_steps=4, arch_kw=arch_kw, frames=Kf, threads=threads)
        sec = cpu_reference_step_time(arch_kw, Kf, b, h, w, threads, steps=3, warmup=1)
        cpu_baseline = {"value": b / (sec * (H * W) / (h * w)), "unit": "samples/s", "cores": threads, "kind": "port",
                        "sample": f"oracle port (fp32 torch CPU) of the step (loss fwd+bwd, clip, AdamW), {b} sample at {h}x{w}"
                                  + (f", 1/{frac * frac} of the grid, scaled by pixel count" if frac > 1 else "")
                                  + ", mean of 3 timed steps after 1 warm-up"}
    if rank == 0 and world == 1 and not args.no_gpu_comparator:
        try:
            comparator = gpu_comparator(arch_kw, Kf, B, H, W, dev)
        except Exception as exc:  # e.g. out of memory next to the engines: report, do not hide
            comparator = {"unavailable": f"{type(exc).__name__}: {exc}"[:200]}

    # ---- BASELINE.json's other two numbers at this N (untimed by the driver; same event timing) --------
    extra = {}
    if not args.no_extra:
        extra["ensemble_gen"] = measure_sampling(args, H, W, BASELINE_KW, dev, rank, world, steps=10, warmup=3)
        extra["more_blocks"] = measure_more_blocks(args, dev, rank, world, peaks, steps=5, warmup=3)
        if rank == 0 and world == 1:
            extra["long_window_attention"] = measure_long_window_attention(dev, H, W)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_res / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "fp16", "data": "synthetic",
            "config": {**workload_config(args, H, W, B), "cuda_graph": not args.no_graph,
                       "l2": "256 MiB buffer zeroed between steps (L2 is 126 MB); per-step activations >> L2"},
            "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                    "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": launches, "launches_per_step": eng.launches_per_step,
            "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu_baseline, "gpu_comparator": comparator,
            "extra": extra, "ranks_in_sync": in_sync,
            "loss_scale": {"final": float(eng.opt.state[2]), "skipped_steps": int(eng.opt.state[5])},
            "loss_first_last": [losses[0], losses[-1]] if losses else None,
        }
        emit(line)
    if world > 1:
        # Tear-down: the captured graphs hold NCCL kernels, and destroying the communicator under them
        # can block; everything is measured and printed, so synchronise, meet at a barrier and leave.
        sys.stdout.flush()
        sys.stderr.flush()
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        os._exit(0)


def measure_sampling(args, H, W, arch_kw, dev, rank, world, steps, warmup, B=16, dump_dir=""):
    """BASELINE.json's second metric, "ensemble-gen fields/s": reverse-diffusion steps for a batch of independent
    fields (inference.py:217-232 -> model.py:186-194), one CUDA-graph replay per step, fields sharded over ranks
    (each rank its own batch, no collective inside the chain).  A step = one UNet call (F = 1) + fused p_sample
    update; fields/s = world * batch / (T * step time), T = 1000, step time = max over ranks."""
    import torch
    import torch.distributed as dist
    from cesm_emulator_b200 import ops
    from cesm_emulator_b200.engine import SampleEngine
    from cesm_emulator_b200.model import Diffusion, UNet
    ops.set_grad_sink(None)
    torch.manual_seed(0)
    diff = Diffusion(UNet(**arch_kw), timesteps=1000).to(dev)
    diff.eval()
    for p_ in diff.parameters():
        p_.requires_grad_(False)
    eng = SampleEngine(diff, (B, 1, H, W), use_graph=not args.no_graph)
    torch.manual_seed(4321 + rank)   # every rank generates different fields
    eng.cond.normal_()
    eng.x.normal_()
    eng.t.fill_(999)
    for _ in range(1 + warmup):
        eng.step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        eng.step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, {"x": eng.x})   # the fields after the last timed reverse step
    finite = bool(torch.isfinite(eng.x).all())
    gflop = 178.5 * (H * W) / (192 * 288) if arch_kw is BASELINE_KW else None  # SURVEY 8(d): per UNet call per field
    peaks = load_peaks()
    tf = gflop * B / ms if gflop else None
    out = {"metric": "ensemble-gen fields/s (1000-step DDPM chain)", "value": B * world / (1000 * ms * 1e-3),
           "unit": "fields/s", "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms,
           "fields_per_gpu_batch": B, "grid": [H, W], "frames": 1, "finite": finite,
           "note": f"{steps} timed reverse steps of a {B}-field batch per GPU (fields sharded over ranks, no collective); "
                   "value extrapolated to the full 1000-step chain",
           "launches_per_step": eng.launches_per_step,
           "roofline": {"bound": "tensor", "achieved": tf, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                        "frac": tf / peaks["bf16_tflops_sustained"] if tf else None,
                        "note": "whole reverse step: algorithmic 178.5 GFLOP per field per UNet call at 192x288"}}
    del eng, diff
    torch.cuda.empty_cache()
    return out


def measure_long_window_attention(dev, H, W, frames=(32, 64, 128), heads=8, steps=5):
    """BASELINE.json configs[4] (SURVEY.md section 8(d) item 5): the temporal-attention core in isolation on the full
    grid for multi-decade windows, B = 1: q|k|v [F*H*W, 768] fp16 -> out [F*H*W, 256] (cesm_tattn_long_fwd / _bwd).
    HBM-bound: algorithmic bytes = q|k|v + out forward (2 KB per row); q|k|v, out, dout, dq|dk|dv backward (4 KB per
    row) against the measured copy bandwidth; tensor work (mma.sync) is reported beside it."""
    import torch
    from cesm_emulator_b200 import kernels as K
    peaks = load_peaks()
    D, HW, res = 32, H * W, {}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    for F in frames:
        rows = F * HW
        torch.manual_seed(F)
        qkv = (torch.randn(rows, 3 * heads * D, device=dev) * 0.5).half()
        dout = (torch.randn(rows, heads * D, device=dev) * 0.1).half()
        diag = torch.randn(heads, 2 * F - 1, device=dev) * 0.1
        i = torch.arange(F, device=dev)
        bias = diag[:, (i[None, :] - i[:, None]) + F - 1].contiguous()
        freqs = (1.0 / (10000 ** (torch.arange(0, D, 2).float() / D))).to(dev)
        ang = torch.arange(F, device=dev, dtype=torch.float32)[:, None] * freqs[None]
        cs, sn = ang.cos().contiguous(), ang.sin().contiguous()
        out, lse = K.tattn_fwd(qkv, bias, cs, sn, 1, F, HW, heads, D, D ** -0.5)     # warm-up
        K.tattn_bwd(qkv, bias, cs, sn, out, lse, dout, 1, F, HW, heads, D, D ** -0.5)
        torch.cuda.synchronize()
        t = {}
        for name, fn in (("fwd", lambda: K.tattn_fwd(qkv, bias, cs, sn, 1, F, HW, heads, D, D ** -0.5)),
                         ("bwd", lambda: K.tattn_bwd(qkv, bias, cs, sn, out, lse, dout, 1, F, HW, heads, D, D ** -0.5))):
            ms = 0.0
            for _ in range(steps):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn()
                e1.record()
                torch.cuda.synchronize()
                ms += e0.elapsed_time(e1)
            t[name] = ms / steps
        by_f = rows * (3 + 1) * heads * D * 2.0
        by_b = rows * (3 + 1 + 1 + 3) * heads * D * 2.0
        fl_f = 4.0 * rows * heads * F * D            # QK^T + PV
        fl_b = 14.0 * rows * heads * F * D           # 7 F x F x 32 contractions (S and dP recomputed in both passes)
        res[f"F{F}"] = {
            "rows": rows, "fwd_ms": t["fwd"], "bwd_ms": t["bwd"],
            "fwd_rows_per_s": rows / (t["fwd"] * 1e-3), "bwd_rows_per_s": rows / (t["bwd"] * 1e-3),
            "roofline_fwd": {"bound": "hbm", "achieved": by_f / t["fwd"] / 1e6, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                             "frac": by_f / t["fwd"] / 1e6 / peaks["hbm_gbs"], "tensor_tflops": fl_f / t["fwd"] / 1e9},
            "roofline_bwd": {"bound": "hbm", "achieved": by_b / t["bwd"] / 1e6, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                             "frac": by_b / t["bwd"] / 1e6 / peaks["hbm_gbs"], "tensor_tflops": fl_b / t["bwd"] / 1e9}}
        del qkv, dout, out, lse
        torch.cuda.empty_cache()
    return {"metric": "temporal attention core, long windows (rows = frames x pixels)", "grid": [H, W], "heads": heads,
            "batch": 1, "steps": steps, "by_frames": res}


def measure_more_blocks(args, dev, rank, world, peaks, steps, warmup):
    """BASELINE.json configs[2]: config/more_blocks (ch_mults [1,2,4,8]) training at its own crop and batch
    (config/more_blocks: 64x64, batch_size 64 per GPU, K = 3), data-parallel over the same ranks."""
    import torch
    import torch.distributed as dist
    from cesm_emulator_b200 import ops
    from cesm_emulator_b200.engine import TrainEngine
    from cesm_emulator_b200.model import Diffusion, UNet
    B, Kf, H, W = 64, 3, 64, 64
    ops.set_grad_sink(None)
    torch.manual_seed(0)
    diff = Diffusion(UNet(**MORE_BLOCKS_KW), timesteps=1000).to(dev)
    diff.train()
    eng = TrainEngine(diff, (B, 1, H, W), (B, 1, Kf, H, W), use_graph=not args.no_graph)
    torch.manual_seed(99 + rank)
    eng.x0.normal_()
    eng.cond.normal_()
    for _ in range(3 + warmup):
        eng.step_resident()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        flush.zero_()
        eng.step_resident()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
        torch.cuda.synchronize()
    tf = GFLOP_PER_PIXEL["more_blocks"] * H * W * B / ms
    out = {"metric": "train samples/s (more_blocks cfg)", "value": B * world / (ms * 1e-3), "unit": "samples/s",
           "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms, "per_gpu_batch": B, "grid": [H, W],
           "frames": Kf, "loss": float(eng.loss), "launches_per_step": eng.launches_per_step,
           "roofline": {"bound": "tensor", "achieved": tf, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                        "frac": tf / peaks["bf16_tflops_sustained"],
                        "note": "whole step: algorithmic 137.5 GFLOP per sample (SURVEY 8(d)) / step time"}}
    for h in eng.buckets._hooks:
        h.remove()
    ops.set_grad_sink(None)
    del eng, diff
    torch.cuda.empty_cache()
    return out


def run_sample(args, H, W, arch_kw):
    """`--workload sample`: the ensemble-generation measurement as the headline line (torchrun for N > 1)."""
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the B200 path has no CPU fallback")
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    B = args.batch if args.batch != 2 else 16  # inference.py:180 default batch_size 16
    out = measure_sampling(args, H, W, arch_kw, dev, rank, world, steps=args.steps, warmup=args.warmup, B=B,
                           dump_dir=args.dump_outputs)
    if rank == 0 and args.kernel_table:
        # untimed instrumented reverse step: per-C-ABI-call device time
        from cesm_emulator_b200 import _lib
        from cesm_emulator_b200.engine import SampleEngine
        from cesm_emulator_b200.model import Diffusion, UNet
        torch.manual_seed(0)
        diff = Diffusion(UNet(**arch_kw), timesteps=1000).to(dev)
        diff.eval()
        eng = SampleEngine(diff, (B, 1, H, W), use_graph=False)
        eng.cond.normal_(); eng.x.normal_(); eng.t.fill_(999)
        eng.step()
        torch.cuda.synchronize()
        _lib.PROFILER = _lib.KernelProfiler()
        eng.step()
        table = _lib.PROFILER.summary()
        _lib.PROFILER = None
        total_ms = sum(v["ms"] for v in table.values())
        lines = [f"# bench.py --workload sample kernel pass: arch={args.arch} fields={B} grid={H}x{W}",
                 f"{'kernel':40s} {'calls':>6s} {'ms':>9s} {'share':>7s} {'TFLOP/s':>9s} {'GB/s':>9s}"]
        for k, v in sorted(table.items(), key=lambda kv: -kv[1]["ms"]):
            tf = v["flops"] / (v["ms"] * 1e-3) / 1e12 if v["flops"] else 0.0
            gb = v["bytes"] / (v["ms"] * 1e-3) / 1e9 if v["bytes"] else 0.0
            lines.append(f"{k:40s} {v['calls']:6d} {v['ms']:9.3f} {v['ms'] / total_ms:7.1%} {tf:9.1f} {gb:9.1f}")
        lines.append(f"{'total (instrumented eager step)':40s} {sum(v['calls'] for v in table.values()):6d} {total_ms:9.3f}")
        with open(args.kernel_table, "w") as f:
            f.write("\n".join(lines) + "\n")
    if rank == 0:
        out.update({"higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp16", "data": "synthetic",
                    "config": {"workload": f"config/{args.arch} sampling, {B} fields per GPU batch, {H}x{W}, F=1",
                               "cuda_graph": not args.no_graph},
                    "gpu_launches": out["launches_per_step"] * args.steps})
        emit(out)
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        os._exit(0)


_REAL_STDOUT = None


def emit(line: dict) -> None:
    """The ONE JSON line goes to the process's original stdout; everything else any library prints (NCCL's version
    banner, torchrun notices) has been routed to stderr by main()."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    args = parse_args()
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)   # fd 1 -> stderr for C libraries and stray prints; emit() writes the JSON line to the saved fd
    if args.impl == "b200":
        from cesm_emulator_b200 import build as _build
        if not _build.LIB_PATH.exists():  # fresh checkout: build artefacts are git-ignored
            if int(os.environ.get("LOCAL_RANK", "0")) == 0:
                _build.build()
            else:  # the other ranks of a torchrun launch wait for rank 0's build
                t0 = time.time()
                while not _build.LIB_PATH.exists() and time.time() - t0 < 600:
                    time.sleep(1.0)
    H, W = (int(v) for v in args.hw.lower().split("x"))
    arch_kw = BASELINE_KW if args.arch == "baseline" else MORE_BLOCKS_KW
    if args.impl == "reference":
        run_reference(args, H, W, arch_kw)
    elif args.workload == "sample":
        run_sample(args, H, W, arch_kw)
    else:
        run_b200(args, H, W, arch_kw)


if __name__ == "__main__":
    main()
