"""DPM-Solver++(2M) sampling against strided DDIM (eta = 0) on the B200, at bench.py's sampling workload
(config/baseline architecture, random weights, 16 fields of 192x288, F = 1, one CUDA-graph replay per step).

    python tools/bench_dpm.py [--rounds 3] [--steps 50] [--out profiles/r06_dpm_sampling.txt]
                              [--compare-tree DIR]

Prints the device name, power limit and max SM clock first: every number below belongs to them.
(a) ms per reverse step: a DDIM-mode and a 2M-mode SampleEngine (both N = 50) are built in one process and timed in
    alternating segments of `--steps` replays (CUDA events, after warm-up).  The 2M update kernel moves 20 B per
    element (x, eps and the history read; x and the history written), 18 MB per step here and 8 B per element more
    than the DDIM update, against a UNet call of about 6.5 ms.  launches_per_step counts libcesm_b200 kernel launches
    of one replay.
(b) fields/s per GPU: the whole chain, `SampleEngine.sample(cond)` (weights refresh, x_T draw, N replays, copy of the
    result), timed with a host clock around a device synchronise, for 2M at N = 10, 15, 20, 25 and DDIM at N = 25,
    alternating within each round.  fields/s = 16 / chain time.
(c) with --compare-tree DIR (a checkout of another commit, built): `bench.py --workload sample` from DIR and from this
    tree, alternated twice, to show the default DDPM path's step time is unchanged.
Nothing here measures sample quality (random weights); tools/sampler_accuracy.py has the toy-distribution accuracy."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

B, H, W = 16, 192, 288
DPM_N = (10, 15, 20, 25)
BASELINE_KW = dict(in_channels=2, out_channels=1, base_ch=64, ch_mults=(1, 2, 4), num_res_blocks=2, time_dim=124,
                   groups=8, dropout=0.0, use_checkpoint=False)          # config/baseline "unet"
BENCH_ARGS = ["--gpus", "1", "--steps", "30", "--warmup", "5", "--workload", "sample", "--no-cpu-baseline"]


def device_line():
    import torch
    name = torch.cuda.get_device_name(0)
    q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                       capture_output=True, text=True)
    pl, clk = (s.strip() for s in q.stdout.strip().split(","))
    return name, float(pl), float(clk)


def bench_sample(tree):
    """One `bench.py --workload sample` run from `tree`; returns its JSON line."""
    r = subprocess.run([sys.executable, "bench.py", *BENCH_ARGS], cwd=tree, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"bench.py in {tree} failed:\n{r.stderr[-4000:]}")
    return json.loads(r.stdout.strip().splitlines()[-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=50, help="replays per timed step segment in (a)")
    ap.add_argument("--out", default="", help="also write the report to this file")
    ap.add_argument("--compare-tree", default="", help="built checkout to compare bench.py --workload sample against")
    args = ap.parse_args()
    import torch
    from cesm_emulator_b200 import ops
    from cesm_emulator_b200.engine import SampleEngine
    from cesm_emulator_b200.model import Diffusion, UNet
    assert torch.cuda.is_available(), "bench_dpm needs a CUDA device"
    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    name, pl, clk = device_line()
    say(f"device: {name}, power limit {pl:.0f} W, max SM clock {clk:.0f} MHz")
    say(f"workload: config/baseline UNet (random weights, seed 0), {B} fields x 1 x {H} x {W}, F = 1, CUDA graph per step")
    dev = torch.device("cuda:0")
    ops.set_grad_sink(None)
    torch.manual_seed(0)
    diff = Diffusion(UNet(**BASELINE_KW), timesteps=1000).to(dev)
    diff.eval()
    for p in diff.parameters():
        p.requires_grad_(False)
    torch.manual_seed(4321)
    cond = torch.randn(B, 1, H, W, device=dev)

    # (a) ms per step, alternating segments
    engines = {"ddim N=50": SampleEngine(diff, (B, 1, H, W), ddim_steps=50),
               "2M N=50": SampleEngine(diff, (B, 1, H, W), dpm_steps=50)}
    for eng in engines.values():
        eng.cond.copy_(cond)
        eng.x.normal_()
        for _ in range(4):  # warm-up + capture + replays
            eng.t.fill_(999)
            eng.step()
    torch.cuda.synchronize()
    ms = {k: [] for k in engines}
    for _ in range(args.rounds):
        for k, eng in engines.items():
            eng.x.normal_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(args.steps):
                if i % 50 == 0:   # an N = 50 chain ends after 50 replays: restart both modes at t = 999 alike
                    eng.t.fill_(999)
                eng.step()
            e1.record()
            torch.cuda.synchronize()
            ms[k].append(e0.elapsed_time(e1) / args.steps)
    say()
    say(f"(a) ms per reverse step, {args.rounds} alternating segments of {args.steps} replays each")
    say(f"{'mode':12s} {'launches/step':>13s} {'mean ms':>8s}  per segment")
    for k, eng in engines.items():
        v = ms[k]
        say(f"{k:12s} {eng.launches_per_step:13d} {sum(v) / len(v):8.3f}  " + " ".join(f"{x:.3f}" for x in v))
    del engines
    torch.cuda.empty_cache()

    # (b) whole chains, alternating within each round
    chains = {f"2M N={n}": SampleEngine(diff, (B, 1, H, W), dpm_steps=n) for n in DPM_N}
    chains["ddim N=25"] = SampleEngine(diff, (B, 1, H, W), ddim_steps=25)
    for eng in chains.values():   # capture every graph before timing
        eng.cond.copy_(cond)
        eng.t.fill_(999)
        eng.step()
    torch.cuda.synchronize()
    secs = {k: [] for k in chains}
    finite = {}
    for _ in range(args.rounds):
        for k, eng in chains.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            y = eng.sample(cond)
            torch.cuda.synchronize()
            secs[k].append(time.perf_counter() - t0)
            finite[k] = bool(torch.isfinite(y).all())
    say()
    say(f"(b) whole chain of {B} fields, {args.rounds} alternating rounds (host clock around a device synchronise)")
    say(f"{'chain':12s} {'UNet calls':>10s} {'mean s':>8s} {'ms/step':>8s} {'fields/s':>9s} finite  per round (s)")
    for k, eng in chains.items():
        v = secs[k]
        mean = sum(v) / len(v)
        n = eng.dpm_steps if eng.dpm_steps is not None else eng.ddim_steps
        say(f"{k:12s} {n:10d} {mean:8.3f} {1e3 * mean / n:8.3f} {B / mean:9.2f} {str(finite[k]):6s}  "
            + " ".join(f"{x:.3f}" for x in v))
    del chains, diff
    torch.cuda.empty_cache()

    if args.compare_tree:
        say()
        say(f"(c) bench.py {' '.join(BENCH_ARGS)}, the other tree and this one alternated (other, this, other, this)")
        runs = {"other": [], "this": []}
        for _ in range(2):
            for label, tree in (("other", os.path.abspath(args.compare_tree)), ("this", ROOT)):
                runs[label].append(bench_sample(tree))
        for label, rs in runs.items():
            say(f"  {label:5s} " + " | ".join(f"{r['ms_per_step']:.3f} ms/step {r['value']:.3f} fields/s, "
                                             f"{r['launches_per_step']} launches/step, finite {r['finite']}" for r in rs))
    if args.out:
        d = os.path.dirname(args.out)
        if d:
            os.makedirs(d, exist_ok=True)
        with open(args.out, "w") as f:
            f.write("tools/bench_dpm.py: DPM-Solver++(2M) sampling vs strided DDIM (eta = 0)\n")
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
