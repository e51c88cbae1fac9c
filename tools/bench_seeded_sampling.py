"""Per-step cost of seeded (counter-based, in-kernel) sampling noise against torch-RNG noise on the B200, at bench.py's
sampling workload (config/baseline architecture, random weights, 16 fields of 192x288, F = 1, one CUDA-graph replay
per step).

    python tools/bench_seeded_sampling.py [--rounds 5] [--steps 50] [--out profiles/r09_seeded_sampling.txt]

Prints the device name, power limit and max SM clock first: every number below belongs to them.
(a) ms per reverse step of four SampleEngines built in one process -- DDPM and DDIM (N = 50, eta = 1), each
    unseeded (a `normal_` into the z buffer + the update reading it) and seeded (the update drawing z in registers) --
    timed in alternating segments of `--steps` replays with CUDA events after warm-up.
(b) the noise + update alone, outside any graph, averaged over 200 calls: `normal_` + `p_sample` + copy against
    `p_sample_seeded` in place, and `normal_` + `ddim_step` against `ddim_step_seeded`, each in place on the same
    16 x 192 x 288 fields (14 MB per buffer, inside the 126 MB L2)."""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

B, H, W = 16, 192, 288
SEED = 1234
BASELINE_KW = dict(in_channels=2, out_channels=1, base_ch=64, ch_mults=(1, 2, 4), num_res_blocks=2, time_dim=124,
                   groups=8, dropout=0.0, use_checkpoint=False)          # config/baseline "unet"


def device_line():
    import torch
    name = torch.cuda.get_device_name(0)
    q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                       capture_output=True, text=True)
    pl, clk = (s.strip() for s in q.stdout.strip().split(","))
    return name, float(pl), float(clk)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=50, help="replays per timed step segment in (a)")
    ap.add_argument("--out", default="", help="also write the report to this file")
    args = ap.parse_args()
    import torch
    from cesm_emulator_b200 import kernels as K
    from cesm_emulator_b200 import ops
    from cesm_emulator_b200.engine import SampleEngine
    from cesm_emulator_b200.model import Diffusion, UNet
    assert torch.cuda.is_available(), "bench_seeded_sampling needs a CUDA device"
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
    shape = (B, 1, H, W)

    # (a) ms per step, alternating segments
    engines = {"ddpm": SampleEngine(diff, shape), "ddpm seeded": SampleEngine(diff, shape, seed=SEED),
               "ddim eta=1": SampleEngine(diff, shape, ddim_steps=50, eta=1.0),
               "ddim eta=1 seeded": SampleEngine(diff, shape, ddim_steps=50, eta=1.0, seed=SEED)}
    x0 = torch.randn(shape, device=dev)
    for eng in engines.values():
        eng.cond.copy_(cond)
        eng.x.copy_(x0)
        for _ in range(4):  # warm-up + capture + replays
            eng.t.fill_(999)
            eng.step()
    torch.cuda.synchronize()
    ms = {k: [] for k in engines}
    for _ in range(args.rounds):
        for k, eng in engines.items():
            eng.x.copy_(x0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(args.steps):
                if i % 50 == 0:   # the N = 50 chain ends after 50 replays: restart every mode at t = 999 alike
                    eng.t.fill_(999)
                eng.step()
            e1.record()
            torch.cuda.synchronize()
            ms[k].append(e0.elapsed_time(e1) / args.steps)
    say()
    say(f"(a) ms per reverse step, {args.rounds} alternating segments of {args.steps} replays each")
    say(f"{'mode':18s} {'launches/step':>13s} {'mean ms':>8s}  per segment")
    for k, eng in engines.items():
        v = ms[k]
        say(f"{k:18s} {eng.launches_per_step:13d} {sum(v) / len(v):8.3f}  " + " ".join(f"{x:.3f}" for x in v))
    ddim_coef = engines["ddim eta=1"].ddim_coef
    del engines
    torch.cuda.empty_cache()

    # (b) the noise + update alone
    x, e, z = (torch.randn(shape, device=dev) for _ in range(3))
    ids = torch.arange(B, dtype=torch.int64, device=dev)
    t = torch.full((B,), 500, dtype=torch.int64, device=dev)
    td = torch.full((B,), 979, dtype=torch.int64, device=dev)   # a DDIM N = 50 row
    tabs = (diff.betas, diff.sqrt_one_minus_alphas_cumprod, diff.sqrt_recip_alphas, diff.posterior_variance)

    def ddpm_torch():
        z.normal_()
        x.copy_(K.p_sample(x, e, z, t, *tabs))

    def ddim_torch():
        z.normal_()
        K.ddim_step(x, e, z, td, ddim_coef, 1000, out=x)

    cases = {"ddpm: normal_ + p_sample + copy": ddpm_torch,
             "ddpm: p_sample_seeded": lambda: K.p_sample_seeded(x, e, SEED, ids, t, *tabs, out=x),
             "ddim: normal_ + ddim_step": ddim_torch,
             "ddim: ddim_step_seeded": lambda: K.ddim_step_seeded(x, e, SEED, ids, td, ddim_coef, 1000, out=x)}
    us = {k: [] for k in cases}
    for fn in cases.values():
        for _ in range(20):
            fn()
    for _ in range(args.rounds):
        for k, fn in cases.items():
            x.copy_(x0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(200):
                fn()
            e1.record()
            torch.cuda.synchronize()
            us[k].append(1e3 * e0.elapsed_time(e1) / 200)
    say()
    say(f"(b) noise + update alone, us per call over 200 calls, {args.rounds} alternating rounds")
    for k, v in us.items():
        say(f"{k:34s} {sum(v) / len(v):8.1f}  " + " ".join(f"{x:.1f}" for x in v))
    if args.out:
        d = os.path.dirname(args.out)
        if d:
            os.makedirs(d, exist_ok=True)
        with open(args.out, "w") as f:
            f.write("tools/bench_seeded_sampling.py: per-step cost of seeded (in-kernel Philox) vs torch-RNG sampling noise\n")
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
