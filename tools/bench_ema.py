"""Cost of the weight EMA fused into the optimizer step, on the B200.

    python tools/bench_ema.py [--rounds 6] [--out profiles/r08_ema.txt]

Prints the device name, power limit and max SM clock first: every number below belongs to them.
(a) The optimizer launch sequence alone (grad_sumsq -> adamw_clip -> scaler_update), `cesm_adamw_step` against
    `cesm_adamw_ema_step`, at the trainable-parameter counts of config/baseline and config/more_blocks.  Each is timed
    with CUDA events over segments of 100 back-to-back calls, the two alternating, `--rounds` segments each.  The
    buffers (28 or 36 B per parameter: 372 MB and more) exceed the 126 MB L2, so every call streams from HBM.
    GB/s = (28 or 36 B) x parameters / time per call; grad_sumsq's extra 4 B read of the gradient is not counted.
(b) The graph-replayed training step at bench.py's workload (config/baseline, B = 2, K = 3, 192x288), one TrainEngine
    without and one with the EMA (decay 0.9999) in one process, timed in alternating segments of 20 replays.  Both
    models exist before either graph is captured, so each replay's weight re-pack covers both models' weights: the
    absolute step time is a little above bench.py's; the difference between the two is what this measures.
"""
import argparse
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

BASELINE_KW = dict(in_channels=2, out_channels=1, base_ch=64, ch_mults=(1, 2, 4), num_res_blocks=2, time_dim=124,
                   groups=8, dropout=0.0, use_checkpoint=False)          # config/baseline "unet"
MORE_BLOCKS_KW = dict(BASELINE_KW, ch_mults=(1, 2, 4, 8), num_res_blocks=6)  # config/more_blocks "unet"
B, K, H, W = 2, 3, 192, 288
DECAY = 0.9999


def device_line():
    import torch
    name = torch.cuda.get_device_name(0)
    q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                       capture_output=True, text=True)
    pl, clk = (s.strip() for s in q.stdout.strip().split(","))
    return name, float(pl), float(clk)


def trainable(kw):
    from cesm_emulator_b200.model import UNet
    return sum(p.numel() for p in UNet(**kw).parameters() if p.requires_grad)


def spread(xs):
    return f"median {statistics.median(xs):.4f}, min {min(xs):.4f}, max {max(xs):.4f}"


def time_segment(fn, n):
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def bench_optimizer(say, rounds):
    import torch
    from cesm_emulator_b200 import _lib, kernels as K
    dev = torch.device("cuda", 0)
    for arch, kw in (("baseline", BASELINE_KW), ("more_blocks", MORE_BLOCKS_KW)):
        n = trainable(kw)
        n_pad = (n + 3) // 4 * 4
        gen = torch.Generator(device=dev).manual_seed(0)
        p, g = (torch.randn(n_pad, device=dev, generator=gen) for _ in range(2))
        m, v, e = torch.zeros(n_pad, device=dev), torch.zeros(n_pad, device=dev), p.clone()
        st = torch.zeros(K.OPT_STATE_FLOATS)
        st[K.OPT_LR], st[K.OPT_WD], st[K.OPT_SCALE] = 1e-6, 0.0, 1.0
        state, partials = st.to(dev), torch.zeros(_lib.load().cesm_adamw_partials(), device=dev)
        plain = lambda: K.adamw_step(p, g, m, v, partials, state, 0.9, 0.999, 1e-8, 1.0)
        ema = lambda: K.adamw_ema_step(p, g, m, v, e, partials, state, 0.9, 0.999, 1e-8, 1.0, DECAY, 0)
        for fn in (plain, ema):  # warm-up
            time_segment(fn, 20)
        t = {"off": [], "on": []}
        for _ in range(rounds):
            t["off"].append(time_segment(plain, 100) * 1e3)
            t["on"].append(time_segment(ema, 100) * 1e3)
        assert int(state[K.OPT_SKIPPED].item()) == 0
        say(f"\n(a) optimizer launch sequence, {arch}: {n:,} trainable parameters "
            f"({28 * n / 1e6:.0f} MB without, {36 * n / 1e6:.0f} MB with the EMA per call)")
        for key, bpp in (("off", 28), ("on", 36)):
            us = t[key]
            gbs = [bpp * n / (x * 1e-6) / 1e9 for x in us]
            say(f"  EMA {key:3s}: us/call {spread(us)};  GB/s on {bpp} B/param {spread(gbs)}")
        r_gbs = statistics.median([36 / x for x in t["on"]]) / statistics.median([28 / x for x in t["off"]])
        r_t = statistics.median(t["on"]) / statistics.median(t["off"])
        say(f"  EMA on / off: achieved GB/s {r_gbs:.3f}, time per call {r_t:.3f} (bytes ratio 36/28 = {36 / 28:.3f})")
        del p, g, m, v, e


def bench_step(say, rounds):
    import torch
    from cesm_emulator_b200.engine import TrainEngine
    from cesm_emulator_b200.model import Diffusion, UNet
    dev = torch.device("cuda", 0)
    engines = {}
    for key, kw in (("off", {}), ("on", dict(ema_decay=DECAY))):
        torch.manual_seed(0)
        d = Diffusion(UNet(**BASELINE_KW), timesteps=1000).to(dev)
        d.train()
        eng = TrainEngine(d, (B, 1, H, W), (B, 1, K, H, W), **kw)
        g = torch.Generator().manual_seed(1)
        eng.x0.copy_(torch.randn(B, 1, H, W, generator=g))
        eng.cond.copy_(torch.randn(B, 1, K, H, W, generator=g))
        engines[key] = eng
    for _ in range(2):      # eager warm-up steps of both engines: every weight is registered before any capture
        for eng in engines.values():
            eng.step_resident()
    for _ in range(4):      # capture, then replays
        for eng in engines.values():
            eng.step_resident()
    torch.cuda.synchronize()
    assert all(eng.graph is not None for eng in engines.values())
    lp = {k: eng.launches_per_step for k, eng in engines.items()}
    t = {"off": [], "on": []}
    for r in range(rounds):
        order = ("off", "on") if r % 2 == 0 else ("on", "off")
        for key in order:
            t[key].append(time_segment(engines[key].step_resident, 20))
    diffs = [a - b for a, b in zip(t["on"], t["off"])]
    say(f"\n(b) graph-replayed training step, config/baseline B={B} K={K} {H}x{W} (library launches per step: "
        f"{lp['off']} without, {lp['on']} with the EMA), {rounds} alternating segments of 20 replays")
    for key in ("off", "on"):
        say(f"  EMA {key:3s}: ms/step {spread(t[key])}")
    say(f"  on - off per round (ms): {', '.join(f'{x:+.4f}' for x in diffs)}; median {statistics.median(diffs):+.4f}")
    skipped = {k: int(eng.opt.state[5].item()) for k, eng in engines.items()}
    say(f"  skipped steps: {skipped}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--out", default="", help="also write the report to this file")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_ema.py needs a CUDA device")
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    name, pl, clk = device_line()
    say(f"device: {name}, power limit {pl:.0f} W, max SM clock {clk:.0f} MHz")
    bench_optimizer(say, args.rounds)
    bench_step(say, args.rounds)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
