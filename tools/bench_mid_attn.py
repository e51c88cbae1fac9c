"""use_mid_attn=True on the B200: (a) the bottleneck softmax-attention core (csrc/mid_attn.cu) against its MUFU and
tensor-core bounds and against stock torch SDPA on the same inputs; (b) the bench training step and a 16-field
sampling step with the block off and on, alternated in one process.

    python tools/bench_mid_attn.py [--reps 20] [--steps 10] [--rounds 3] [--core-only]

Prints the device name, power limit and max SM clock first: every number below belongs to them.
(a) Each call is timed with CUDA events around the call only; a 256 MB buffer (> the 126 MB L2) is overwritten
    before every call, so q|k|v start in HBM.  FLOPs are algorithmic: forward 4 n^2 d per (image, head), backward
    2.5x that (10 n^2 d; the kernels execute 14 n^2 d: S and dP are recomputed in both backward passes).  exp count:
    n^2 per (image, head) forward, 2 n^2 backward (P is recomputed in the dQ and in the dK/dV pass).  MUFU bound =
    16 ex2 / clock / SM x 148 SMs x max SM clock.  SDPA runs on its preferred layout (contiguous [NI, H, n, 32]
    q, k, v made from the same fp16 values) with whichever backend torch picks.
(b) TrainEngine.step_resident (CUDA graph) at bench.py's workload (config/baseline, B=2, K=3, 192x288) and
    SampleEngine.step (16 fields, F=1, 192x288); the "off" and "on" engines are built in one process and timed in
    alternating segments.  The "on" training engine is captured second, so its graph's once-per-step weight re-pack
    also covers the "off" model's weights (one kernel over a few MB: conservative for "on")."""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CORE_SHAPES = [  # (label, NI, n, H, backward?)
    ("bench train step, 48x72 bottleneck", 6, 3456, 8, True),
    ("config/baseline crop 128x128, 32x32", 6, 1024, 8, True),
    ("sampling step, 16 fields F=1", 16, 3456, 8, False),
    ("more_blocks at 192x288, 24x36", 6, 864, 8, True),
    ("ch_mults=(1,2) at 192x288, 96x144", 1, 13824, 8, True),
]
D = 32


def device_line():
    import torch
    name = torch.cuda.get_device_name(0)
    q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                       capture_output=True, text=True)
    pl, clk = (s.strip() for s in q.stdout.strip().split(","))
    return name, float(pl), float(clk)


def timed(fn, reps, flush):
    import torch
    fn()
    torch.cuda.synchronize()
    tot = 0.0
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        tot += e0.elapsed_time(e1)
    return tot / reps


def core(args, mufu_per_s):
    import torch
    import torch.nn.functional as Fn
    from cesm_emulator_b200 import kernels as K
    dev = torch.device("cuda:0")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    scale = D ** -0.5
    print("\n(a) core: time per call (ms), algorithmic TFLOP/s, exp/s and share of the MUFU bound; SDPA fp16 alongside")
    print(f"{'shape':40s} {'NI':>3s} {'n':>6s} {'pass':4s} {'mattn ms':>9s} {'TFLOP/s':>8s} {'Gexp/s':>8s} {'MUFU %':>7s} "
          f"{'sdpa ms':>8s} {'sdpa TF/s':>9s} {'mattn/sdpa':>10s} {'max|diff|/max':>13s}")
    for label, NI, n, H, bwd in CORE_SHAPES:
        g = torch.Generator(device=dev).manual_seed(n)
        qkv = torch.randn(NI * n, 3 * H * D, device=dev, generator=g).half()
        dout = torch.randn(NI * n, H * D, device=dev, generator=g).half()
        out, lse = K.mattn_fwd(qkv, NI, n, H, D, scale)
        q, k, v = (qkv.view(NI, n, 3, H, D)[:, :, i].permute(0, 2, 1, 3).contiguous().requires_grad_(True) for i in range(3))
        do4 = dout.view(NI, n, H, D).permute(0, 2, 1, 3).contiguous()
        with torch.no_grad():
            o_s = Fn.scaled_dot_product_attention(q, k, v, scale=scale)
        o_m = out.view(NI, n, H, D).permute(0, 2, 1, 3).float()
        diff = ((o_m - o_s.float()).abs().max() / o_s.float().abs().max()).item()
        t_f = timed(lambda: K.mattn_fwd(qkv, NI, n, H, D, scale), args.reps, flush)

        def sdpa_f():
            with torch.no_grad():
                Fn.scaled_dot_product_attention(q, k, v, scale=scale)
        t_sf = timed(sdpa_f, args.reps, flush)
        fl = 4.0 * NI * H * n * n * D
        ex = float(NI * H * n * n)
        print(f"{label:40s} {NI:3d} {n:6d} fwd  {t_f:9.4f} {fl / t_f / 1e9:8.1f} {ex / t_f / 1e6:8.0f} "
              f"{100 * ex / t_f * 1e3 / mufu_per_s:6.1f}% {t_sf:8.4f} {fl / t_sf / 1e9:9.1f} {t_f / t_sf:10.2f} {diff:13.2e}")
        if not bwd:
            continue
        dq = K.mattn_bwd(qkv, out, lse, dout, NI, n, H, D, scale)
        o_g = Fn.scaled_dot_product_attention(q, k, v, scale=scale)
        gq, gk, gv = torch.autograd.grad(o_g, (q, k, v), do4, retain_graph=True)
        hid = H * D
        gd = 0.0
        for i, gs in enumerate((gq, gk, gv)):
            gm = dq[:, i * hid:(i + 1) * hid].view(NI, n, H, D).permute(0, 2, 1, 3).float()
            gd = max(gd, ((gm - gs.float()).abs().max() / gs.float().abs().max()).item())
        t_b = timed(lambda: K.mattn_bwd(qkv, out, lse, dout, NI, n, H, D, scale), args.reps, flush)
        t_sb = timed(lambda: torch.autograd.grad(o_g, (q, k, v), do4, retain_graph=True), args.reps, flush)
        flb, exb = 2.5 * fl, 2 * ex
        print(f"{label:40s} {NI:3d} {n:6d} bwd  {t_b:9.4f} {flb / t_b / 1e9:8.1f} {exb / t_b / 1e6:8.0f} "
              f"{100 * exb / t_b * 1e3 / mufu_per_s:6.1f}% {t_sb:8.4f} {flb / t_sb / 1e9:9.1f} {t_b / t_sb:10.2f} {gd:13.2e}")
        del q, k, v, o_g, gq, gk, gv
        torch.cuda.empty_cache()


def end_to_end(args):
    import torch
    from cesm_emulator_b200 import ops
    from cesm_emulator_b200.engine import SampleEngine, TrainEngine
    from cesm_emulator_b200.model import Diffusion, UNet
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from _parity import BASELINE_KW
    dev = torch.device("cuda:0")
    H, W = 192, 288

    def seg(fn, steps):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    def report(what, res, unit, per):
        import statistics
        med = {k: statistics.median(v) for k, v in res.items()}
        for k in ("off", "on"):
            print(f"  {what} use_mid_attn={k:3s}: " + " ".join(f"{x:.3f}" for x in res[k]) +
                  f" ms  (median {med[k]:.3f} ms, {per / med[k] * 1e3:.1f} {unit})")
        print(f"  {what} on - off: {med['on'] - med['off']:+.3f} ms ({100 * (med['on'] / med['off'] - 1):+.1f} %)")

    print(f"\n(b) end to end, {args.rounds} alternating segments of {args.steps} steps per arm")
    engs = {}
    for k in ("off", "on"):
        torch.manual_seed(0)
        d = Diffusion(UNet(**dict(BASELINE_KW, use_mid_attn=(k == "on"))), timesteps=1000).to(dev)
        d.train()
        e = TrainEngine(d, (2, 1, H, W), (2, 1, 3, H, W))
        torch.manual_seed(1)
        e.x0.normal_()
        e.cond.normal_()
        for _ in range(3 + 3):
            e.step_resident()
        engs[k] = e
    res = {"off": [], "on": []}
    for _ in range(args.rounds):
        for k in ("off", "on"):
            res[k].append(seg(engs[k].step_resident, args.steps))
    print(f"  training step launches: off {engs['off'].launches_per_step}, on {engs['on'].launches_per_step}")
    report("train step (B=2, K=3)", res, "samples/s", 2)
    del engs
    ops.set_grad_sink(None)
    torch.cuda.empty_cache()

    engs = {}
    for k in ("off", "on"):
        torch.manual_seed(0)
        d = Diffusion(UNet(**dict(BASELINE_KW, use_mid_attn=(k == "on"))), timesteps=1000).to(dev)
        d.eval()
        for p in d.parameters():
            p.requires_grad_(False)
        e = SampleEngine(d, (16, 1, H, W))
        torch.manual_seed(2)
        e.cond.normal_()
        e.x.normal_()
        e.t.fill_(999)
        for _ in range(4):
            e.step()
        engs[k] = e
    res = {"off": [], "on": []}
    for _ in range(args.rounds):
        for k in ("off", "on"):
            engs[k].t.fill_(999)
            res[k].append(seg(engs[k].step, args.steps))
    print(f"  sampling step launches: off {engs['off'].launches_per_step}, on {engs['on'].launches_per_step}")
    report("sampling step (16 fields)", res, "field-steps/s", 16)
    assert all(bool(torch.isfinite(e.x).all()) for e in engs.values())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--core-only", action="store_true")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_mid_attn.py needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    name, pl, clk = device_line()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    mufu = 16 * sms * clk * 1e6
    print(f"device: {name}, power limit {pl:.0f} W, max SM clock {clk:.0f} MHz, {sms} SMs; torch {torch.__version__}")
    print(f"MUFU ex2 bound: 16 / clock / SM -> {mufu / 1e12:.2f} T exp/s; dense fp16 tensor data-sheet rate 2250 TFLOP/s "
          f"(tcgen05; these kernels use mma.sync)")
    core(args, mufu)
    if not args.core_only:
        end_to_end(args)


if __name__ == "__main__":
    main()
