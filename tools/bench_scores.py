#!/usr/bin/env python
"""Time cesm_ensemble_scores (kernels.ensemble_scores) with CUDA events over many calls after a warm-up.

Sizes: T = 64 years of n = m = 50 members at 192x288 (1.4 GB of input, above the 126 MB L2, so every call reads HBM),
and n = 1024 generated against m = 50 target members at T = 4.  Reports ms per call, achieved GB/s over the bytes the
call must move (both inputs read once, the five maps and the histogram written once) and that time's share of the
HBM bound at 7.7 TB/s (NVIDIA's HGX B200 data-sheet bandwidth per GPU).  The card's name, power limit and max SM clock
are read in the same run.

    python tools/bench_scores.py [--calls 20] [--warmup 3] [--out profiles/x.json]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_BYTES_PER_S = 7.7e12


def _card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def bench(T, n, m, HW, calls, warmup):
    from cesm_emulator_b200 import _lib
    from cesm_emulator_b200 import kernels as K
    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randn((T, n, HW), generator=g, device="cuda")
    y = torch.randn((T, m, HW), generator=g, device="cuda")
    for _ in range(warmup):
        K.ensemble_scores(x, y)
    torch.cuda.synchronize()
    before = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(calls):
        K.ensemble_scores(x, y)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / calls
    nbytes = 4 * T * HW * (n + m + 5) + 8 * T * (n + 1)
    return {"T": T, "n": n, "m": m, "HW": HW, "ms": round(ms, 4), "GB": round(nbytes / 1e9, 3),
            "GB_per_s": round(nbytes / ms / 1e6, 1), "share_of_hbm_bound": round(nbytes / HBM_BYTES_PER_S * 1e3 / ms, 3),
            "launches_per_call": (_lib.launch_count() - before) / calls}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_scores.py needs a CUDA device")
    res = {"card": _card(), "hbm_bound_bytes_per_s": HBM_BYTES_PER_S,
           "runs": [bench(64, 50, 50, 192 * 288, a.calls, a.warmup), bench(4, 1024, 50, 192 * 288, a.calls, a.warmup)]}
    print(json.dumps(res, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
