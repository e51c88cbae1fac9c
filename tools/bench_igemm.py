"""Time the implicit-GEMM kernel on the shapes of the baseline model (run on the GPU box).

    python tools/bench_igemm.py            # CASE=substring: only the matching shapes; PLAIN=1: 3 ungraphed calls each
"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cesm_emulator_b200 import kernels as K  # noqa: E402


def timeit(fn, iters=20):
    """Device time per call: the calls are captured into a CUDA graph so that the ~40 us of
    Python/ctypes work per launch does not become the measured cadence."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(iters):
            fn()
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def main():
    dev = "cuda"
    torch.manual_seed(0)
    cases = [  # (name, n, h, w, cin, cin1, cout, taps, gn)
        ("L0 3x3 64->64", 6, 192, 288, 64, 0, 64, 9, False),
        ("L0 3x3 64->64 +gn", 6, 192, 288, 64, 0, 64, 9, True),
        ("L0 3x3 128->64 cat", 6, 192, 288, 64, 64, 64, 9, False),
        ("L1 3x3 128->128", 6, 96, 144, 128, 0, 128, 9, False),
        ("L2 3x3 256->256", 6, 48, 72, 256, 0, 256, 9, False),
        ("L2 3x3 512->256 cat", 6, 48, 72, 256, 256, 256, 9, False),
        ("L3 3x3 512->512", 6, 24, 36, 512, 0, 512, 9, False),
        ("L1 3x3 256->128 cat", 6, 96, 144, 128, 128, 128, 9, False),
        ("L0 1x1 64->768", 6, 192, 288, 64, 0, 768, 1, False),
        ("L0 1x1 256->64", 6, 192, 288, 256, 0, 64, 1, False),
        ("L0 1x1 768->64", 6, 192, 288, 768, 0, 64, 1, False),
        ("L1 1x1 128->768", 6, 96, 144, 128, 0, 768, 1, False),
        ("L2 1x1 256->768", 6, 48, 72, 256, 0, 768, 1, False),
    ]
    only = os.environ.get("CASE")
    plain = os.environ.get("PLAIN")  # no graph, 3 calls: for ncu
    for name, n, h, w, c0, c1, cout, taps, gn in cases:
        if only and only not in name:
            continue
        x0 = torch.randn(n, h, w, c0, device=dev).half()
        x1 = torch.randn(n, h, w, c1, device=dev).half() if c1 else None
        wt = (torch.randn(cout, taps * (c0 + c1), device=dev) * 0.05).half()
        bias = torch.randn(cout, device=dev)
        tp = K.TAPS_3x3 if taps == 9 else K.TAPS_1x1
        sums = torch.empty(2, 8, 2, device=dev) if gn else None
        out = torch.empty(n, h, w, cout, device=dev, dtype=torch.float16)
        if plain:
            for _ in range(3):
                K.igemm(x0, wt, a1=x1, taps=tp, bias=bias, out=out, gn_sums=sums, gn_frames=3)
            torch.cuda.synchronize()
            continue
        ms = timeit(lambda: K.igemm(x0, wt, a1=x1, taps=tp, bias=bias, out=out, gn_sums=sums, gn_frames=3))
        fl = 2.0 * n * h * w * cout * taps * (c0 + c1)
        by = 2.0 * n * h * w * (c0 + c1 + cout)
        print(f"{name:22s} {ms*1e3:8.1f} us  {fl/ms/1e9:7.1f} TFLOP/s  {by/ms/1e6:7.0f} GB/s")


if __name__ == "__main__":
    main()
