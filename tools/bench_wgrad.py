"""Time the tcgen05 weight-gradient kernel on the shapes of the baseline model (run on the GPU box).

    python tools/bench_wgrad.py            # CASE=substring times only the matching shapes
"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cesm_emulator_b200 import kernels as K  # noqa: E402
from tools.bench_igemm import timeit  # noqa: E402


def main():
    dev = "cuda"
    torch.manual_seed(0)
    cases = [  # (name, n, h, w, cin, cout, taps)
        ("L0 3x3 64->64", 6, 192, 288, 64, 64, 9),
        ("L0 3x3 128->64", 6, 192, 288, 128, 64, 9),
        ("L1 3x3 128->128", 6, 96, 144, 128, 128, 9),
        ("L2 3x3 256->256", 6, 48, 72, 256, 256, 9),
        ("L0 1x1 64->768", 6, 192, 288, 64, 768, 1),
        ("L0 1x1 256->64", 6, 192, 288, 256, 64, 1),
        ("L1 1x1 128->768", 6, 96, 144, 128, 768, 1),
        ("L2 1x1 256->768", 6, 48, 72, 256, 768, 1),
    ]
    only = os.environ.get("CASE")
    for name, n, h, w, cin, cout, taps in cases:
        if only and only not in name:
            continue
        x = torch.randn(n, h, w, cin, device=dev).half()
        dy = torch.randn(n, h, w, cout, device=dev).half()
        tp = K.TAPS_3x3 if taps == 9 else K.TAPS_1x1
        into = torch.zeros(cout, taps, cin, device=dev)
        layout = (taps * cin, 1, [t * cin for t in range(taps)])
        ms = timeit(lambda: K.wgrad(x, dy, taps=tp, into=into, layout=layout))
        fl = 2.0 * n * h * w * cout * taps * cin
        by = 2.0 * n * h * w * (cin + cout)
        print(f"{name:22s} {ms*1e3:8.1f} us  {fl/ms/1e9:7.1f} TFLOP/s  {by/ms/1e6:7.0f} GB/s")


if __name__ == "__main__":
    main()
