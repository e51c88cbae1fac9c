"""One call each of the round-2 kernels at full-resolution-like sizes, for `ncu --set full -k regex:"tattn_proj|tattn_long"`."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from cesm_emulator_b200 import kernels as K  # noqa: E402

H, D = 8, 32
torch.manual_seed(0)
freqs = (1.0 / (10000 ** (torch.arange(0, D, 2).float() / D))).cuda()


def tables(F):
    ang = torch.arange(F, device="cuda", dtype=torch.float32)[:, None] * freqs[None]
    return ang.cos().contiguous(), ang.sin().contiguous()


for rep in range(2):
    # long windows: F = 64, 148*2*8 pixel columns
    F, HW = 64, 148 * 2 * 8
    qkv = (torch.randn(F * HW, 3 * H * D, device="cuda") * 0.5).half()
    dout = (torch.randn(F * HW, H * D, device="cuda") * 0.1).half()
    diag = torch.randn(H, 2 * F - 1, device="cuda") * 0.1
    i = torch.arange(F, device="cuda")
    bias = diag[:, (i[None, :] - i[:, None]) + F - 1].contiguous()
    cs, sn = tables(F)
    out, lse = K.tattn_fwd(qkv, bias, cs, sn, 1, F, HW, H, D, D ** -0.5)
    K.tattn_bwd(qkv, bias, cs, sn, out, lse, dout, 1, F, HW, H, D, D ** -0.5)
    # fused projection + attention: the bench workload's full-resolution block (B=2, F=3, 192x288)
    B, F, HW = 2, 3, 192 * 288
    xn = torch.randn(B * F * HW, 64, device="cuda").half()
    w = (torch.randn(3 * H * D, 64, device="cuda") * 0.1).half()
    bias3 = torch.randn(H, F, F, device="cuda")
    cs, sn = tables(F)
    K.tattn_proj_fwd(xn, w, bias3, cs, sn, B, F, HW, H, D, D ** -0.5)
    torch.cuda.synchronize()
print("ok")
