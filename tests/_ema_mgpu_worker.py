"""Worker of tests/test_ema_multigpu_gpu.py: run under `python -m torch.distributed.run --nproc-per-node N` on N GPUs.

N ranks start from different weights (the engine broadcasts rank 0's) and train 6 steps (2 eager + capture + 3 replays)
on DIFFERENT data with the weight EMA on.  The parameters are bit-identical on every rank after the all-reduce and the
AdamW step, so the EMA, computed from them in the same kernel with no collective of its own, must be too.
Rank 0 prints one JSON line.
"""
import json
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from _parity import BASELINE_KW  # noqa: E402


def signature(flat):
    bits = flat.view(torch.int32).to(torch.int64)
    return torch.stack([bits.sum(), (bits * (torch.arange(bits.numel(), device=flat.device) % 8191 + 1)).sum()])


def in_sync(flat, world):
    sig = signature(flat)
    sigs = [torch.zeros_like(sig) for _ in range(world)]
    dist.all_gather(sigs, sig)
    return all(torch.equal(sigs[0], s) for s in sigs)


def main():
    from cesm_emulator_b200.engine import TrainEngine
    from cesm_emulator_b200.model import Diffusion, UNet
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    B, K, H, W = 1, 3, 32, 48
    g = torch.Generator().manual_seed(200 + rank)   # different data per rank
    torch.manual_seed(rank)                         # different initial weights per rank
    d = Diffusion(UNet(**BASELINE_KW)).to(dev)
    d.train()
    eng = TrainEngine(d, (B, 1, H, W), (B, 1, K, H, W), lr=1e-3, ema_decay=0.9, ema_start=2)
    torch.manual_seed(1234 + rank)                  # different (t, noise) draws per rank
    losses = [eng.step(torch.randn(B, 1, H, W, generator=g), torch.randn(B, 1, K, H, W, generator=g)).item()
              for _ in range(6)]
    out = {"world": world, "graph": eng.graph is not None, "steps": int(eng.opt.state[0]),
           "skipped_steps": int(eng.opt.state[5]), "losses_rank0": losses,
           "params_in_sync": in_sync(eng.opt.p, world), "ema_in_sync": in_sync(eng.opt.ema, world),
           "ema_differs_from_params": not torch.equal(eng.opt.ema, eng.opt.p)}
    if rank == 0:
        print("MGPU_EMA_RESULT " + json.dumps(out), flush=True)
    torch.cuda.synchronize()
    dist.barrier()
    os._exit(0)


if __name__ == "__main__":
    main()
