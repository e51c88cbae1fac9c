"""Worker of tests/test_guidance_multigpu_gpu.py: run under `python -m torch.distributed.run --nproc-per-node N`.

Every rank trains a few steps with condition dropout on its B samples of a global batch of N * B, then generates a
seeded guided ensemble sharded over the N ranks.  Rank 0 repeats both alone (a process group of its own, world = 1):
one engine on the whole global batch, and the whole ensemble.  It prints one JSON line: whether the dropout masks of
every step match, and how far the sharded guided ensemble is from the single-rank one.
"""
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from _parity import BASELINE_KW, rel_err  # noqa: E402

SEED = 20261022
KW = dict(BASELINE_KW, ch_mults=(1, 2))


def masks(world_group, B, steps, dev):
    from cesm_emulator_b200 import ops
    from cesm_emulator_b200.engine import TrainEngine
    from cesm_emulator_b200.model import Diffusion, UNet
    torch.manual_seed(0)  # the same weights and the same mask key everywhere
    d = Diffusion(UNet(**KW)).to(dev)
    d.train()
    eng = TrainEngine(d, (B, 1, 16, 16), (B, 1, 3, 16, 16), process_group=world_group, cond_drop_prob=0.5)
    out = []
    for _ in range(steps):
        eng.step(torch.randn(B, 1, 16, 16, device=dev), torch.randn(B, 1, 3, 16, 16, device=dev))
        out.append(eng.keep.clone())
    ops.set_grad_sink(None)
    return torch.stack(out)  # [steps, B]


def main():
    import inference
    from cesm_emulator_b200.model import Diffusion, UNet
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    alone_group = dist.new_group([0])
    B, steps = 2, 6
    mine = masks(None, B, steps, dev)
    gathered = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(gathered, mine)
    torch.manual_seed(0)
    d = Diffusion(UNet(**KW)).to(dev).eval()
    cond = np.random.default_rng(0).standard_normal((2, 3, 1, 32, 32)).astype(np.float32)
    kw = dict(batch_size=2, dpm_steps=4, device=dev, seed=SEED, guidance=2.0)
    sharded = inference.predict_temperature_from_emissions(d, cond, rank=rank, world=world, **kw)
    if rank == 0:
        single = masks(alone_group, B * world, steps, dev)
        alone = inference.predict_temperature_from_emissions(d, cond, rank=0, world=1, **kw)
        out = {"world": world, "masks_equal": bool(torch.equal(torch.cat(gathered, dim=1), single)),
               "dropped": int((single == 0).sum()), "draws": single.numel(),
               "guided_vs_single_rank_worst_rel_err": rel_err(torch.from_numpy(sharded), torch.from_numpy(alone)),
               "finite": bool(np.isfinite(sharded).all())}
        print("MGPU_GUIDANCE_RESULT " + json.dumps(out), flush=True)
    torch.cuda.synchronize()
    dist.barrier()
    os._exit(0)


if __name__ == "__main__":
    main()
