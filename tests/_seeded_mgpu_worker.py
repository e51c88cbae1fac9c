"""Worker of tests/test_seeded_multigpu_gpu.py: run under `python -m torch.distributed.run --nproc-per-node N`.

Every rank generates the same (years, members) ensemble with `predict_temperature_from_emissions`, sharded over the
N ranks, once without a seed and once with one.  The members of a year share their condition, so without a seed
they differ only through the noise their rank draws.  Rank 0 also generates the seeded ensemble alone (world = 1)
and prints one JSON line: how far the sharded seeded ensemble is from the single-rank one, and how many member
pairs of a year coincide with and without the seed.
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

SEED = 20261021


def coinciding_pairs(pred, tol=1e-2):
    T, M = pred.shape[:2]
    t = torch.from_numpy(pred)
    return sum(rel_err(t[y, a], t[y, b]) < tol for y in range(T) for a in range(M) for b in range(a))


def main():
    import inference
    from cesm_emulator_b200.model import Diffusion, UNet
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    torch.manual_seed(0)   # the same weights on every rank; torch's CUDA generator starts equal on every rank anyway
    d = Diffusion(UNet(**dict(BASELINE_KW, ch_mults=(1, 2)))).to(dev).eval()
    years, members, bs = 2, 4, 2
    cond = np.random.default_rng(0).standard_normal((years, 1, 1, 32, 32)).astype(np.float32)
    cond = np.repeat(cond, members, axis=1)        # one condition per year, shared by its members
    kw = dict(batch_size=bs, ddim_steps=10, eta=1.0, device=dev)
    unseeded = inference.predict_temperature_from_emissions(d, cond, rank=rank, world=world, **kw)
    seeded = inference.predict_temperature_from_emissions(d, cond, rank=rank, world=world, seed=SEED, **kw)
    if rank == 0:
        alone = inference.predict_temperature_from_emissions(d, cond, rank=0, world=1, seed=SEED, **kw)
        worst = max(rel_err(torch.from_numpy(seeded[y, m]), torch.from_numpy(alone[y, m]))
                    for y in range(years) for m in range(members))
        out = {"world": world, "fields": years * members, "member_pairs": years * members * (members - 1) // 2,
               "seeded_vs_single_rank_worst_rel_err": worst,
               "coinciding_pairs_seeded": coinciding_pairs(seeded),
               "coinciding_pairs_unseeded": coinciding_pairs(unseeded),
               "finite": bool(np.isfinite(seeded).all() and np.isfinite(unseeded).all())}
        print("MGPU_SEEDED_RESULT " + json.dumps(out), flush=True)
    torch.cuda.synchronize()
    dist.barrier()
    os._exit(0)


if __name__ == "__main__":
    main()
