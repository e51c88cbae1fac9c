"""Seeded ensemble generation sharded over 2 ranks: the same prediction as one rank computes alone, with every member
of a year its own field.  Without a seed the worker only reports how many member pairs coincide.  Needs >= 2 GPUs
(`python -m pytest tests/test_seeded_multigpu_gpu.py -m gpu`); skipped on a 1-GPU box."""
import json
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_seeded_ensemble_does_not_depend_on_world_size(cuda):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least 2 GPUs")
    world = 2
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", "29536", os.path.join(ROOT, "tests", "_seeded_mgpu_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("MGPU_SEEDED_RESULT ")][-1]
    res = json.loads(line[len("MGPU_SEEDED_RESULT "):])
    print(line)
    assert res["world"] == world and res["finite"], res
    assert res["seeded_vs_single_rank_worst_rel_err"] < 1e-2, res
    assert res["coinciding_pairs_seeded"] == 0, res
