"""Condition dropout and guided sampling over 2 ranks: the dropout masks of a global batch split over the ranks equal
those of one rank training on the whole batch, and a seeded guided ensemble sharded over the ranks equals the one a
single rank generates.  Needs >= 2 GPUs (`python -m pytest tests/test_guidance_multigpu_gpu.py -m gpu`); skipped on a
1-GPU box."""
import json
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_masks_and_guided_fields_do_not_depend_on_world_size(cuda):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least 2 GPUs")
    world = 2
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", "29537",
           os.path.join(ROOT, "tests", "_guidance_mgpu_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("MGPU_GUIDANCE_RESULT ")][-1]
    res = json.loads(line[len("MGPU_GUIDANCE_RESULT "):])
    print(line)
    assert res["world"] == world and res["finite"], res
    assert res["masks_equal"] and 0 < res["dropped"] < res["draws"], res
    assert res["guided_vs_single_rank_worst_rel_err"] < 1e-2, res
