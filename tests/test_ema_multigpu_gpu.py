"""The weight EMA under data-parallel training: after graph-replayed steps the parameters and the EMA are bit-identical
on every rank.  Needs >= 2 GPUs (`python -m pytest tests/test_ema_multigpu_gpu.py -m gpu`); skipped on a 1-GPU box."""
import json
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_ema_bit_identical_on_every_rank(cuda):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least 2 GPUs")
    world = 2
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}",
           "--master-addr", "127.0.0.1", "--master-port", "29534", os.path.join(ROOT, "tests", "_ema_mgpu_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("MGPU_EMA_RESULT ")][-1]
    res = json.loads(line[len("MGPU_EMA_RESULT "):])
    print(line)
    assert res["world"] == world and res["graph"] and res["steps"] + res["skipped_steps"] == 6, res
    assert res["params_in_sync"] is True and res["ema_in_sync"] is True, res
    assert res["ema_differs_from_params"] is True, res   # past ema_start: the EMA is not a copy, the check is not vacuous
