"""Host tests of the weight EMA: argument validation, the refusal on host tensors, and the checkpoint paths
(train.save_checkpoint writes "ema" in the UNet state-dict layout; inference.load_diffusion_from_checkpoint(ema=True)
loads it, and refuses a checkpoint without one).  The kernel and the engine are tests/test_ema_gpu.py's."""
import os

import numpy as np
import pytest
import torch

GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.mark.parametrize("decay,start", [(True, 0), (float("nan"), 0), (float("inf"), 0), (-0.1, 0), (1.0, 0),
                                         (1.5, 0), ("0.9", 0), (0.9, -1), (0.9, 1.5), (0.9, True), (0.9, "2")])
def test_invalid_ema_arguments_raise(decay, start):
    from torch import nn
    from cesm_emulator_b200.engine import FusedAdamW, TrainEngine, check_ema_args
    from cesm_emulator_b200.model import Diffusion
    with pytest.raises(ValueError):
        check_ema_args(decay, start)
    with pytest.raises(ValueError):  # before the optimizer touches its buckets
        FusedAdamW(None, 1e-3, (0.9, 0.999), 0.0, 1e-8, 1.0, ema_decay=decay, ema_start=start)
    with pytest.raises(ValueError):
        TrainEngine(Diffusion(nn.Linear(1, 1)), (1, 1, 8, 8), (1, 1, 3, 8, 8), ema_decay=decay, ema_start=start)


def test_valid_ema_arguments():
    from cesm_emulator_b200.engine import check_ema_args
    assert check_ema_args(None, 0) == (None, 0)
    assert check_ema_args(0, 0) == (0.0, 0)
    assert check_ema_args(0.9999, 3) == (0.9999, 3)
    assert check_ema_args(np.float32(0.5), np.int64(2)) == (0.5, 2)


def test_ema_on_host_tensors_raises():
    """The gloo / CPU path of TrainEngine has no fused optimizer step, so there is no EMA there and no fallback."""
    from torch import nn
    from cesm_emulator_b200 import kernels as K
    from cesm_emulator_b200._lib import CesmError
    from cesm_emulator_b200.engine import TrainEngine
    from cesm_emulator_b200.model import Diffusion
    with pytest.raises(RuntimeError, match="EMA"):
        TrainEngine(Diffusion(nn.Linear(1, 1)), (1, 1, 8, 8), (1, 1, 3, 8, 8), ema_decay=0.9)
    z = torch.zeros(16)
    with pytest.raises(CesmError):
        K.adamw_ema_step(z, z, z, z, z, torch.zeros(1024), torch.zeros(K.OPT_STATE_FLOATS), 0.9, 0.999, 1e-8, 1.0,
                         0.9, 0)


class _EngineWithEma:
    """What train.save_checkpoint reads of a TrainEngine, with a given EMA state dict."""

    def __init__(self, ema):
        self.has_ema = True
        self._ema = ema
        self.opt = torch.optim.AdamW([torch.nn.Parameter(torch.zeros(1))])

    def ema_state_dict(self):
        return self._ema


def _tiny_checkpoint(tmp_path, with_ema: bool):
    """A checkpoint of the tiny reference UNet written by train.save_checkpoint on the CPU; its EMA (if any) is the
    model's weights transformed so that every trainable tensor differs from "model"."""
    import train as train_entry
    from cesm_emulator_b200.model import Diffusion
    ref = torch.load(os.path.join(GOLD, "ref_ckpt_tiny.pt"), map_location="cpu", weights_only=False)
    diffusion = Diffusion(train_entry.build_model_from_config(ref["config"]["unet"]), timesteps=1000)
    diffusion.model.load_state_dict(ref["model"], strict=True)
    trainable = {n for n, p in diffusion.model.named_parameters() if p.requires_grad}
    ema = {k: (0.5 * v + 0.25 if k in trainable else v.clone()) for k, v in diffusion.model.state_dict().items()}
    path = str(tmp_path / ("ema.pt" if with_ema else "plain.pt"))
    engine = _EngineWithEma(ema)
    engine.has_ema = with_ema
    train_entry.save_checkpoint(path, 1, diffusion, engine, ref["config"])
    return path, ref["model"], ema, trainable


def test_checkpoint_ema_loads_into_unet_strict(tmp_path):
    import train as train_entry
    path, model_sd, ema, trainable = _tiny_checkpoint(tmp_path, with_ema=True)
    ckpt = torch.load(path, map_location="cpu", weights_only=False)
    assert set(ckpt) == {"epoch", "model", "diffusion_buffers", "optimizer", "config", "ema"}
    assert list(ckpt["ema"]) == list(ckpt["model"])
    unet = train_entry.build_model_from_config(ckpt["config"]["unet"])
    unet.load_state_dict(ckpt["ema"], strict=True)
    for k, v in unet.state_dict().items():
        assert torch.equal(v, ema[k]), k
    frozen = [k for k in ckpt["model"] if k not in trainable]
    assert frozen and all(torch.equal(ckpt["ema"][k], ckpt["model"][k]) for k in frozen)


def test_load_diffusion_from_checkpoint_ema(tmp_path):
    import inference
    path, model_sd, ema, _ = _tiny_checkpoint(tmp_path, with_ema=True)
    d_ema, _ = inference.load_diffusion_from_checkpoint(path, "cpu", ema=True)
    d_raw, _ = inference.load_diffusion_from_checkpoint(path, "cpu")
    for k, v in d_ema.model.state_dict().items():
        assert torch.equal(v, ema[k]), k
    for k, v in d_raw.model.state_dict().items():
        assert torch.equal(v, model_sd[k]), k


def test_load_diffusion_from_checkpoint_without_ema_fails(tmp_path):
    import inference
    path, _, _, _ = _tiny_checkpoint(tmp_path, with_ema=False)
    assert "ema" not in torch.load(path, map_location="cpu", weights_only=False)
    with pytest.raises(KeyError, match='"ema"'):
        inference.load_diffusion_from_checkpoint(path, "cpu", ema=True)
    inference.load_diffusion_from_checkpoint(path, "cpu")  # the raw weights still load

