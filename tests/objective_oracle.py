"""fp32 CPU reference of the weighted diffusion objective (v-prediction target, per-timestep Min-SNR weights), the
checker for `ops.DiffusionLossFn` and `Diffusion(prediction_type=...).loss(..., weights=...)`.

The UNet and q_sample are the existing oracle's (`oracle.cesm_oracle`); only the target and the weighting are new.
"""
from __future__ import annotations

from typing import Dict, Optional

import torch
from torch import Tensor

from oracle import cesm_oracle as O


def weighted_diffusion_loss(sd: O.StateDict, cfg: O.OracleConfig, buf: Dict[str, Tensor], x0: Tensor, cond: Tensor,
                            t: Tensor, noise: Tensor, prediction_type: str = "v", weights: Optional[Tensor] = None,
                            pre: str = "net.") -> Tensor:
    """The loss of `Diffusion(prediction_type=...).loss(x0, cond, t, noise, weights)`: target eps = noise or
    v = sqrt(ab) noise - sqrt(1 - ab) x0, and the batch mean of weights[t_b] * mean_pixels (pred - target)^2 (uniform
    when weights is None)."""
    x_t = O.q_sample(buf, x0, t, noise)
    pred = O.unet_forward(sd, cfg, x_t, cond, t, pre)
    if prediction_type == "v":
        a = buf["sqrt_alphas_cumprod"][t].view(-1, 1, 1, 1)
        s = buf["sqrt_one_minus_alphas_cumprod"][t].view(-1, 1, 1, 1)
        target = a * noise - s * x0
    elif prediction_type == "eps":
        target = noise
    else:
        raise ValueError(f"unknown prediction_type {prediction_type!r}")
    per_sample = ((pred - target) ** 2).flatten(1).mean(dim=1)
    w = torch.ones_like(per_sample) if weights is None else weights[t].to(per_sample.dtype)
    return (w * per_sample).mean()
