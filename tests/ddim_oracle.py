"""fp32 CPU reference of the strided DDIM sampler (Song et al., "Denoising Diffusion Implicit Models"), the checker
for `model.ddim_schedule`, `kernels.ddim_step`, `Diffusion.ddim_sample` and `SampleEngine(ddim_steps=N)`.

It is written in the x0-prediction form directly from alpha_bar (the `alphas_cumprod` buffer of
`oracle.cesm_oracle.diffusion_buffers`) and recomputes the trailing timestep spacing itself, so it shares no code
or coefficient table with the product.  The UNet is the existing oracle's `unet_forward`.
"""
from __future__ import annotations

from typing import Dict, List, Optional

import torch
from torch import Tensor

from oracle import cesm_oracle as O


def ddim_timesteps(T: int, steps: int) -> List[int]:
    """Trailing spacing: tau_i = floor(T (N - i) / N) - 1, i = 0..N-1."""
    return [T * (steps - i) // steps - 1 for i in range(steps)]


def ddim_update(buf: Dict[str, Tensor], x_t: Tensor, eps: Tensor, t: Tensor, t_prev: Tensor, eta: float,
                noise: Optional[Tensor]) -> Tensor:
    """One DDIM step given the predicted eps: t -> t_prev per sample, t_prev = -1 meaning alpha_bar = 1.
        x0 = (x_t - sqrt(1 - ab_t) eps) / sqrt(ab_t)
        sigma = eta sqrt((1 - ab_p) / (1 - ab_t)) sqrt(1 - ab_t / ab_p)
        x_p = sqrt(ab_p) x0 + sqrt(1 - ab_p - sigma^2) eps + sigma z
    No x0 clipping.  `noise` may be None when eta == 0."""
    ac = buf["alphas_cumprod"].to(x_t.dtype)
    shape = (-1,) + (1,) * (x_t.ndim - 1)
    a_t = ac[t].view(shape)
    a_p = torch.where(t_prev >= 0, ac[t_prev.clamp(min=0)], torch.ones((), dtype=x_t.dtype)).view(shape)
    x0 = (x_t - torch.sqrt(1 - a_t) * eps) / torch.sqrt(a_t)
    sigma = eta * torch.sqrt((1 - a_p) / (1 - a_t)) * torch.sqrt(1 - a_t / a_p)
    out = torch.sqrt(a_p) * x0 + torch.sqrt(torch.clamp(1 - a_p - sigma * sigma, min=0)) * eps
    if eta > 0:
        out = out + sigma * noise
    return out


def ddim_step(sd: O.StateDict, cfg: O.OracleConfig, buf: Dict[str, Tensor], x_t: Tensor, cond: Tensor, t: Tensor,
              t_prev: Tensor, eta: float, noise: Optional[Tensor], pre: str = "net.") -> Tensor:
    """One DDIM reverse step with the oracle UNet's eps."""
    eps = O.unet_forward(sd, cfg, x_t, cond, t, pre)
    return ddim_update(buf, x_t, eps, t, t_prev, eta, noise)


@torch.no_grad()
def ddim_sample(sd: O.StateDict, cfg: O.OracleConfig, buf: Dict[str, Tensor], cond: Tensor, x_T: Tensor, steps: int,
                eta: float, noises: Optional[List[Tensor]] = None, pre: str = "net.") -> Tensor:
    """The whole strided chain from x_T; with eta > 0, `noises[i]` is the z of step i."""
    T = buf["alphas_cumprod"].shape[0]
    taus = ddim_timesteps(T, steps)
    B = x_T.shape[0]
    x = x_T
    for i, tt in enumerate(taus):
        t = torch.full((B,), tt, dtype=torch.long)
        tp = torch.full((B,), taus[i + 1] if i + 1 < steps else -1, dtype=torch.long)
        x = ddim_step(sd, cfg, buf, x, cond, t, tp, eta, noises[i] if eta > 0 else None, pre)
    return x
