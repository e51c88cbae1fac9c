"""fp32 CPU reference of the DPM-Solver++(2M) sampler (Lu et al., "DPM-Solver++: Fast Solver for Guided Sampling of
Diffusion Probabilistic Models"), the checker for `model.dpm_schedule`, `kernels.dpm_step`, `Diffusion.dpm_sample`
and `SampleEngine(dpm_steps=N)`.

It is written in the paper's multistep form directly from alpha_bar (the `alphas_cumprod` buffer of
`oracle.cesm_oracle.diffusion_buffers`): lambda = log(alpha / sigma), h, r and the corrected data prediction D.  It
recomputes the trailing timestep spacing itself, so it shares no code or coefficient table with the product.  The
UNet is the existing oracle's `unet_forward`.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Tuple

import torch
from torch import Tensor

from oracle import cesm_oracle as O


def dpm_timesteps(T: int, steps: int) -> List[int]:
    """Trailing spacing: tau_i = floor(T (N - i) / N) - 1, i = 0..N-1."""
    return [T * (steps - i) // steps - 1 for i in range(steps)]


def dpm_update(buf: Dict[str, Tensor], x_t: Tensor, eps: Tensor, t: Tensor, steps: int,
               x0_prev: Optional[Tensor]) -> Tuple[Tensor, Tensor]:
    """One 2M step of an N = `steps` chain given the predicted eps, per sample at its own timestep t (one of the
    chain's taus).  Returns (x_p, x0).  With s = t, p the next tau (alpha_bar_p = 1 after the last) and q the previous:
        x0 = (x_t - sigma_s eps) / alpha_s,   h = lambda_p - lambda_s
        first step:   D = x0
        middle steps: r = (lambda_s - lambda_q) / h,  D = (1 + 1/(2r)) x0 - 1/(2r) x0_prev
        x_p = (sigma_p / sigma_s) x_t - alpha_p (exp(-h) - 1) D,   and x_p = x0 at the last step.
    `x0_prev` (the previous step's x0) is used only by middle steps and may be None when there are none."""
    T = buf["alphas_cumprod"].shape[0]
    taus = dpm_timesteps(T, steps)
    ac = buf["alphas_cumprod"].to(x_t.dtype)
    one = torch.ones((), dtype=x_t.dtype)
    shape = (-1,) + (1,) * (x_t.ndim - 1)

    def lam(a):
        return torch.log(torch.sqrt(a) / torch.sqrt(1 - a))

    pos = [taus.index(int(s)) for s in t.tolist()]
    a_s = ac[t].view(shape)
    x0 = (x_t - torch.sqrt(1 - a_s) * eps) / torch.sqrt(a_s)
    out = torch.empty_like(x_t)
    for b, i in enumerate(pos):
        if i + 1 == steps:
            out[b] = x0[b]
            continue
        a_b, a_p = a_s[b], ac[taus[i + 1]]
        h = lam(a_p) - lam(a_b)
        if i == 0:
            D = x0[b]
        else:
            r = (lam(a_b) - lam(ac[taus[i - 1]])) / h
            D = (1 + 1 / (2 * r)) * x0[b] - 1 / (2 * r) * x0_prev[b]
        out[b] = torch.sqrt(1 - a_p) / torch.sqrt(1 - a_b) * x_t[b] - torch.sqrt(a_p) * (torch.exp(-h) - one) * D
    return out, x0


def dpm_step(sd: O.StateDict, cfg: O.OracleConfig, buf: Dict[str, Tensor], x_t: Tensor, cond: Tensor, t: Tensor,
             steps: int, x0_prev: Optional[Tensor], pre: str = "net.") -> Tuple[Tensor, Tensor]:
    """One 2M reverse step with the oracle UNet's eps; returns (x_p, x0)."""
    eps = O.unet_forward(sd, cfg, x_t, cond, t, pre)
    return dpm_update(buf, x_t, eps, t, steps, x0_prev)


@torch.no_grad()
def dpm_sample(sd: O.StateDict, cfg: O.OracleConfig, buf: Dict[str, Tensor], cond: Tensor, x_T: Tensor, steps: int,
               pre: str = "net.") -> Tensor:
    """The whole 2M chain of `steps` UNet calls from x_T."""
    T = buf["alphas_cumprod"].shape[0]
    B = x_T.shape[0]
    x, x0 = x_T, None
    for tt in dpm_timesteps(T, steps):
        x, x0 = dpm_step(sd, cfg, buf, x, cond, torch.full((B,), tt, dtype=torch.long), steps, x0, pre)
    return x
