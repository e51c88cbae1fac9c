"""float64 reference of classifier-free guidance (Ho & Salimans, "Classifier-Free Diffusion Guidance"), the checker for
the guided update kernels (`kernels.p_sample / ddim_step / dpm_step / *_seeded` with `guidance`), the guided chains of
`Diffusion` and `SampleEngine(guidance=w)`, and the training loss under condition dropout.

Guidance combines the network's two predictions at the same (x, t) -- with the field's condition and with the null
(all-zero) condition -- as (1 + w) out_cond - w out_null, in the network's own output space.  The chains below convert
that output to eps in float64 and reuse the independent DDIM / DPM-Solver++(2M) references (ddim_oracle.py,
dpm_oracle.py) and the DDPM posterior step written out here, so they share no code or table with the product.  A
network is any callable net(x, cond, t) -> output; `oracle_net` wraps the existing oracle's UNet.
"""
from __future__ import annotations

from typing import Callable, Dict, List, Optional

import torch
from torch import Tensor

import ddim_oracle as DO
import dpm_oracle as PO
from objective_oracle import weighted_diffusion_loss
from oracle import cesm_oracle as O

Net = Callable[[Tensor, Tensor, Tensor], Tensor]


def combine(out_cond: Tensor, out_null: Tensor, w: float) -> Tensor:
    """The guided output (1 + w) out_cond - w out_null."""
    return (1 + w) * out_cond - w * out_null


def guided_output(net: Net, x: Tensor, cond: Tensor, t: Tensor, w: float) -> Tensor:
    """The network's guided output at (x, t); w = 0 is net(x, cond, t) itself (no null-condition call)."""
    c = net(x, cond, t)
    return c if w == 0 else combine(c, net(x, torch.zeros_like(cond), t), w)


def _col(v: Tensor, x: Tensor) -> Tensor:
    return v.to(x.dtype).view((-1,) + (1,) * (x.ndim - 1))


def to_eps(buf: Dict[str, Tensor], x: Tensor, out: Tensor, t: Tensor, prediction_type: str) -> Tensor:
    """The eps an output means at (x, t): itself for "eps", sqrt(ab) v + sqrt(1 - ab) x for "v"."""
    if prediction_type == "eps":
        return out
    ac = buf["alphas_cumprod"].double()[t]
    return _col(ac.sqrt(), x) * out + _col((1 - ac).sqrt(), x) * x


def ddpm_update(buf: Dict[str, Tensor], x: Tensor, eps: Tensor, t: Tensor, z: Tensor) -> Tensor:
    """The DDPM posterior step (model.py:168-183): 1/sqrt(alpha) (x - beta / sqrt(1 - ab) eps) + sqrt(var) z."""
    d = {k: v.double()[t] for k, v in buf.items()}
    mean = _col(1 / d["alphas"].sqrt(), x) * (x - _col(d["betas"] / (1 - d["alphas_cumprod"]).sqrt(), x) * eps)
    return mean + _col(d["posterior_variance"].sqrt(), x) * z


def oracle_net(sd: O.StateDict, cfg: O.OracleConfig, pre: str = "net.") -> Net:
    return lambda x, cond, t: O.unet_forward(sd, cfg, x, cond, t, pre)


@torch.no_grad()
def guided_ddpm_sample(net: Net, buf: Dict[str, Tensor], cond: Tensor, x_T: Tensor, w: float, noises: List[Tensor],
                       prediction_type: str = "eps") -> Tensor:
    """len(noises) DDPM steps from t = T - 1 down; noises[i] is the z of step i."""
    T = buf["alphas_cumprod"].shape[0]
    x = x_T.double()
    for i, z in enumerate(noises):
        t = torch.full((x.shape[0],), T - 1 - i, dtype=torch.long)
        out = guided_output(net, x.float(), cond, t, w).double()
        x = ddpm_update(buf, x, to_eps(buf, x, out, t, prediction_type), t, z.double())
    return x


@torch.no_grad()
def guided_ddim_sample(net: Net, buf: Dict[str, Tensor], cond: Tensor, x_T: Tensor, steps: int, eta: float, w: float,
                       noises: Optional[List[Tensor]] = None, prediction_type: str = "eps") -> Tensor:
    """The strided DDIM chain of ddim_oracle with the guided output; noises[i] is the z of step i when eta > 0."""
    buf64 = {k: v.double() for k, v in buf.items()}
    T = buf["alphas_cumprod"].shape[0]
    taus = DO.ddim_timesteps(T, steps)
    x = x_T.double()
    for i, tt in enumerate(taus):
        t = torch.full((x.shape[0],), tt, dtype=torch.long)
        tp = torch.full((x.shape[0],), taus[i + 1] if i + 1 < steps else -1, dtype=torch.long)
        out = guided_output(net, x.float(), cond, t, w).double()
        x = DO.ddim_update(buf64, x, to_eps(buf, x, out, t, prediction_type), t, tp, eta,
                           noises[i].double() if eta > 0 else None)
    return x


@torch.no_grad()
def guided_dpm_sample(net: Net, buf: Dict[str, Tensor], cond: Tensor, x_T: Tensor, steps: int, w: float,
                      prediction_type: str = "eps") -> Tensor:
    """The DPM-Solver++(2M) chain of dpm_oracle with the guided output."""
    buf64 = {k: v.double() for k, v in buf.items()}
    T = buf["alphas_cumprod"].shape[0]
    x, x0 = x_T.double(), None
    for tt in PO.dpm_timesteps(T, steps):
        t = torch.full((x.shape[0],), tt, dtype=torch.long)
        out = guided_output(net, x.float(), cond, t, w).double()
        x, x0 = PO.dpm_update(buf64, x, to_eps(buf, x, out, t, prediction_type), t, steps, x0)
    return x


def masked_condition(cond: Tensor, keep: Tensor) -> Tensor:
    """cond with the samples where keep == 0 replaced by the null (all-zero) condition."""
    return torch.where(_col(keep, cond) != 0, cond, torch.zeros_like(cond))


def masked_diffusion_loss(sd: O.StateDict, cfg: O.OracleConfig, buf: Dict[str, Tensor], x0: Tensor, cond: Tensor,
                          t: Tensor, noise: Tensor, keep: Tensor, prediction_type: str = "eps",
                          weights: Optional[Tensor] = None, pre: str = "net.") -> Tensor:
    """The loss of `Diffusion.loss(x0, cond, t, noise, weights, keep=keep)`: the objective on masked_condition."""
    return weighted_diffusion_loss(sd, cfg, buf, x0, masked_condition(cond, keep), t, noise, prediction_type, weights,
                                   pre)
