"""2-D facing wrapper and DDPM maths of the CESM emulator (mirror of the reference's model.py).

`UNet` and `Diffusion` keep the reference's constructor signatures, attribute names
(`UNet.net`, `Diffusion.model`, `.T`, the eight schedule buffers) and call surface
(`forward(x_t, cond, t)`, `loss`, `q_sample`, `p_sample`, `sample`), so train.py / inference.py
style drivers and reference checkpoints work unchanged.  All tensor work runs in the sm_100a
kernels of libcesm_b200.so; there is no CPU path.
"""
from __future__ import annotations

import math
import numbers

import torch
from torch import nn

from . import kernels as K
from . import ops
from .video_net import UNetModel3D


class UNet(nn.Module):
    """model.py:37-134.  `in_channels`, `num_res_blocks`, `time_dim` and `dropout` are accepted
    and ignored exactly as in the reference (model.py:46-52)."""

    def __init__(self, in_channels: int = 2, out_channels: int = 1, base_ch: int = 64, ch_mults=(1, 2, 4),
                 num_res_blocks: int = 2, time_dim: int = 256, groups: int = 8, dropout: float = 0.0,
                 attn_heads: int = 8, attn_dim_head: int = 32, use_sparse_linear_attn: bool = True,
                 use_mid_attn: bool = False, init_kernel_size: int = 7, use_checkpoint: bool = False,
                 use_temp_attn: bool = True, day_cond: bool = False, year_cond: bool = False,
                 cond_map: bool = True):
        super().__init__()
        self.net = UNetModel3D(
            n_vars=out_channels, model_dim=base_ch, dim_mults=tuple(ch_mults), attn_heads=attn_heads,
            attn_dim_head=attn_dim_head, use_sparse_linear_attn=use_sparse_linear_attn, use_mid_attn=use_mid_attn,
            init_kernel_size=init_kernel_size, resnet_groups=groups, use_checkpoint=use_checkpoint,
            use_temp_attn=use_temp_attn, day_cond=day_cond, year_cond=year_cond, cond_map=cond_map)

    def forward(self, x_t, cond, t):
        """x_t: [B,1,H,W] or [B,1,F,H,W]; cond: [B,1,H,W] or [B,1,F,H,W]; t: [B] -> [B,1,H,W].

        The reference expands the single-frame side to F frames, runs the 3-D net on all frames
        and keeps frame F//2 (model.py:110-130).  Here the broadcast happens inside the input-conv
        kernel and the 1x1x1 output conv is evaluated for the centre frame only."""
        if x_t.ndim == 4:
            x_t = x_t.unsqueeze(2)
        elif x_t.ndim != 5:
            raise ValueError(f"x_t must be 4D or 5D, got {x_t.ndim}D")
        if cond is None:
            raise ValueError("cond must be provided")
        if cond.ndim == 4:
            cond = cond.unsqueeze(2)
        elif cond.ndim != 5:
            raise ValueError(f"cond must be 4D or 5D, got {cond.ndim}D")
        Fx, Fc = x_t.shape[2], cond.shape[2]
        if Fx != Fc and not (Fx == 1 or Fc == 1):
            raise ValueError(f"Frame mismatch: x_t F={Fx}, cond F={Fc}")
        F = max(Fx, Fc)
        out = self.net.forward_frames(x_t, t, cond, frames=[F // 2])
        return out.squeeze(2)


PREDICTION_TYPES = ("eps", "v")


def check_prediction_type(prediction_type) -> str:
    """The network's output: "eps" (the noise, the reference's target) or "v" = sqrt(ab) eps - sqrt(1 - ab) x0
    (Salimans & Ho, "Progressive Distillation for Fast Sampling of Diffusion Models")."""
    if not isinstance(prediction_type, str) or prediction_type not in PREDICTION_TYPES:
        raise ValueError(f"prediction_type must be one of {PREDICTION_TYPES}, got {prediction_type!r}")
    return prediction_type


def ddim_schedule(alphas_cumprod: torch.Tensor, steps: int, eta: float = 0.0, prediction_type: str = "eps"):
    """Strided DDIM reverse chain (Song et al., "Denoising Diffusion Implicit Models") over the trained DDPM schedule.

    Timesteps use "trailing" spacing, tau_i = floor(T (N - i) / N) - 1 for i = 0..N-1: the chain starts at T - 1,
    where x ~ N(0, I) is valid, its last step goes to alpha_bar = 1, and N = T gives T-1, ..., 0.  One step from
    tau to p (the next tau, alpha_bar_p = 1 after the last one) is, in the x0-prediction form rewritten as three
    coefficients (no x0 clipping, as in p_sample):
        sigma = eta sqrt((1 - ab_p) / (1 - ab_tau)) sqrt(1 - ab_tau / ab_p)
        x_p = A x + B eps + S z,  A = sqrt(ab_p / ab_tau),  S = sigma,
        B = sqrt(max(0, 1 - ab_p - sigma^2)) - sqrt(ab_p) sqrt(1 - ab_tau) / sqrt(ab_tau)
    eta = 0 is deterministic; eta = 1 with N = T is the DDPM posterior step.  The coefficients are computed in float64
    from the fp32 alphas_cumprod (1 - ab cancels at small tau in fp32) and stored as fp32.

    For prediction_type "v" the network output is v and eps = sqrt(ab_tau) v + sqrt(1 - ab_tau) x, so the rows become
    (A + B sqrt(1 - ab_tau), B sqrt(ab_tau), S), written in the closed form
        A_v = sqrt(ab_p) sqrt(ab_tau) + c sqrt(1 - ab_tau),   B_v = c sqrt(ab_tau) - sqrt(ab_p) sqrt(1 - ab_tau),
    c = sqrt(max(0, 1 - ab_p - sigma^2)), which does not subtract two terms of size 1 / sqrt(ab_tau).

    Returns (taus: list of N ints, coef: fp32 [T, 3] rows (A, B, S), next_t: int64 [T]), both tables on the CPU.
    Rows off the schedule hold NaN coefficients and next_t = -1; next_t of the last step is -1."""
    T = int(alphas_cumprod.shape[0])
    if isinstance(steps, bool) or not isinstance(steps, numbers.Integral):
        raise ValueError(f"DDIM steps must be an integer, got {steps!r}")
    steps = int(steps)
    if not 1 <= steps <= T:
        raise ValueError(f"DDIM steps must be in [1, {T}], got {steps}")
    eta = float(eta)
    if not eta >= 0.0:  # also rejects NaN
        raise ValueError(f"DDIM eta must be >= 0, got {eta}")
    v = check_prediction_type(prediction_type) == "v"
    ac = alphas_cumprod.detach().to("cpu", torch.float64)
    taus = [T * (steps - i) // steps - 1 for i in range(steps)]
    coef = torch.full((T, 3), float("nan"), dtype=torch.float64)
    next_t = torch.full((T,), -1, dtype=torch.int64)
    one = torch.ones((), dtype=torch.float64)
    for i, tau in enumerate(taus):
        a_t = ac[tau]
        a_p = ac[taus[i + 1]] if i + 1 < steps else one
        sigma = eta * torch.sqrt((1 - a_p) / (1 - a_t)) * torch.sqrt(1 - a_t / a_p)
        c = torch.sqrt(torch.clamp(1 - a_p - sigma * sigma, min=0))
        if v:
            coef[tau, 0] = torch.sqrt(a_p) * torch.sqrt(a_t) + c * torch.sqrt(1 - a_t)
            coef[tau, 1] = c * torch.sqrt(a_t) - torch.sqrt(a_p) * torch.sqrt(1 - a_t)
        else:
            coef[tau, 0] = torch.sqrt(a_p / a_t)
            coef[tau, 1] = c - torch.sqrt(a_p) * torch.sqrt(1 - a_t) / torch.sqrt(a_t)
        coef[tau, 2] = sigma
        if i + 1 < steps:
            next_t[tau] = taus[i + 1]
    return taus, coef.float(), next_t


def dpm_schedule(alphas_cumprod: torch.Tensor, steps: int, prediction_type: str = "eps"):
    """DPM-Solver++(2M) reverse chain (Lu et al., "DPM-Solver++: Fast Solver for Guided Sampling of Diffusion
    Probabilistic Models"), multistep second order in the data-prediction form, over the trained DDPM schedule.

    The timesteps and the next_t chain are ddim_schedule's (trailing spacing), so the two samplers compare at equal N.
    With alpha = sqrt(ab), sigma = sqrt(1 - ab), lambda = log(alpha / sigma), step i goes from s = tau_i to p =
    tau_{i+1} (ab_p = 1 after the last step), h_i = lambda_p - lambda_s and phi = -alpha_p expm1(-h_i).  The row of
    tau_i holds (P, Q, R, K0, K1) for
        x0 = P x + Q eps,   x_p = R x + K0 x0 + K1 x0_prev,   P = 1 / alpha_s,  Q = -sigma_s / alpha_s,
        R = sigma_p / sigma_s,   and with r = h_{i-1} / h_i:  K0 = phi (1 + 1 / (2r)),  K1 = -phi / (2r),
    where x0_prev is the previous step's x0.  The first and the last step are first order (the usual lower order at
    the ends): the first has K0 = phi, K1 = 0; the last lands on ab = 1 with R = 0, K0 = 1, K1 = 0, i.e. x_0 is the
    x0 prediction.  Both are DDIM eta = 0 steps, so N <= 2 is exactly the DDIM eta = 0 chain.  The chain is
    deterministic after x_T.  The coefficients are computed in float64 from the fp32 alphas_cumprod and stored as fp32.
    For prediction_type "v" the network output is v and x0 = sqrt(ab_s) x - sqrt(1 - ab_s) v: P = alpha_s, Q = -sigma_s
    (written directly; P + Q sqrt(1 - ab_s) of the eps rows would subtract two terms of size 1 / alpha_s).

    Returns (taus: list of N ints, coef: fp32 [T, 5] rows (P, Q, R, K0, K1), next_t: int64 [T]), both tables on the
    CPU.  Rows off the schedule hold NaN coefficients and next_t = -1; next_t of the last step is -1."""
    T = int(alphas_cumprod.shape[0])
    if isinstance(steps, bool) or not isinstance(steps, numbers.Integral):
        raise ValueError(f"DPM-Solver steps must be an integer, got {steps!r}")
    steps = int(steps)
    if not 1 <= steps <= T:
        raise ValueError(f"DPM-Solver steps must be in [1, {T}], got {steps}")
    v = check_prediction_type(prediction_type) == "v"
    taus, _, next_t = ddim_schedule(alphas_cumprod, steps)
    ac = alphas_cumprod.detach().to("cpu", torch.float64).tolist()
    lam = lambda a: 0.5 * math.log(a / (1.0 - a))  # noqa: E731  log(alpha / sigma)
    coef = torch.full((T, 5), float("nan"), dtype=torch.float64)
    h_prev = None
    for i, s in enumerate(taus):
        a_s = ac[s]
        if v:
            P, Q = math.sqrt(a_s), -math.sqrt(1.0 - a_s)
        else:
            P, Q = 1.0 / math.sqrt(a_s), -math.sqrt(1.0 - a_s) / math.sqrt(a_s)
        if i + 1 == steps:
            coef[s] = torch.tensor([P, Q, 0.0, 1.0, 0.0], dtype=torch.float64)
            break
        a_p = ac[taus[i + 1]]
        h = lam(a_p) - lam(a_s)
        phi = -math.sqrt(a_p) * math.expm1(-h)
        R = math.sqrt(1.0 - a_p) / math.sqrt(1.0 - a_s)
        if h_prev is None:
            K0, K1 = phi, 0.0
        else:
            r = h_prev / h
            K0, K1 = phi * (1.0 + 0.5 / r), -phi * 0.5 / r
        coef[s] = torch.tensor([P, Q, R, K0, K1], dtype=torch.float64)
        h_prev = h
    return taus, coef.float(), next_t


class Diffusion(nn.Module):
    """model.py:141-208.

    `prediction_type` (keyword only, an addition beyond the reference) names what the network predicts: "eps", the
    reference's noise target, or "v" = sqrt(ab) eps - sqrt(1 - ab) x0, from which x0 = sqrt(ab) x_t - sqrt(1 - ab) v
    carries no 1 / sqrt(ab) amplification (157 at t = 999 on the linear schedule).  A v-model samples with every chain
    of the eps-model through coefficient tables that fold the conversion in (ddim_schedule, dpm_schedule).  Its
    tables are non-persistent buffers: state_dict() and checkpoints are the same for both targets."""

    def __init__(self, model, img_channels=1, timesteps=1000, beta_schedule="linear", *, prediction_type="eps"):
        super().__init__()
        self.prediction_type = check_prediction_type(prediction_type)
        self.model = model
        self.img_channels = img_channels
        self.T = timesteps
        if beta_schedule == "linear":
            beta_start, beta_end = 1e-4, 2e-2
            betas = torch.linspace(beta_start, beta_end, timesteps)
        else:
            raise ValueError("Only 'linear' beta_schedule implemented")
        alphas = 1.0 - betas
        alphas_cumprod = torch.cumprod(alphas, dim=0)
        alphas_cumprod_prev = torch.cat([torch.tensor([1.0]), alphas_cumprod[:-1]], dim=0)
        self.register_buffer("betas", betas)
        self.register_buffer("alphas", alphas)
        self.register_buffer("alphas_cumprod", alphas_cumprod)
        self.register_buffer("alphas_cumprod_prev", alphas_cumprod_prev)
        self.register_buffer("sqrt_alphas_cumprod", torch.sqrt(alphas_cumprod))
        self.register_buffer("sqrt_one_minus_alphas_cumprod", torch.sqrt(1.0 - alphas_cumprod))
        self.register_buffer("sqrt_recip_alphas", torch.sqrt(1.0 / alphas))
        self.register_buffer("posterior_variance", betas * (1.0 - alphas_cumprod_prev) / (1.0 - alphas_cumprod))
        v_coef = ddpm_coef = None
        if self.prediction_type == "v":
            ac = alphas_cumprod.double()
            # target = c_n noise + c_x x0 (DiffusionLossFn): v = sqrt(ab) eps - sqrt(1 - ab) x0
            v_coef = torch.stack([ac.sqrt(), -(1 - ac).sqrt()], dim=1).float()
            # the DDPM chain of a v-model: the folded DDIM table at N = T, eta = 1, which is the posterior step
            ddpm_coef = ddim_schedule(alphas_cumprod, timesteps, 1.0, "v")[1]
        self.register_buffer("target_coef", v_coef, persistent=False)
        self.register_buffer("ddpm_coef", ddpm_coef, persistent=False)

    def min_snr_weights(self, gamma) -> torch.Tensor:
        """Min-SNR-gamma loss weights (Hang et al., "Efficient Diffusion Training via Min-SNR Weighting Strategy") for
        this Diffusion's target, SNR = ab / (1 - ab): min(SNR, gamma) / SNR for eps, min(SNR, gamma) / (SNR + 1) for v.
        Both weight the x0 error by min(SNR, gamma).  gamma is a finite real number > 0 (an int is accepted, a bool
        is not).  Computed in float64 -> fp32 [T] on the schedule's device."""
        if isinstance(gamma, bool) or not isinstance(gamma, numbers.Real):
            raise ValueError(f"min_snr_gamma must be a real number > 0, got {gamma!r}")
        gamma = float(gamma)
        if not (math.isfinite(gamma) and gamma > 0):
            raise ValueError(f"min_snr_gamma must be finite and > 0, got {gamma}")
        ac = self.alphas_cumprod.double()
        snr = ac / (1 - ac)
        w = snr.clamp(max=gamma) / (snr + 1 if self.prediction_type == "v" else snr)
        return w.float()

    # -- sampling ------------------------------------------------------------------------------
    def p_sample(self, x_t, cond, t, noise=None):
        """model.py:168-183.  One reverse step.  posterior_variance[0] == 0, so the reference's
        `(t == 0).all()` branch (a host sync per step) is the same arithmetic as always adding
        sqrt(var_t) * z; the fused kernel does that without the sync.  `noise` may be supplied
        for deterministic parity tests."""
        with torch.no_grad():
            eps_theta = self.model(x_t, cond, t)
            z = torch.randn_like(x_t) if noise is None else noise
            if self.prediction_type == "v":  # eps_theta is v: the posterior step through the folded table
                return K.ddim_step(x_t.float().contiguous(), eps_theta, z.float().contiguous(), t.contiguous(),
                                   self.ddpm_coef, self.T)
            return K.p_sample(x_t.float().contiguous(), eps_theta, z.float().contiguous(), t.contiguous(),
                              self.betas, self.sqrt_one_minus_alphas_cumprod, self.sqrt_recip_alphas,
                              self.posterior_variance)

    def _x_T(self, shape, device, seed, field_ids):
        """Initial noise: torch's CUDA generator without a seed; with one, the counter-based draw of each field id
        (kernels.field_normal), which is what SampleEngine(seed=...) starts from too.  -> (x_T, ids or None)."""
        if seed is None:
            if field_ids is not None:
                raise ValueError("field_ids needs a seed (they select counter-based noise)")
            return torch.randn(shape, device=device), None
        K.split_seed(seed)
        ids = K.field_id_vector(field_ids, shape[0], device)
        return K.field_normal(seed, ids, K.X_T_DRAW, shape), ids

    def sample(self, cond, shape, device, *, seed=None, field_ids=None):
        """model.py:186-194.  With `seed` (an int in [0, 2^64)) every field's noise is drawn from (seed, its id in
        `field_ids`, default arange(B)) instead of torch's generator, so a field does not depend on its row or batch."""
        with torch.no_grad():
            B = shape[0]
            x, ids = self._x_T(shape, device, seed, field_ids)
            for tt in reversed(range(self.T)):
                t_tensor = torch.full((B,), tt, device=device, dtype=torch.long)
                if ids is None:
                    x = self.p_sample(x, cond, t_tensor)
                    continue
                eps_theta = self.model(x, cond, t_tensor)
                if self.prediction_type == "v":
                    x = K.ddim_step_seeded(x.float().contiguous(), eps_theta, seed, ids, t_tensor, self.ddpm_coef,
                                           self.T)
                    continue
                x = K.p_sample_seeded(x.float().contiguous(), eps_theta, seed, ids, t_tensor, self.betas,
                                      self.sqrt_one_minus_alphas_cumprod, self.sqrt_recip_alphas,
                                      self.posterior_variance)
            return x

    def ddim_sample(self, cond, shape, device, steps=50, eta=0.0, *, seed=None, field_ids=None):
        """Strided DDIM chain of `steps` UNet calls (ddim_schedule), eager; an addition beyond the reference.
        Fewer steps trade fidelity for speed; eta = 0 draws no noise after x_T.  `seed` / `field_ids` as in `sample`."""
        taus, coef, _ = ddim_schedule(self.alphas_cumprod, steps, eta, self.prediction_type)
        coef = coef.to(device)
        with torch.no_grad():
            B = shape[0]
            x, ids = self._x_T(shape, device, seed, field_ids)
            for tt in taus:
                t_tensor = torch.full((B,), tt, device=device, dtype=torch.long)
                eps_theta = self.model(x, cond, t_tensor)
                if ids is not None and eta > 0:
                    x = K.ddim_step_seeded(x, eps_theta, seed, ids, t_tensor, coef, self.T)
                    continue
                z = torch.randn_like(x) if eta > 0 else None
                x = K.ddim_step(x, eps_theta, z, t_tensor, coef, self.T)
            return x

    def dpm_sample(self, cond, shape, device, steps=20, *, seed=None, field_ids=None):
        """DPM-Solver++(2M) chain of `steps` UNet calls (dpm_schedule), eager; an addition beyond the reference.
        Deterministic after x_T.  `hist` carries the previous step's x0 prediction; the first step does not read it.
        `seed` / `field_ids` as in `sample` (only x_T is random)."""
        taus, coef, _ = dpm_schedule(self.alphas_cumprod, steps, self.prediction_type)
        coef = coef.to(device)
        with torch.no_grad():
            B = shape[0]
            x, _ = self._x_T(shape, device, seed, field_ids)
            hist = torch.empty_like(x)
            for tt in taus:
                t_tensor = torch.full((B,), tt, device=device, dtype=torch.long)
                eps_theta = self.model(x, cond, t_tensor)
                x = K.dpm_step(x, eps_theta, hist, t_tensor, coef, self.T)
            return x

    # -- training ------------------------------------------------------------------------------
    def q_sample(self, x0, t, noise=None):
        """model.py:196-201.  Differentiable in x0 and noise (ops.QSampleFn)."""
        if noise is None:
            noise = torch.randn_like(x0)
        x_t = ops.QSampleFn.apply(x0.float().contiguous(), noise.float().contiguous(), t.contiguous(),
                                  self.sqrt_alphas_cumprod, self.sqrt_one_minus_alphas_cumprod)
        return x_t, noise

    def loss(self, x0, cond, t=None, noise=None, weights=None):
        """model.py:203-208.  `t` / `noise` default to the reference's draws (randint, then
        randn_like); passing them makes parity tests deterministic.  `weights` (fp32 [T], e.g. `min_snr_weights`)
        weights each sample's squared error by weights[t]; the loss is sum_b weights[t_b] sum_pixels err^2 / numel.
        With the eps target and no weights this is the reference's MSE (ops.MseLossFn); otherwise the fused
        objective (ops.DiffusionLossFn) computes the target and the weighting."""
        if weights is not None and (not torch.is_tensor(weights) or tuple(weights.shape) != (self.T,)):
            raise ValueError(f"weights must be a tensor of shape ({self.T},)")
        B = x0.size(0)
        if t is None:
            t = torch.randint(0, self.T, (B,), device=x0.device).long()
        x_t, noise = self.q_sample(x0, t, noise)
        eps_pred = self.model(x_t, cond, t)
        if self.prediction_type == "eps" and weights is None:
            return ops.MseLossFn.apply(eps_pred, noise.float())
        w = None if weights is None else weights.float().contiguous()
        return ops.DiffusionLossFn.apply(eps_pred, x0.float(), noise.float(), t.contiguous(), self.target_coef, w)
