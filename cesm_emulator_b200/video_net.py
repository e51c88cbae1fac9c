"""Space-time U-Net of the CESM emulator on the B200 kernel library.

Mirror of the reference's video_net.py: the same class names, constructor arguments, attribute
tree and state-dict keys (so `load_state_dict(strict=True)` works in both directions and
`torch.manual_seed(s)` followed by construction yields bit-identical initial weights), but every
forward/backward runs through the sm_100a kernels of libcesm_b200.so (see ops.py).  nn.Conv3d /
nn.Linear / nn.GroupNorm / nn.Embedding appear below only as PARAMETER HOLDERS with the
reference's initialisers; their aten forward is never called.

Internal activation layout: channels-last fp16 `[B*F, H, W, C]`.  Every module offers
  * `forward(x, ...)`     -- the reference's signature on [B, C, F, H, W] tensors (layout is
                             converted at this boundary), and
  * `forward_cl(x, B, F)` -- the same computation on the internal layout, which is what
                             `UNetModel3D` chains so that no permutes happen inside the network.
There is no CPU path: a CPU tensor raises (kernels._req_cuda).
"""
from __future__ import annotations

import math
from functools import partial
from typing import Optional

import torch
from torch import nn

from . import kernels as K
from . import ops
from .rotary_embedding import RotaryEmbedding


def exists(val):
    return val is not None


def default(val, d):
    if exists(val):
        return val
    return d() if callable(d) else d


def cast_to_tuple(val, n):
    if isinstance(val, tuple):
        return val
    if isinstance(val, list):
        return tuple(val)
    if isinstance(val, (int, bool)):
        return [val] * n
    return tuple(val)


def prob_mask_like(shape, prob, device):
    """video_net.py:44-50."""
    if prob == 1:
        return torch.ones(shape, device=device, dtype=torch.bool)
    if prob == 0:
        return torch.zeros(shape, device=device, dtype=torch.bool)
    return torch.zeros(shape, device=device).float().uniform_(0, 1) < prob


def checkpoint(fn, *args, enabled=False):
    """video_net.py:15-19.  Activation checkpointing is a 16 GB-V100 memory trick; on a 180 GB
    B200 the fused kernels keep what they need, so `enabled` is accepted and ignored."""
    return fn(*args)


class Identity(nn.Module):
    def __init__(self, *args, **kwargs):
        super().__init__()

    def forward(self, x, *args, **kwargs):
        return x

    def forward_cl(self, x, B, F, **kwargs):
        return x


class _ResampleMixin:
    """Gives a Conv3d / ConvTranspose3d (1,4,4)/(1,2,2)/(0,1,1) parameter holder (reference key
    names `weight`, `bias`) a forward on the B200 kernels."""

    fn = None

    def _pack_cache(self):
        c = self.__dict__.get("_cache")
        if c is None:
            c = self.__dict__["_cache"] = ops.PackCache()
        return c

    def forward_cl(self, x, B, F, **kwargs):
        return type(self).fn.apply(x, self.weight, self.bias, self._pack_cache())

    def forward(self, x):
        xc, B, F = ops.to_cl(x)
        return ops.from_cl(self.forward_cl(xc, B, F), B, F).to(x.dtype)


class _DownsampleConv(_ResampleMixin, nn.Conv3d):
    fn = ops.DownsampleFn


class _UpsampleConv(_ResampleMixin, nn.ConvTranspose3d):
    fn = ops.UpsampleFn


def Downsample(dim):
    """video_net.py:61-62."""
    return _DownsampleConv(dim, dim, (1, 4, 4), (1, 2, 2), (0, 1, 1))


def Upsample(dim):
    """video_net.py:65-66."""
    return _UpsampleConv(dim, dim, (1, 4, 4), (1, 2, 2), (0, 1, 1))


class Residual(nn.Module):
    """video_net.py:69-75.  The add is fused into the wrapped op's output-projection epilogue."""

    def __init__(self, fn):
        super().__init__()
        self.fn = fn

    def forward_cl(self, x, B, F, **kwargs):
        fused = _fused_attention_block(self, x, B, F, **kwargs)
        if fused is not None:
            return fused
        return self.fn.forward_cl(x, B, F, residual=x, **kwargs)

    def forward(self, x, *args, **kwargs):
        xc, B, F = ops.to_cl(x)
        return ops.from_cl(self.forward_cl(xc, B, F, **kwargs), B, F).to(x.dtype)


def _fused_attention_block(res: "Residual", x, B, F, pos_bias=None, focus_present_mask=None):
    """Residual(PreNorm(SpatialLinearAttention)), Residual(PreNorm(EinopsToAndFrom(Attention))) over frames
    with the default all-False focus mask, and the use_mid_attn block Residual(PreNorm(EinopsToAndFrom(Attention)))
    over pixels run as ONE autograd node (ops.*AttnBlockFn); anything else returns None and takes the generic
    op-by-op path."""
    pre = res.fn
    if not isinstance(pre, PreNorm):
        return None
    inner = pre.fn
    if isinstance(inner, SpatialLinearAttention):
        meta = inner.__dict__.get("_bmeta")
        if meta is None:
            meta = inner.__dict__["_bmeta"] = ops.BlockMeta(heads=inner.heads, dim_head=inner.dim_head,
                                                            eps=pre.norm.eps, cq=ops.PackCache(), co=ops.PackCache())
        return ops.SpatialAttnBlockFn.apply(x, pre.norm.gamma, inner.to_qkv.weight, inner.to_out.weight,
                                            inner.to_out.bias, meta)
    if (isinstance(inner, EinopsToAndFrom) and inner.to_einops == "b (h w) f c" and isinstance(inner.fn, Attention)
            and focus_present_mask is None and exists(inner.fn.rotary_emb)):
        att = inner.fn
        meta = att.__dict__.get("_bmeta")
        if meta is None:
            meta = att.__dict__["_bmeta"] = ops.BlockMeta(heads=att.heads, dim_head=att.dim_head, eps=pre.norm.eps,
                                                          cq=ops.PackCache(), co=ops.PackCache())
        cs, sn = att.rotary_emb.tables(F)
        if pos_bias is None:
            pos_bias = torch.zeros((att.heads, F, F), dtype=torch.float32, device=x.device)
        return ops.TemporalAttnBlockFn.apply(x, pre.norm.gamma, att.to_qkv.weight, att.to_out.weight, pos_bias, cs, sn,
                                             B, F, meta)
    if (isinstance(inner, EinopsToAndFrom) and inner.to_einops == "b f (h w) c" and isinstance(inner.fn, Attention)
            and focus_present_mask is None):
        att = inner.fn
        meta = att.__dict__.get("_bmeta")
        if meta is None:
            meta = att.__dict__["_bmeta"] = ops.BlockMeta(heads=att.heads, dim_head=att.dim_head, eps=pre.norm.eps,
                                                          cq=ops.PackCache(), co=ops.PackCache())
        return ops.MidAttnBlockFn.apply(x, pre.norm.gamma, att.to_qkv.weight, att.to_out.weight, meta)
    return None


class LayerNorm(nn.Module):
    """video_net.py:78-87: channel LayerNorm, biased variance, eps inside the sqrt, gain only."""

    def __init__(self, dim, eps=1e-5):
        super().__init__()
        self.eps = eps
        self.gamma = nn.Parameter(torch.ones(1, dim, 1, 1, 1))

    def forward_cl(self, x, B=None, F=None):
        return ops.LayerNormFn.apply(x, self.gamma, self.eps)

    def forward(self, x):
        xc, B, F = ops.to_cl(x)
        return ops.from_cl(self.forward_cl(xc), B, F).to(x.dtype)


class PreNorm(nn.Module):
    """video_net.py:90-98."""

    def __init__(self, dim, fn):
        super().__init__()
        self.fn = fn
        self.norm = LayerNorm(dim)

    def forward_cl(self, x, B, F, **kwargs):
        return self.fn.forward_cl(self.norm.forward_cl(x), B, F, **kwargs)

    def forward(self, x, **kwargs):
        xc, B, F = ops.to_cl(x)
        return ops.from_cl(self.forward_cl(xc, B, F, **kwargs), B, F).to(x.dtype)


class SinusoidalPosEmb(nn.Module):
    """video_net.py:101-113."""

    def __init__(self, dim):
        super().__init__()
        self.dim = dim

    def forward(self, x):
        return K.sinusoidal(x.to(torch.int64).contiguous(), self.dim)


class Block(nn.Module):
    """video_net.py:211-227: Conv3d(1,3,3) -> GroupNorm -> FiLM -> SiLU (+ fused residual)."""

    def __init__(self, dim, dim_out, groups=8):
        super().__init__()
        self.proj = nn.Conv3d(dim, dim_out, (1, 3, 3), padding=(0, 1, 1))
        self.norm = nn.GroupNorm(groups, dim_out)
        self.act = nn.SiLU()
        self._cache = ops.PackCache()

    def forward_cl(self, x, B, F, film=None, x1=None, residual=None):
        y = ops.ConvFn.apply(x, x1, self.proj.weight, self.proj.bias, None, 3, self._cache)
        return ops.GroupNormSiLUFn.apply(y, self.norm.weight, self.norm.bias, film, residual, B,
                                         self.norm.num_groups, self.norm.eps)

    def forward(self, x, scale_shift=None):
        xc, B, F = ops.to_cl(x)
        film = None
        if exists(scale_shift):
            scale, shift = scale_shift
            film = torch.cat((scale.reshape(B, -1), shift.reshape(B, -1)), dim=1).float().contiguous()
        return ops.from_cl(self.forward_cl(xc, B, F, film=film), B, F).to(x.dtype)


class ResnetBlock(nn.Module):
    """video_net.py:230-265."""

    def __init__(self, dim, dim_out, *, time_emb_dim=None, groups=8, use_checkpoint=False):
        super().__init__()
        self.use_checkpoint = use_checkpoint
        self.mlp = (nn.Sequential(nn.SiLU(), nn.Linear(time_emb_dim, dim_out * 2))
                    if exists(time_emb_dim) else None)
        self.block1 = Block(dim, dim_out, groups=groups)
        self.block2 = Block(dim_out, dim_out, groups=groups)
        self.res_conv = nn.Conv3d(dim, dim_out, 1) if dim != dim_out else nn.Identity()
        self._meta = ops.BlockMeta(G=groups, eps=self.block1.norm.eps, c1=ops.PackCache(), c2=ops.PackCache(),
                                   cres=ops.PackCache())

    def forward_cl(self, x, B, F, time_emb=None, x1=None, film=None):
        """x1: optional second channels-last source, concatenated after x (U-Net skip).
        `film`: this block's FiLM vector when the caller has already computed it (the network pass computes
        all of them in one launch, ops.FilmAllFn).  The whole block is one autograd node (ops.ResnetBlockFn)."""
        if exists(self.mlp) and film is None:
            assert exists(time_emb), "time emb must be passed in"
            film = ops.SmallLinearFn.apply(time_emb, self.mlp[1].weight, self.mlp[1].bias, True)
        if isinstance(self.res_conv, nn.Identity):
            assert x1 is None
            wres = bres = None
        else:
            wres, bres = self.res_conv.weight, self.res_conv.bias
        b1, b2 = self.block1, self.block2
        return ops.ResnetBlockFn.apply(x, x1, film, b1.proj.weight, b1.proj.bias, b1.norm.weight, b1.norm.bias,
                                       b2.proj.weight, b2.proj.bias, b2.norm.weight, b2.norm.bias, wres, bres, B,
                                       self._meta)

    def forward(self, x, time_emb=None):
        xc, B, F = ops.to_cl(x)
        te = None if time_emb is None else time_emb.float().contiguous()
        return ops.from_cl(self.forward_cl(xc, B, F, time_emb=te), B, F).to(x.dtype)


class RelativePositionBias(nn.Module):
    """video_net.py:268-310.  The bucket table depends only on the frame count, so it is built on
    the host once per n; the Embedding gather is a [n, n] index into a [32, heads] table."""

    def __init__(self, heads=8, num_buckets=32, max_distance=128):
        super().__init__()
        self.num_buckets = num_buckets
        self.max_distance = max_distance
        self.relative_attention_bias = nn.Embedding(num_buckets, heads)
        self._tables = {}

    @staticmethod
    def _relative_position_bucket(relative_position, num_buckets=32, max_distance=128):
        n = -relative_position
        num_buckets //= 2
        ret = (n < 0).long() * num_buckets
        n = torch.abs(n)
        max_exact = num_buckets // 2
        is_small = n < max_exact
        val_if_large = max_exact + (torch.log(n.float() / max_exact) / math.log(max_distance / max_exact)
                                    * (num_buckets - max_exact)).long()
        val_if_large = torch.min(val_if_large, torch.full_like(val_if_large, num_buckets - 1))
        return ret + torch.where(is_small, n, val_if_large)

    def bucket_table(self, n, device):
        key = (n, str(device))
        t = self._tables.get(key)
        if t is None:
            pos = torch.arange(n, dtype=torch.long)
            rel = pos[None, :] - pos[:, None]
            t = self._relative_position_bucket(rel, self.num_buckets, self.max_distance).to(device)
            self._tables[key] = t
        return t

    def forward(self, n, device):
        w = self.relative_attention_bias.weight
        idx = self.bucket_table(n, w.device)
        return ops.RelPosBiasFn.apply(w, idx)


class SpatialLinearAttention(nn.Module):
    """video_net.py:313-347: per-frame linear attention (softmax(q) over d, softmax(k) over pixels)."""

    def __init__(self, dim, heads=4, dim_head=32, use_checkpoint=False):
        super().__init__()
        self.use_checkpoint = use_checkpoint
        self.scale = dim_head ** -0.5
        self.heads = heads
        self.dim_head = dim_head
        hidden_dim = dim_head * heads
        self.to_qkv = nn.Conv2d(dim, hidden_dim * 3, 1, bias=False)
        self.to_out = nn.Conv2d(hidden_dim, dim, 1)
        self._cache = ops.PackCache()
        self._cache_out = ops.PackCache()

    def forward_cl(self, x, B, F, residual=None):
        NI, H, W, _ = x.shape
        qkv = ops.ConvFn.apply(x, None, self.to_qkv.weight, None, None, 1, self._cache)
        out = ops.LinearAttnCoreFn.apply(qkv.view(NI * H * W, -1), NI, H * W, self.heads, self.dim_head)
        out = out.view(NI, H, W, self.heads * self.dim_head)
        return ops.ConvFn.apply(out, None, self.to_out.weight, self.to_out.bias, residual, 1, self._cache_out)

    def forward(self, x):
        xc, B, F = ops.to_cl(x)
        return ops.from_cl(self.forward_cl(xc, B, F), B, F).to(x.dtype)


class EinopsToAndFrom(nn.Module):
    """video_net.py:350-365.  The reference materialises "b c f h w" <-> "b (h w) f c" (temporal) or
    "b f (h w) c" (use_mid_attn's spatial block) copies around the wrapped attention; with the channels-last
    internal layout the attention kernels index frames or pixels directly, so this wrapper only records which
    axis is the sequence -- and tells a wrapped Attention (`Attention.seq`)."""

    def __init__(self, from_einops, to_einops, fn):
        super().__init__()
        self.from_einops = from_einops
        self.to_einops = to_einops
        self.fn = fn
        if from_einops != "b c f h w" or to_einops not in ("b (h w) f c", "b f (h w) c"):
            raise NotImplementedError(f"unsupported rearrangement {from_einops} -> {to_einops}")
        if isinstance(fn, Attention):
            fn.seq = "pixels" if to_einops == "b f (h w) c" else "frames"

    def forward_cl(self, x, B, F, **kwargs):
        return self.fn.forward_cl(x, B, F, **kwargs)

    def forward(self, x, **kwargs):
        xc, B, F = ops.to_cl(x)
        return ops.from_cl(self.forward_cl(xc, B, F, **kwargs), B, F).to(x.dtype)


class Attention(nn.Module):
    """video_net.py:368-454.  `seq` (set by the EinopsToAndFrom wrapper) names the sequence axis: "frames" (temporal
    use, the default: the F frames of each pixel column) or "pixels" (use_mid_attn: the h*w pixels of each frame,
    no rotary embedding, no position bias)."""

    def __init__(self, dim, heads=4, dim_head=32, rotary_emb=None, use_checkpoint=False):
        super().__init__()
        self.use_checkpoint = use_checkpoint
        self.scale = dim_head ** -0.5
        self.heads = heads
        self.dim_head = dim_head
        hidden_dim = dim_head * heads
        self.rotary_emb = rotary_emb
        self.to_qkv = nn.Linear(dim, hidden_dim * 3, bias=False)
        self.to_out = nn.Linear(hidden_dim, dim, bias=False)
        self._cache = ops.PackCache()
        self._cache_out = ops.PackCache()
        self.seq = "frames"

    def forward_cl(self, x, B, F, pos_bias=None, focus_present_mask=None, residual=None):
        NI, H, W, _ = x.shape
        hidden = self.heads * self.dim_head
        qkv = ops.ConvFn.apply(x, None, self.to_qkv.weight, None, None, 1, self._cache)
        if exists(focus_present_mask):
            # video_net.py:405-409 / :433-443.  Both branches cost the reference a host sync too.
            if bool(focus_present_mask.all()):
                v = qkv[..., 2 * hidden:].contiguous()
                return ops.ConvFn.apply(v, None, self.to_out.weight, None, residual, 1, self._cache_out)
            if bool(focus_present_mask.any()):
                raise NotImplementedError("per-sample focus_present_mask is not supported by the fused kernel")
        if self.seq == "pixels":
            out = ops.MidAttnCoreFn.apply(qkv.view(NI * H * W, 3 * hidden), NI, H * W, self.heads, self.dim_head)
            return ops.ConvFn.apply(out.view(NI, H, W, hidden), None, self.to_out.weight, None, residual, 1,
                                    self._cache_out)
        if not exists(self.rotary_emb):
            raise NotImplementedError("temporal attention without rotary embedding has no B200 kernel")
        cs, sn = self.rotary_emb.tables(F)
        if pos_bias is None:
            pos_bias = torch.zeros((self.heads, F, F), dtype=torch.float32, device=x.device)
        out = ops.TemporalAttnCoreFn.apply(qkv.view(NI * H * W, 3 * hidden), pos_bias, cs, sn, B, F, H * W,
                                           self.heads, self.dim_head)
        out = out.view(NI, H, W, hidden)
        return ops.ConvFn.apply(out, None, self.to_out.weight, None, residual, 1, self._cache_out)

    def forward(self, x, pos_bias=None, focus_present_mask=None):
        """x: [b, (h w), f, c] (temporal) or [b, f, (h w), c] (seq == "pixels") as the reference's EinopsToAndFrom
        hands it over; attention runs over dim -2 either way."""
        if x.dim() != 4:
            raise ValueError(f"expected a 4-D [b, ., n_seq, c] tensor, got {tuple(x.shape)}")
        if self.seq == "pixels":
            b, f, n, c = x.shape
            xc = x.reshape(b * f, n, 1, c).to(torch.float16).contiguous()
            y = self.forward_cl(xc, b, f, pos_bias=pos_bias, focus_present_mask=focus_present_mask)
            return y.view(b, f, n, c).to(x.dtype)
        b, n, f, c = x.shape
        xc = x.permute(0, 2, 1, 3).reshape(b * f, n, 1, c).to(torch.float16).contiguous()
        y = self.forward_cl(xc, b, f, pos_bias=pos_bias, focus_present_mask=focus_present_mask)
        return y.view(b, f, n, c).permute(0, 2, 1, 3).to(x.dtype)


class UNetModel3D(nn.Module):
    """video_net.py:533-871.  Construction order (and therefore RNG consumption) follows the
    reference line by line, including the second `time_rel_pos_bias` that replaces the first."""

    def __init__(self, n_vars, model_dim, dim_mults=(1, 2, 4, 8), attn_heads=8, attn_dim_head=32,
                 use_sparse_linear_attn=True, use_mid_attn=False, init_kernel_size=7, resnet_groups=8,
                 use_checkpoint=False, use_temp_attn=True, day_cond=True, year_cond=True, cond_map=True):
        super().__init__()
        self.use_temp_attn = use_temp_attn
        self.year_cond = year_cond
        self.day_cond = day_cond
        self.n_vars = n_vars
        self.model_dim = model_dim
        in_channels = n_vars
        out_channels = n_vars
        if cond_map:
            in_channels += n_vars
        init_padding = init_kernel_size // 2
        self.input_conv = nn.Conv3d(in_channels, model_dim, (1, init_kernel_size, init_kernel_size),
                                    padding=(0, init_padding, init_padding))
        rotary_emb = RotaryEmbedding(min(32, attn_dim_head))
        if use_temp_attn:
            self.time_rel_pos_bias = RelativePositionBias(heads=attn_heads, max_distance=32)

            def temporal_op(dim):
                return EinopsToAndFrom("b c f h w", "b (h w) f c",
                                       Attention(dim, heads=attn_heads, dim_head=attn_dim_head, rotary_emb=rotary_emb,
                                                 use_checkpoint=use_checkpoint))
        else:
            def temporal_op(dim):
                raise NotImplementedError(
                    "use_temp_attn=False (TemporalCNN, video_net.py:486-530) is never configured by the "
                    "reference's configs and has no B200 kernel")

        self.time_rel_pos_bias = RelativePositionBias(heads=attn_heads, max_distance=32)

        def temporal_attn(dim):
            return EinopsToAndFrom("b c f h w", "b (h w) f c",
                                   Attention(dim, heads=attn_heads, dim_head=attn_dim_head, rotary_emb=rotary_emb))

        self.input_temp_op = Residual(PreNorm(model_dim, temporal_op(model_dim)))

        dims = [model_dim, *map(lambda m: int(model_dim * m), dim_mults)]
        in_out = list(zip(dims[:-1], dims[1:]))

        time_dim = model_dim * 4
        self.time_mlp = nn.Sequential(SinusoidalPosEmb(model_dim), nn.Linear(model_dim, time_dim), nn.SiLU(),
                                      nn.Linear(time_dim, time_dim))
        if day_cond:
            self.class_emb = nn.Embedding(366, time_dim)
        if year_cond:
            self.year_emb = nn.Embedding(252, time_dim)

        self.downs = nn.ModuleList([])
        self.ups = nn.ModuleList([])
        num_resolutions = len(in_out)
        block_klass = partial(ResnetBlock, groups=resnet_groups, use_checkpoint=use_checkpoint)
        block_klass_cond = partial(block_klass, time_emb_dim=time_dim)

        for ind, (dim_in, dim_out) in enumerate(in_out):
            is_last = ind >= (num_resolutions - 1)
            has_attn = ind >= (num_resolutions - 3)
            self.downs.append(nn.ModuleList([
                block_klass_cond(dim_in, dim_out),
                block_klass_cond(dim_out, dim_out),
                (Residual(PreNorm(dim_out, SpatialLinearAttention(dim_out, heads=attn_heads,
                                                                  use_checkpoint=use_checkpoint)))
                 if use_sparse_linear_attn or has_attn else nn.Identity()),
                Residual(PreNorm(dim_out, temporal_op(dim_out) if not has_attn else temporal_attn(dim_out))),
                Downsample(dim_out) if not is_last else nn.Identity(),
            ]))

        mid_dim = dims[-1]
        self.mid_block1 = block_klass_cond(mid_dim, mid_dim)
        if use_mid_attn:
            spatial_attn = EinopsToAndFrom("b c f h w", "b f (h w) c",
                                           Attention(mid_dim, heads=attn_heads, use_checkpoint=use_checkpoint))
            self.mid_spatial_attn = Residual(PreNorm(mid_dim, spatial_attn))
        else:
            self.mid_spatial_attn = nn.Identity()
        self.mid_temporal_attn = Residual(PreNorm(mid_dim, temporal_attn(mid_dim)))
        self.mid_block2 = block_klass_cond(mid_dim, mid_dim)

        for ind, (dim_in, dim_out) in enumerate(reversed(in_out)):
            is_last = ind >= (num_resolutions - 1)
            has_attn = ind in [0, 1, 2]
            self.ups.append(nn.ModuleList([
                block_klass_cond(dim_out * 2, dim_in),
                block_klass_cond(dim_in, dim_in),
                (Residual(PreNorm(dim_in, SpatialLinearAttention(dim_in, heads=attn_heads,
                                                                 use_checkpoint=use_checkpoint)))
                 if use_sparse_linear_attn or has_attn else nn.Identity()),
                Residual(PreNorm(dim_in, temporal_op(dim_in) if not has_attn else temporal_attn(dim_in))),
                Upsample(dim_in) if not is_last else nn.Identity(),
            ]))

        self.out_conv = nn.Sequential(block_klass(model_dim * 2, model_dim), nn.Conv3d(model_dim, out_channels, 1))

    # ------------------------------------------------------------------------------------------
    @staticmethod
    def _call(mod, x, B, F, **kwargs):
        """Run a child on the internal layout; plain nn.Identity holders pass through."""
        if isinstance(mod, nn.Identity):
            return x
        return mod.forward_cl(x, B, F, **kwargs)

    def _film_blocks(self):
        """ResnetBlocks with a FiLM projection, in forward order (cached)."""
        blks = self.__dict__.get("_film_blocks_cache")
        if blks is None:
            blks = [m for m in self.modules() if isinstance(m, ResnetBlock) and exists(m.mlp)]
            self.__dict__["_film_blocks_cache"] = blks
        return blks

    def _time_embedding(self, timesteps, days, years):
        """video_net.py:822-829."""
        emb = self.time_mlp[0](timesteps)
        h = ops.SmallLinearFn.apply(emb, self.time_mlp[1].weight, self.time_mlp[1].bias, False)
        t = ops.SmallLinearFn.apply(h, self.time_mlp[3].weight, self.time_mlp[3].bias, True)
        if self.day_cond:
            t = t + torch.nn.functional.embedding(days, self.class_emb.weight)
        if self.year_cond:
            t = t + torch.nn.functional.embedding(years, self.year_emb.weight)
        return t

    def forward_frames(self, x, timesteps, cond_map, days=None, years=None, focus_present_mask=None,
                       prob_focus_present=0, frames=None):
        """The network pass.  x: fp32 [B, 1, Fx, H, W] and cond_map: [B, 1, Fc, H, W] with
        Fx, Fc in {1, F} (a single frame is broadcast inside the input-conv kernel instead of
        being expanded, model.py:110-118).  Returns fp32 [B, 1, len(frames), H, W] for the
        requested output frames (default: all F)."""
        if self.n_vars != 1 or cond_map is None:
            raise NotImplementedError("the B200 input/output conv kernels cover n_vars=1 with a cond_map "
                                      "(the only configuration model.UNet builds)")
        B, _, Fx, H, W = x.shape
        Fc = cond_map.shape[2]
        F = max(Fx, Fc)
        if not torch.is_tensor(timesteps):
            timesteps = torch.tensor([timesteps], dtype=torch.long, device=x.device)
        elif timesteps.dim() == 0:
            timesteps = timesteps[None].to(x.device)

        pos_bias = None
        if exists(self.time_rel_pos_bias):
            pos_bias = self.time_rel_pos_bias(F, device=x.device)
            if focus_present_mask is None and prob_focus_present != 0:
                focus_present_mask = prob_mask_like((B,), prob_focus_present, device=x.device)
            # prob 0 -> all-False mask -> the mask branches are never taken (video_net.py:405,433)
        akw = dict(pos_bias=pos_bias, focus_present_mask=focus_present_mask)

        x = ops.InputConvFn.apply(x, cond_map, self.input_conv.weight, self.input_conv.bias, F)
        x = self.input_temp_op.forward_cl(x, B, F, pos_bias=pos_bias)
        r = x
        t = self._time_embedding(timesteps, days, years)
        # every block's FiLM projection of t in ONE launch (they differ only in their weights)
        fb = self._film_blocks()
        films = ops.FilmAllFn.apply(t, *[p for blk in fb for p in (blk.mlp[1].weight, blk.mlp[1].bias)]) if fb else ()
        films = {id(blk): f for blk, f in zip(fb, films)}
        flm = lambda blk: dict(film=films[id(blk)]) if id(blk) in films else dict(time_emb=t)

        h = []
        for block1, block2, spatial_attn, temporal_attn, downsample in self.downs:
            x = block1.forward_cl(x, B, F, **flm(block1))
            x = block2.forward_cl(x, B, F, **flm(block2))
            x = self._call(spatial_attn, x, B, F)
            x = temporal_attn.forward_cl(x, B, F, **akw)
            h.append(x)
            x = self._call(downsample, x, B, F)

        x = self.mid_block1.forward_cl(x, B, F, **flm(self.mid_block1))
        x = self._call(self.mid_spatial_attn, x, B, F)
        x = self.mid_temporal_attn.forward_cl(x, B, F, **akw)
        x = self.mid_block2.forward_cl(x, B, F, **flm(self.mid_block2))

        for block1, block2, spatial_attn, temporal_attn, upsample in self.ups:
            x = block1.forward_cl(x, B, F, x1=h.pop(), **flm(block1))
            x = block2.forward_cl(x, B, F, **flm(block2))
            x = self._call(spatial_attn, x, B, F)
            x = temporal_attn.forward_cl(x, B, F, **akw)
            x = self._call(upsample, x, B, F)

        x = self.out_conv[0].forward_cl(x, B, F, x1=r)
        frames = list(range(F)) if frames is None else list(frames)
        outs = [ops.OutConvFn.apply(x, self.out_conv[1].weight, self.out_conv[1].bias, B, F, f) for f in frames]
        return outs[0].unsqueeze(2) if len(outs) == 1 else torch.stack(outs, dim=2)

    def forward(self, x, timesteps, days=None, years=None, cond_map=None, lowres_cond=None,
                focus_present_mask=None, prob_focus_present=0):
        """video_net.py:766-871.  x, cond_map: [B, 1, F, H, W] -> [B, 1, F, H, W]."""
        if exists(lowres_cond):
            raise NotImplementedError("lowres_cond is never passed by model.UNet (model.py:121)")
        if x.dim() == 5 and x.shape[2] > 1 and x.stride(2) == 0:
            x = x[:, :, :1]  # an `expand`ed single frame (model.py:112): broadcast in-kernel
        if exists(cond_map) and cond_map.dim() == 5 and cond_map.shape[2] > 1 and cond_map.stride(2) == 0:
            cond_map = cond_map[:, :, :1]
        return self.forward_frames(x, timesteps, cond_map, days=days, years=years,
                                   focus_present_mask=focus_present_mask, prob_focus_present=prob_focus_present)
