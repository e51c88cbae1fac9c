"""torch.autograd.Function wrappers: forward and backward both run in the C ABI kernels.

Internal activation layout is channels-last fp16 `[N, H, W, C]` with N = batch*frames (the
reference's NCDHW tensors, permuted once at the network boundary).  Parameters stay fp32 in the
reference's layouts; the fp16 GEMM operand copies (forward layout and data-gradient layout) live in
a registry (`PackCache`) and are refreshed by ONE batched kernel per optimizer step.

Two granularities are offered:
  * block level (`ResnetBlockFn`, `TemporalAttnBlockFn`, `SpatialAttnBlockFn`, `MidAttnBlockFn`): one autograd node
    per reference block (video_net.py ResnetBlock / Residual(PreNorm(attention))), with a
    hand-ordered backward in which residual-gradient adds live in GEMM / LayerNorm epilogues and
    conv-bias gradients come out of the GroupNorm backward's per-channel sums.  `UNetModel3D` uses these.
  * op level (`ConvFn`, `GroupNormSiLUFn`, `LayerNormFn`, ... ): the same kernels one at a time,
    used by the reference-style stand-alone module calls (Block(x), LayerNorm(x), ...).
"""
from __future__ import annotations

import weakref
from typing import Optional, Tuple

import torch

from . import _lib
from . import kernels as K

H16 = torch.float16

# sub-pixel decomposition of a k4/s2/p1 transposed conv: output phase -> [(input offset, kernel index)]
_PHASE_TAPS = {0: [(0, 1), (-1, 3)], 1: [(1, 0), (0, 2)]}


# `ctx.needs_input_grad` is True for a parameter that requires grad even when the call is made under torch.no_grad()
# (and grad mode is always off INSIDE Function.forward), so "will this forward be back-propagated?" has to be read
# at the call site: every Function here goes through _Fn.apply, which records the caller's grad mode.  Without it a
# no-grad call on a trainable model packs data-gradient operands it never uses and -- at F = 1 -- misses the folded
# temporal-attention path that sampling relies on.
_OUTER_GRAD = [True]


class _Fn(torch.autograd.Function):
    @classmethod
    def apply(cls, *args, **kwargs):
        _OUTER_GRAD[0] = torch.is_grad_enabled()
        return super().apply(*args, **kwargs)


def _train(ctx) -> bool:
    return _OUTER_GRAD[0] and any(ctx.needs_input_grad)


def _c(t: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
    return None if t is None else t.contiguous()


def _phase(ph: int, pw: int):
    taps, koff = [], []
    for dh, kh in _PHASE_TAPS[ph]:
        for dw, kw in _PHASE_TAPS[pw]:
            taps.append((dh, dw))
            koff.append(kh * 4 + kw)
    return taps, koff


# ------------------------------------------------------------------------------------------------
# packed fp16 operand copies of the fp32 parameters
# ------------------------------------------------------------------------------------------------
# Fused / capturable optimizers update parameters without bumping `Tensor._version`, so validity is
# also keyed on a global epoch that every torch optimizer step advances.
_WEIGHT_EPOCH = [0]


def invalidate_weight_cache(*_args, **_kwargs) -> None:
    """Call after modifying parameters by any means torch cannot see (raw pointer writes)."""
    _WEIGHT_EPOCH[0] += 1


try:
    from torch.optim.optimizer import register_optimizer_step_post_hook as _reg_hook
    _reg_hook(invalidate_weight_cache)
except Exception:  # pragma: no cover - very old torch
    pass


class _PackEntry:
    __slots__ = ("wref", "src_off", "O", "T", "I", "so", "si", "taps", "out", "key", "serial")


_ENTRIES: list = []          # every packed copy ever requested (weak refs to the parameters)
_PLAN = {"n": -1, "ptrs": None, "descs": None}
_PREPACK_SERIAL = [0]        # bumped by prepack_all(); entries packed in the current step carry it


def _key(weight: torch.Tensor):
    return (weight.data_ptr(), weight._version, _WEIGHT_EPOCH[0])


class PackCache:
    """Per-layer view of the packed-operand registry: `get(weight, tag, spec)` returns the fp16 copy
    `dst[o][t][i] = weight.flatten()[src_off + o*so + i*si + taps[t]]`, re-packing it (in place, so
    the address is stable for CUDA graphs) when the parameter changed.  While a training step is
    being captured, a copy that was not refreshed by `prepack_all()` in this step is always
    re-packed so that the pack is part of the graph."""

    def __init__(self):
        self._d = {}

    def get(self, weight: torch.Tensor, tag, spec, train: bool = False) -> torch.Tensor:
        """`train`: the caller is the forward of a step that will be back-propagated (inside an
        autograd.Function grad mode is always off, so the caller passes any(ctx.needs_input_grad))."""
        ent = self._d.get(tag)
        if ent is None or ent.wref() is not weight:
            ent = _PackEntry()
            ent.wref = weakref.ref(weight)
            ent.src_off, ent.O, ent.T, ent.I, ent.so, ent.si, ent.taps = spec
            ent.out = torch.empty((ent.O, ent.T * ent.I), dtype=H16, device=weight.device)
            ent.key, ent.serial = None, -1
            self._d[tag] = ent
            _ENTRIES.append(ent)
        key = _key(weight)
        force = (train and weight.is_cuda and torch.cuda.is_current_stream_capturing()
                 and ent.serial != _PREPACK_SERIAL[0])
        if force or ent.key != key:
            src = weight.detach().reshape(-1)
            if ent.src_off:
                src = src[ent.src_off:]
            K.pack_weight(src, ent.O, ent.T, ent.I, ent.so, ent.si, ent.taps, out=ent.out)
            ent.key, ent.serial = key, _PREPACK_SERIAL[0]
        return ent.out

    def __deepcopy__(self, memo):
        return PackCache()


def prepack_all() -> int:
    """Refresh every registered packed copy with one kernel launch (the training engine calls this
    at the top of each step, after the optimizer changed the weights).  Returns the entry count."""
    live = [e for e in _ENTRIES if e.wref() is not None]
    if len(live) != len(_ENTRIES):
        _ENTRIES[:] = live
    if not live:
        return 0
    ptrs = tuple((e.wref().data_ptr(), e.out.data_ptr()) for e in live)
    if _PLAN["n"] != len(live) or _PLAN["ptrs"] != ptrs:
        arr = (_lib.PackDesc * len(live))()
        for d, e in zip(arr, live):
            d.src = e.wref().data_ptr() + 4 * e.src_off
            d.dst = e.out.data_ptr()
            d.O, d.T, d.I, d.so, d.si = e.O, e.T, e.I, e.so, e.si
            for i, o in enumerate(e.taps):
                d.tap_off[i] = int(o)
        host = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8)
        _PLAN.update(n=len(live), ptrs=ptrs, descs=host.to(live[0].out.device))
    _PREPACK_SERIAL[0] += 1
    _lib.call("cesm_pack_weights_batched", _PLAN["descs"].data_ptr(), len(live), K._stream())
    for e in live:
        e.key, e.serial = _key(e.wref()), _PREPACK_SERIAL[0]
    return len(live)


# F = 1 inference fold  W_out W_v  of a temporal-attention block (see TemporalAttnBlockFn.forward): one
# [C, C] fp16 operand per block, rebuilt IN PLACE (stable address for captured sampling graphs) whenever the
# weights changed; `refresh_folds()` lets an engine bring every fold up to date outside its graph.
_FOLDS: list = []


def _fold_compute(ent, wqkv, wout, gamma) -> None:
    """Rebuild the tensors of a fold entry IN PLACE (their addresses are baked into captured graphs)."""
    C, hidden = ent[1].shape[0], ent[4]
    wv = wqkv.detach().reshape(3 * hidden, C)[2 * hidden:].float()
    wo = wout.detach().reshape(C, hidden).float()
    w = wo @ wv                                  # [C out, C in]: the implicit-GEMM operand layout
    ent[1].copy_(w)
    if gamma is not None:                        # LayerNorm folded into the GEMM epilogue (kernels.igemm ln_fold)
        ent[6].copy_(w * gamma.detach().reshape(1, C).float())
        ent[7].copy_(ent[6].float().sum(dim=1))  # of the fp16 values the tensor core multiplies


def _fold_f1(meta, wqkv, wout, hidden: int, C: int, gamma=None):
    """W_out W_v of a temporal-attention block for the one-frame path.  Returns the fp16 [C, C] matrix, or -- with
    `gamma` (C == 64) -- the pair (W * gamma, its row sums) that `kernels.igemm(..., ln_fold=)` takes."""
    key = (_key(wqkv), _key(wout), None if gamma is None else _key(gamma))
    ent = meta.__dict__.get("fold_f1")
    if ent is None or ent[1].device != wqkv.device or (gamma is not None and ent[5] is None):
        dev = wqkv.device
        ent = [None, torch.empty((C, C), dtype=H16, device=dev), weakref.ref(wqkv), weakref.ref(wout), hidden,
               None if gamma is None else weakref.ref(gamma),
               None if gamma is None else torch.empty((C, C), dtype=H16, device=dev),
               None if gamma is None else torch.empty((C,), dtype=torch.float32, device=dev)]
        meta.__dict__["fold_f1"] = ent
        _FOLDS.append(ent)
    if ent[0] != key:
        _fold_compute(ent, wqkv, wout, gamma)
        ent[0] = key
    return ent[1] if gamma is None else (ent[6], ent[7])


def refresh_folds() -> None:
    live = [e for e in _FOLDS if e[2]() is not None and e[3]() is not None and (e[5] is None or e[5]() is not None)]
    _FOLDS[:] = live
    for e in live:
        wqkv, wout = e[2](), e[3]()
        gamma = None if e[5] is None else e[5]()
        key = (_key(wqkv), _key(wout), None if gamma is None else _key(gamma))
        if e[0] != key:
            _fold_compute(e, wqkv, wout, gamma)
            e[0] = key


# ------------------------------------------------------------------------------------------------
# gradient delivery
# ------------------------------------------------------------------------------------------------
# The training engine pre-allocates every parameter gradient as a view into one flat buffer and
# registers itself here; weight gradients are then accumulated straight into those views by the
# un-packing kernel (no temporary, no autograd add) and the sink is told the parameter is ready.
_GRAD_SINK = [None]


def set_grad_sink(sink) -> None:
    _GRAD_SINK[0] = sink


def _direct(weight: torch.Tensor) -> bool:
    sink = _GRAD_SINK[0]
    return sink is not None and weight.grad is not None and sink.owns(weight)


def _direct_all(*params) -> bool:
    return all(p is not None and _direct(p) for p in params)


def _ready(*params) -> None:
    for p in params:
        _GRAD_SINK[0].ready(p)


# Condition-gradient sink (engine.SaliencyEngine): (fp32 buffer, scale) or None.  While set, the input convolution's
# backward adds scale * d cond straight into the buffer (the data-gradient kernel's accumulate mode) and hands
# autograd no gradient for cond, so averaging over draws costs no extra launch.
_COND_GRAD_SINK = [None]


def set_cond_grad_sink(buf: Optional[torch.Tensor], scale: float = 1.0) -> None:
    _COND_GRAD_SINK[0] = None if buf is None else (buf, float(scale))


# Leaf-gradient side stream (engine mode only).  Weight gradients are not on the backward pass's critical chain: they
# are launched on a second stream that forks from the main one where their inputs become available and joins before
# the optimizer (TrainEngine).  At the coarse U-Net levels most kernels have a nearly empty last wave; work from the
# other stream fills those SMs (measured: 11.44 -> 11.03 ms per step, profiles/r02_side_stream_ab.txt).  Inputs are
# kept alive until the join (`_SIDE_KEEP`), so no block is recycled under a kernel that is still reading it -- eagerly
# or inside a captured graph.  (A third stream for the ResnetBlocks' 1x1 residual convolutions, forward and backward,
# was tried as well: no further gain.)
_SIDE = [None]       # torch.cuda.Stream or None
_SIDE_KEEP: list = []


def set_side_stream(stream) -> None:
    _SIDE[0] = stream
    _SIDE_KEEP.clear()


def join_side_stream() -> None:
    """Main stream waits for everything issued on the side stream; the kept inputs may be released."""
    side = _SIDE[0]
    if side is not None:
        torch.cuda.current_stream().wait_stream(side)
    _SIDE_KEEP.clear()


class _on_side:
    """`with _on_side(tensors...):` -- run the enclosed launches on the side stream (if one is set and the gradient
    sink is active), after everything already queued on the current stream."""

    def __init__(self, *tensors):
        self.side = _SIDE[0] if _GRAD_SINK[0] is not None else None
        self.tensors = tensors
        self.ctx = None

    def __enter__(self):
        if self.side is not None:
            self.side.wait_stream(torch.cuda.current_stream())
            _SIDE_KEEP.append(self.tensors)
            self.ctx = torch.cuda.stream(self.side)
            self.ctx.__enter__()
        return self

    def __exit__(self, *exc):
        if self.ctx is not None:
            self.ctx.__exit__(*exc)
        return False


def _wgrad_into_param(weight, x0, x1, dy, taps, so, si, tap_off, last: bool = True,
                      into: Optional[torch.Tensor] = None, **kw):
    """Weight gradient accumulated by the tcgen05 kernel's epilogue directly in `weight`'s own layout:
    into weight.grad (engine mode; returns None and notifies the sink) or into a zeroed tensor."""
    T = len(taps)
    if _direct(weight):
        sink = _GRAD_SINK[0]
        with _on_side(x0, x1, dy):
            if T == 1:  # same layout as the kernel's packed output: coalesced atomics straight into .grad
                K.wgrad(x0, dy, x1=x1, taps=taps, into=weight.grad, layout=(so, si, tap_off), **kw)
            else:       # accumulate into a persistent packed scratch; the sink un-packs a whole bucket at once
                cout = dy.shape[-1]
                ctot = x0.shape[-1] + (0 if x1 is None else x1.shape[-1])
                scratch = sink.scratch(weight, tuple(tap_off), (cout, T, ctot, so, si, list(tap_off)))
                K.wgrad(x0, dy, x1=x1, taps=taps, into=scratch, layout=(T * ctot, 1, [t * ctot for t in range(T)]), **kw)
        if last:
            sink.ready(weight)
        return None
    dwt = torch.zeros_like(weight) if into is None else into
    K.wgrad(x0, dy, x1=x1, taps=taps, into=dwt, layout=(so, si, tap_off), **kw)
    return dwt


# ------------------------------------------------------------------------------------------------
# conv helpers shared by the op-level and block-level functions
# ------------------------------------------------------------------------------------------------
def _sq_taps(ks: int):
    r = ks // 2
    return [(kh - r, kw - r) for kh in range(ks) for kw in range(ks)]


def _conv_fwd_weight(cache: PackCache, weight, cout: int, ctot: int, ks: int, train: bool):
    kk = ks * ks
    return cache.get(weight, "fwd", (0, cout, kk, ctot, ctot * kk, kk, list(range(kk))), train)


def _conv_dgrad_weights(cache: PackCache, weight, cout: int, c0: int, c1: int, ks: int, train: bool):
    """Data-gradient operands [ci][t][co] = W[co, ci, t] for each concatenated source (only made
    for a step that will be back-propagated)."""
    if not train:
        return None, None
    kk, ctot = ks * ks, c0 + c1
    w0 = cache.get(weight, "dgrad0", (0, c0, kk, cout, kk, ctot * kk, list(range(kk))), train)
    w1 = (cache.get(weight, "dgrad1", (c0 * kk, c1, kk, cout, kk, ctot * kk, list(range(kk))), train)
          if c1 else None)
    return w0, w1


def _bias_grad(bias, dy):
    """Column sums of dy as the gradient of a conv bias: added straight into bias.grad on the side stream in engine
    mode (returns None), else returned for autograd to accumulate."""
    if bias is not None and _direct_all(bias):
        with _on_side(dy):
            K.colsum(dy, into=bias.grad)
        _ready(bias)
        return None
    return K.colsum(dy)


def _conv_wgrad(weight, x0, x1, dy, ks: int):
    cout = weight.shape[0]
    ctot = x0.shape[-1] + (0 if x1 is None else x1.shape[-1])
    kk = ks * ks
    return _wgrad_into_param(weight, x0, x1, dy, _sq_taps(ks), ctot * kk, kk, list(range(kk)))


# ------------------------------------------------------------------------------------------------
# op-level: convolutions / linears on the tcgen05 implicit GEMM
# ------------------------------------------------------------------------------------------------
class ConvFn(_Fn):
    """Stride-1 conv with a square k x k kernel (k in {1, 3}) or a linear layer, over one or two
    concatenated channels-last sources, with fused bias and residual.

    weight: fp32 [cout, cin, (1,) k, k] (Conv3d / Conv2d) or [cout, cin] (Linear).
    Reference: video_net.py:215 (Block.proj), :246 (res_conv), :322-323, :380-381.
    """

    @staticmethod
    def forward(ctx, x0, x1, weight, bias, residual, ksize: int, cache: PackCache):
        x0, x1, residual = _c(x0), _c(x1), _c(residual)
        cout = weight.shape[0]
        c0 = x0.shape[-1]
        c1 = 0 if x1 is None else x1.shape[-1]
        assert weight.numel() == cout * (c0 + c1) * ksize * ksize, (weight.shape, c0, c1, ksize)
        train = _train(ctx)
        wt = _conv_fwd_weight(cache, weight, cout, c0 + c1, ksize, train)
        ctx.wd = _conv_dgrad_weights(cache, weight, cout, c0, c1, ksize, train)
        y = K.igemm(x0, wt, a1=x1, taps=_sq_taps(ksize), bias=bias, residual=residual)
        ctx.save_for_backward(x0, x1, weight)
        ctx.ksize, ctx.has_bias, ctx.has_res = ksize, bias is not None, residual is not None
        return y

    @staticmethod
    def backward(ctx, dy):
        x0, x1, weight = ctx.saved_tensors
        dy = dy.contiguous()
        ntaps = [(-dh, -dw) for dh, dw in _sq_taps(ctx.ksize)]
        dx0 = dx1 = dwt = db = None
        if ctx.needs_input_grad[0]:
            dx0 = K.igemm(dy, ctx.wd[0], taps=ntaps)
        if x1 is not None and ctx.needs_input_grad[1]:
            dx1 = K.igemm(dy, ctx.wd[1], taps=ntaps)
        if ctx.needs_input_grad[2]:
            dwt = _conv_wgrad(weight, x0, x1, dy, ctx.ksize)
        if ctx.has_bias and ctx.needs_input_grad[3]:
            db = K.colsum(dy)
        dres = dy if (ctx.has_res and ctx.needs_input_grad[4]) else None
        return dx0, dx1, dwt, db, dres, None, None


class DownsampleFn(_Fn):
    """Conv3d(dim, dim, (1,4,4), (1,2,2), (0,1,1)) -- video_net.py:61-62."""

    TAPS = [(kh - 1, kw - 1) for kh in range(4) for kw in range(4)]

    @staticmethod
    def forward(ctx, x, weight, bias, cache: PackCache):
        x = x.contiguous()
        c = x.shape[-1]
        train = _train(ctx)
        wt = cache.get(weight, "fwd", (0, c, 16, c, c * 16, 16, list(range(16))), train)
        # data gradient: four sub-pixel phases, [ci][t][co] = W[co, ci, kh_t, kw_t]
        ctx.wd = {(ph, pw): cache.get(weight, ("dgrad", ph, pw), (0, c, 4, c, 16, c * 16, _phase(ph, pw)[1]), train)
                  for ph in (0, 1) for pw in (0, 1)} if train else None
        y = K.igemm(x, wt, taps=DownsampleFn.TAPS, stride=2, bias=bias)
        ctx.save_for_backward(x, weight)
        ctx.bias_ref = bias
        return y

    @staticmethod
    def backward(ctx, dy):
        x, weight = ctx.saved_tensors
        dy = dy.contiguous()
        n, h, w, c = x.shape
        dx = dwt = db = None
        if ctx.needs_input_grad[0]:
            dx = torch.empty_like(x)
            for (ph, pw), wd in ctx.wd.items():
                K.igemm(dy, wd, taps=_phase(ph, pw)[0], out=dx, out_hw=(h // 2, w // 2), out_place=(2, 2, ph, pw))
        if ctx.needs_input_grad[1]:
            dwt = _wgrad_into_param(weight, x, None, dy, DownsampleFn.TAPS, c * 16, 16, list(range(16)), stride=2)
        if ctx.needs_input_grad[2]:
            db = _bias_grad(ctx.bias_ref, dy)
        return dx, dwt, db, None


class UpsampleFn(_Fn):
    """ConvTranspose3d(dim, dim, (1,4,4), (1,2,2), (0,1,1)) as four sub-pixel 2x2 convs -- video_net.py:65-66."""

    @staticmethod
    def forward(ctx, x, weight, bias, cache: PackCache):
        x = x.contiguous()
        n, h, w, c = x.shape
        out = torch.empty((n, 2 * h, 2 * w, c), dtype=H16, device=x.device)
        # [ci][t][co] = W[ci, co, kh, kw] for the data gradient (a stride-2 conv of dy)
        train = _train(ctx)
        ctx.wd = cache.get(weight, "dgrad", (0, c, 16, c, c * 16, 16, list(range(16))), train) if train else None
        for ph in (0, 1):
            for pw in (0, 1):
                taps, koff = _phase(ph, pw)
                # [co][t][ci] = W[ci, co, kh_t, kw_t]
                wt = cache.get(weight, ("fwd", ph, pw), (0, c, 4, c, 16, c * 16, koff), train)
                K.igemm(x, wt, taps=taps, out=out, out_hw=(h, w), out_place=(2, 2, ph, pw), bias=bias)
        ctx.save_for_backward(x, weight)
        ctx.bias_ref = bias
        return out

    @staticmethod
    def backward(ctx, dy):
        x, weight = ctx.saved_tensors
        dy = dy.contiguous()
        n, h, w, c = x.shape
        dx = dwt = db = None
        if ctx.needs_input_grad[0]:
            dx = K.igemm(dy, ctx.wd, taps=DownsampleFn.TAPS, stride=2)
        if ctx.needs_input_grad[1]:
            into = None if _direct(weight) else torch.zeros_like(weight)
            for n_ph, (ph, pw) in enumerate([(0, 0), (0, 1), (1, 0), (1, 1)]):
                taps, koff = _phase(ph, pw)
                # ConvTranspose weight is [ci, co, kh, kw]: co stride 16, ci stride c*16
                dwt = _wgrad_into_param(weight, x, None, dy, taps, 16, c * 16, koff, last=(n_ph == 3), into=into,
                                        grid_hw=(h, w), dy_place=(2, 2, ph, pw))
        if ctx.needs_input_grad[2]:
            db = _bias_grad(ctx.bias_ref, dy)
        return dx, dwt, db, None


# ------------------------------------------------------------------------------------------------
# op-level: normalisation
# ------------------------------------------------------------------------------------------------
class GroupNormSiLUFn(_Fn):
    """GroupNorm -> optional FiLM (x*(scale+1)+shift) -> SiLU -> optional residual add
    (video_net.py:221-227, :265).  x: [B*F, H, W, C]; film: fp32 [B, 2C]."""

    @staticmethod
    def forward(ctx, x, gamma, beta, film, residual, B: int, G: int, eps: float):
        x, film, residual = x.contiguous(), _c(film), _c(residual)
        sums = K.gn_stats(x, B, G)
        out = K.gn_apply_fwd(x, sums, gamma, beta, film, residual, B, G, eps)
        ctx.save_for_backward(x, sums, gamma, beta, film)
        ctx.cfg = (B, G, eps, residual is not None)
        return out

    @staticmethod
    def backward(ctx, dout):
        x, sums, gamma, beta, film = ctx.saved_tensors
        B, G, eps, has_res = ctx.cfg
        dout = dout.contiguous()
        dx, dgamma, dbeta, dfilm = K.gn_bwd(x, dout, sums, gamma, beta, film, B, G, eps)
        return dx, dgamma, dbeta, dfilm, (dout if has_res else None), None, None, None


class LayerNormFn(_Fn):
    """Channel LayerNorm with gain only (video_net.py:84-87); gamma is the [1,C,1,1,1] parameter."""

    @staticmethod
    def forward(ctx, x, gamma, eps: float):
        x = x.contiguous()
        g = gamma.reshape(-1)
        ctx.save_for_backward(x, g)
        ctx.eps, ctx.gshape = eps, gamma.shape
        return K.ln_fwd(x, g, eps)

    @staticmethod
    def backward(ctx, dy):
        x, g = ctx.saved_tensors
        dx, dg = K.ln_bwd(x, g, dy.contiguous(), None, ctx.eps)
        return dx, dg.view(ctx.gshape), None


# ------------------------------------------------------------------------------------------------
# op-level: attention cores
# ------------------------------------------------------------------------------------------------
class TemporalAttnCoreFn(_Fn):
    """q*scale, RoPE, q.k + bias, softmax over frames, .v (video_net.py:413-453).  qkv: [B*F*HW, 3*H*D]."""

    @staticmethod
    def forward(ctx, qkv, pos_bias, cs, sn, B: int, F: int, HW: int, H: int, D: int):
        qkv, pos_bias = qkv.contiguous(), pos_bias.contiguous().float()
        scale = D ** -0.5
        out, lse = K.tattn_fwd(qkv, pos_bias, cs, sn, B, F, HW, H, D, scale)
        if F <= 4:  # the small-window kernel recomputes the softmax in the backward
            ctx.save_for_backward(qkv, pos_bias, cs, sn)
        else:
            ctx.save_for_backward(qkv, pos_bias, cs, sn, out, lse)
        ctx.dims = (B, F, HW, H, D, scale)
        return out

    @staticmethod
    def backward(ctx, dout):
        B, F, HW, H, D, scale = ctx.dims
        if F <= 4:
            (qkv, pos_bias, cs, sn), out, lse = ctx.saved_tensors, None, None
        else:
            qkv, pos_bias, cs, sn, out, lse = ctx.saved_tensors
        dqkv, dbias = K.tattn_bwd(qkv, pos_bias, cs, sn, out, lse, dout.contiguous(), B, F, HW, H, D, scale)
        return dqkv, dbias, None, None, None, None, None, None, None


class MidAttnCoreFn(_Fn):
    """softmax((q * scale) k^T) v over all n pixels of each image, no mask / bias / rotary (video_net.py:413-453 as the
    use_mid_attn block calls it).  qkv: [NI*n, 3*H*D] -> [NI*n, H*D]."""

    @staticmethod
    def forward(ctx, qkv, NI: int, n: int, H: int, D: int):
        qkv = qkv.contiguous()
        out, lse = K.mattn_fwd(qkv, NI, n, H, D, D ** -0.5)
        ctx.save_for_backward(qkv, out, lse)
        ctx.dims = (NI, n, H, D)
        return out

    @staticmethod
    def backward(ctx, dout):
        qkv, out, lse = ctx.saved_tensors
        NI, n, H, D = ctx.dims
        return K.mattn_bwd(qkv, out, lse, dout.contiguous(), NI, n, H, D, D ** -0.5), None, None, None, None


class RelPosBiasFn(_Fn):
    """Embedding gather of the T5 bucket table -> [heads, n, n] (video_net.py:302-310).  The
    table has 32 x heads entries; gather and scatter-add are index ops on a few hundred floats."""

    @staticmethod
    def forward(ctx, weight, idx):
        ctx.save_for_backward(idx)
        ctx.shape = weight.shape
        return weight.detach()[idx].permute(2, 0, 1).float().contiguous()

    @staticmethod
    def backward(ctx, dbias):
        (idx,) = ctx.saved_tensors
        dw = torch.zeros(ctx.shape, dtype=dbias.dtype, device=dbias.device)
        dw.index_add_(0, idx.reshape(-1), dbias.permute(1, 2, 0).reshape(-1, ctx.shape[1]))
        return dw, None


class LinearAttnCoreFn(_Fn):
    """softmax(q) over d, softmax(k) over pixels, ctx = k^T v, out = ctx^T q (video_net.py:338-344)."""

    @staticmethod
    def forward(ctx, qkv, NI: int, n: int, H: int, D: int):
        qkv = qkv.contiguous()
        scale = D ** -0.5
        out, ws = K.linattn_fwd(qkv, NI, n, H, D, scale)
        ctx.save_for_backward(qkv, ws)
        ctx.dims = (NI, n, H, D, scale)
        return out

    @staticmethod
    def backward(ctx, dout):
        qkv, ws = ctx.saved_tensors
        NI, n, H, D, scale = ctx.dims
        return K.linattn_bwd(qkv, ws, dout.contiguous(), NI, n, H, D, scale), None, None, None, None


# ------------------------------------------------------------------------------------------------
# block level
# ------------------------------------------------------------------------------------------------
class BlockMeta:
    """Static configuration + pack caches of one block (kept on the nn.Module)."""

    def __init__(self, **kw):
        self.__dict__.update(kw)

    def __deepcopy__(self, memo):
        return BlockMeta(**{k: (PackCache() if isinstance(v, PackCache) else v) for k, v in self.__dict__.items()
                            if k != "fold_f1"})


class ResnetBlockFn(_Fn):
    """video_net.py:254-265 as one node:  out = Block2(Block1(cat(x, x1); film)) + res(cat(x, x1)),
    Block = conv(1,3,3) + bias -> GroupNorm -> FiLM -> SiLU, res = 1x1x1 conv or identity.

    args: x, x1 (or None), film fp32 [B, 2C] (or None), w1, b1, g1w, g1b, w2, b2, g2w, g2b,
          wres, bres (or None, None), B, meta(G, eps, c1, c2, cres: PackCache)."""

    @staticmethod
    def forward(ctx, x, x1, film, w1, b1, g1w, g1b, w2, b2, g2w, g2b, wres, bres, B, meta):
        x, x1, film = x.contiguous(), _c(x1), _c(film)
        G, eps = meta.G, meta.eps
        c0 = x.shape[-1]
        cx1 = 0 if x1 is None else x1.shape[-1]
        cout = w1.shape[0]
        train = _train(ctx)
        if wres is None:
            res = x
        else:
            res = K.igemm(x, _conv_fwd_weight(meta.cres, wres, cout, c0 + cx1, 1, train), a1=x1, bias=bres)
        F = x.shape[0] // B
        # GroupNorm statistics come out of the conv epilogue (no extra pass over y)
        sums1 = K.zero_scratch((B, G, 2), x.device)
        y1 = K.igemm(x, _conv_fwd_weight(meta.c1, w1, cout, c0 + cx1, 3, train), a1=x1, taps=K.TAPS_3x3, bias=b1,
                     gn_sums=sums1, gn_frames=F)
        h1 = K.gn_apply_fwd(y1, sums1, g1w, g1b, film, None, B, G, eps)
        sums2 = K.zero_scratch((B, G, 2), x.device)
        y2 = K.igemm(h1, _conv_fwd_weight(meta.c2, w2, cout, cout, 3, train), taps=K.TAPS_3x3, bias=b2,
                     gn_sums=sums2, gn_frames=F)
        out = K.gn_apply_fwd(y2, sums2, g2w, g2b, None, res, B, G, eps)
        ctx.wd1 = _conv_dgrad_weights(meta.c1, w1, cout, c0, cx1, 3, train)
        ctx.wd2 = _conv_dgrad_weights(meta.c2, w2, cout, cout, 0, 3, train)
        ctx.wdres = None if wres is None else _conv_dgrad_weights(meta.cres, wres, cout, c0, cx1, 1, train)
        ctx.save_for_backward(x, x1, film, y1, sums1, h1, y2, sums2, w1, g1w, g1b, w2, g2w, g2b, wres, b1, b2, bres)
        ctx.cfg = (B, G, eps)
        return out

    @staticmethod
    def backward(ctx, dout):
        x, x1, film, y1, sums1, h1, y2, sums2, w1, g1w, g1b, w2, g2w, g2b, wres, b1, b2, bres = ctx.saved_tensors
        B, G, eps = ctx.cfg
        dout = dout.contiguous()
        ntaps = [(-dh, -dw) for dh, dw in K.TAPS_3x3]
        need = ctx.needs_input_grad  # a frozen weight (requires_grad False) gets no weight-gradient launch
        # GroupNorm / conv-bias gradients go straight into the parameters' .grad in engine mode
        # ---- block 2 ----
        if _direct_all(g2w, g2b, b2):
            dy2, _, _, _, _ = K.gn_bwd(y2, dout, sums2, g2w, g2b, None, B, G, eps, conv_bias_grad=True,
                                       into=(g2w.grad, g2b.grad, b2.grad))
            _ready(g2w, g2b, b2)
            dg2w = dg2b = db2 = None
        else:
            dy2, dg2w, dg2b, _, db2 = K.gn_bwd(y2, dout, sums2, g2w, g2b, None, B, G, eps, conv_bias_grad=True)
        dw2 = _conv_wgrad(w2, h1, None, dy2, 3) if need[7] else None
        dh1 = K.igemm(dy2, ctx.wd2[0], taps=ntaps)
        # ---- block 1 ----
        if _direct_all(g1w, g1b, b1):
            dy1, _, _, dfilm, _ = K.gn_bwd(y1, dh1, sums1, g1w, g1b, film, B, G, eps, conv_bias_grad=True,
                                           into=(g1w.grad, g1b.grad, b1.grad))
            _ready(g1w, g1b, b1)
            dg1w = dg1b = db1 = None
        else:
            dy1, dg1w, dg1b, dfilm, db1 = K.gn_bwd(y1, dh1, sums1, g1w, g1b, film, B, G, eps, conv_bias_grad=True)
        dw1 = _conv_wgrad(w1, x, x1, dy1, 3) if need[3] else None
        # ---- inputs: conv-1 data gradient with the residual-branch gradient added in its epilogue ----
        dx = dx1 = dwres = dbres = None
        if wres is None:
            if need[0]:
                dx = K.igemm(dy1, ctx.wd1[0], taps=ntaps, residual=dout)
        else:
            if need[0]:
                r0 = K.igemm(dout, ctx.wdres[0])
                dx = K.igemm(dy1, ctx.wd1[0], taps=ntaps, residual=r0)
            if x1 is not None and need[1]:
                r1 = K.igemm(dout, ctx.wdres[1])
                dx1 = K.igemm(dy1, ctx.wd1[1], taps=ntaps, residual=r1)
            if need[11]:
                dwres = _conv_wgrad(wres, x, x1, dout, 1)
            if need[12] and _direct_all(bres):
                with _on_side(dout):
                    K.colsum(dout, into=bres.grad)
                _ready(bres)
            elif need[12]:
                dbres = K.colsum(dout)
        return dx, dx1, dfilm, dw1, db1, dg1w, dg1b, dw2, db2, dg2w, dg2b, dwres, dbres, None, None


def _qkv_backward(wqkv, wdq, xn, dqkv4, need_w: bool = True):
    """Data gradient (w.r.t. the projection's input xn) and weight gradient of the bias-free q/k/v projection.
    For 64 input channels both come from ONE pass over dqkv (cesm_qkv_bwd: 101 us instead of 83 + 84 us at
    192x288); otherwise from the implicit-GEMM and weight-gradient kernels.  A frozen projection (`need_w` False)
    takes the data-gradient GEMM alone.  -> (dxn, dwqkv or None)."""
    C, cout = xn.shape[-1], dqkv4.shape[-1]
    if not need_w:
        return K.igemm(dqkv4, wdq), None
    if C == 64 and cout % 128 == 0 and cout <= 768:
        if _direct(wqkv):
            dxn, _ = K.qkv_bwd(dqkv4, xn, wdq, dw_into=wqkv.grad)
            _ready(wqkv)
            return dxn, None
        dxn, dw = K.qkv_bwd(dqkv4, xn, wdq)
        return dxn, dw.view_as(wqkv)
    return K.igemm(dqkv4, wdq), _conv_wgrad(wqkv, xn, None, dqkv4, 1)


class TemporalAttnBlockFn(_Fn):
    """Residual(PreNorm(EinopsToAndFrom(Attention))) (video_net.py:69-98, 357-454) as one node:
    y = to_out(attn(to_qkv(LN(x)))) + x.
    args: x, gamma [1,C,1,1,1], wqkv, wout, pos_bias, cs, sn, B, F, meta(heads, dim_head, eps, cq, co)."""

    @staticmethod
    def forward(ctx, x, gamma, wqkv, wout, pos_bias, cs, sn, B, F, meta):
        x = x.contiguous()
        NI, H_, W_, C = x.shape
        heads, D, eps = meta.heads, meta.dim_head, meta.eps
        hidden = heads * D
        g = gamma.reshape(-1)
        pos_bias = pos_bias.contiguous().float()
        train = _train(ctx)
        if F == 1 and not train and C == 64:
            # (see below) ... and at 64 channels the LayerNorm goes into the same kernel: a thread of the GEMM
            # epilogue holds the whole row of x as its residual, so  y = x + rstd (x (W gamma)^T - mean colsum)
            wln, colsum = _fold_f1(meta, wqkv, wout, hidden, C, gamma=gamma)
            return K.igemm(x, wln, residual=x, ln_fold=(colsum, eps))
        xn = K.ln_fwd(x, g, eps)
        if F == 1 and not train:
            # one frame (every step of the sampling chain): the softmax over a single key is exactly 1, so the
            # attention output IS v -- the reference computes the same thing the long way (video_net.py:
            # 444-450: softmax of a 1-element row).  Only the v third of to_qkv is projected; q, k, RoPE, the
            # position bias and the attention kernel drop out.
            # ... and with nothing non-linear between the v projection and to_out, the two linears collapse
            # into ONE C x C matrix W_out W_v, folded once per weight version: y = x + LN(x) (W_out W_v)^T.
            return K.igemm(xn, _fold_f1(meta, wqkv, wout, hidden, C), residual=x)
        wq = _conv_fwd_weight(meta.cq, wqkv, 3 * hidden, C, 1, train)
        if not train and K.tattn_proj_ok(C, F, H_ * W_, heads, D):
            # 64 input channels, F <= 3, no gradients: q|k|v never reach HBM (csrc/tattn_proj.cu).  A training step
            # keeps the unfused path: a backward that recomputes q|k|v from xn was slower than streaming them back
            # (profiles/r02_fused_tattn_ab.txt).
            o = K.tattn_proj_fwd(xn.view(-1, C), wq, pos_bias, cs, sn, B, F, H_ * W_, heads, D, D ** -0.5)
            return K.igemm(o.view(NI, H_, W_, hidden), _conv_fwd_weight(meta.co, wout, C, hidden, 1, train), residual=x)
        qkv = K.igemm(xn, wq)
        o, lse = K.tattn_fwd(qkv.view(-1, 3 * hidden), pos_bias, cs, sn, B, F, H_ * W_, heads, D, D ** -0.5)
        y = K.igemm(o.view(NI, H_, W_, hidden), _conv_fwd_weight(meta.co, wout, C, hidden, 1, train), residual=x)
        ctx.wdq = _conv_dgrad_weights(meta.cq, wqkv, 3 * hidden, C, 0, 1, train)[0]
        ctx.wdo = _conv_dgrad_weights(meta.co, wout, C, hidden, 0, 1, train)[0]
        saved = [x, g, xn, o, pos_bias, cs, sn, wqkv, wout, gamma, qkv]
        if F > 4:
            saved.append(lse)
        ctx.save_for_backward(*saved)
        ctx.cfg, ctx.gshape = (B, F, heads, D, eps), gamma.shape
        return y

    @staticmethod
    def backward(ctx, dy):
        saved = ctx.saved_tensors
        x, g, xn, o, pos_bias, cs, sn, wqkv, wout, gamma, qkv = saved[:11]
        lse = saved[11] if len(saved) > 11 else None
        B, F, heads, D, eps = ctx.cfg
        hidden = heads * D
        NI, H_, W_, C = x.shape
        dy = dy.contiguous()
        do = K.igemm(dy, ctx.wdo)
        dwout = _conv_wgrad(wout, o.view(NI, H_, W_, hidden), None, dy, 1) if ctx.needs_input_grad[3] else None
        dqkv, dbias = K.tattn_bwd(qkv.view(-1, 3 * hidden), pos_bias, cs, sn, o if F > 4 else None, lse,
                                  do.view(-1, hidden), B, F, H_ * W_, heads, D, D ** -0.5)
        dqkv4 = dqkv.view(NI, H_, W_, 3 * hidden)
        dxn, dwqkv = _qkv_backward(wqkv, ctx.wdq, xn, dqkv4, ctx.needs_input_grad[2])
        # + dy: the residual branch, added in the LN-backward epilogue
        if _direct_all(gamma):
            dx, _ = K.ln_bwd(x, g, dxn, dy, eps, into=gamma.grad.view(-1))
            _ready(gamma)
            dgamma = None
        else:
            dx, dg = K.ln_bwd(x, g, dxn, dy, eps)
            dgamma = dg.view(ctx.gshape)
        return dx, dgamma, dwqkv, dwout, dbias, None, None, None, None, None


class MidAttnBlockFn(_Fn):
    """Residual(PreNorm(EinopsToAndFrom('b c f h w' -> 'b f (h w) c', Attention))) (use_mid_attn=True,
    video_net.py:713-719) as one node: y = x + to_out(softmax attention over the h*w pixels of each frame of
    to_qkv(LN(x))).  No rotary embedding, no position bias; every frame (also F = 1) runs the full attention.
    args: x, gamma [1,C,1,1,1], wqkv [3*hidden, C], wout [C, hidden], meta(heads, dim_head, eps, cq, co)."""

    @staticmethod
    def forward(ctx, x, gamma, wqkv, wout, meta):
        x = x.contiguous()
        NI, H_, W_, C = x.shape
        heads, D, eps = meta.heads, meta.dim_head, meta.eps
        hidden, n = heads * D, H_ * W_
        g = gamma.reshape(-1)
        train = _train(ctx)
        xn = K.ln_fwd(x, g, eps)
        qkv = K.igemm(xn, _conv_fwd_weight(meta.cq, wqkv, 3 * hidden, C, 1, train))
        o, lse = K.mattn_fwd(qkv.view(-1, 3 * hidden), NI, n, heads, D, D ** -0.5)
        y = K.igemm(o.view(NI, H_, W_, hidden), _conv_fwd_weight(meta.co, wout, C, hidden, 1, train), residual=x)
        if train:
            ctx.wdq = _conv_dgrad_weights(meta.cq, wqkv, 3 * hidden, C, 0, 1, train)[0]
            ctx.wdo = _conv_dgrad_weights(meta.co, wout, C, hidden, 0, 1, train)[0]
            ctx.save_for_backward(x, g, xn, qkv, o, lse, wqkv, wout, gamma)
            ctx.cfg, ctx.gshape = (heads, D, eps), gamma.shape
        return y

    @staticmethod
    def backward(ctx, dy):
        x, g, xn, qkv, o, lse, wqkv, wout, gamma = ctx.saved_tensors
        heads, D, eps = ctx.cfg
        hidden = heads * D
        NI, H_, W_, C = x.shape
        dy = dy.contiguous()
        do = K.igemm(dy, ctx.wdo)
        dwout = _conv_wgrad(wout, o.view(NI, H_, W_, hidden), None, dy, 1) if ctx.needs_input_grad[3] else None
        dqkv = K.mattn_bwd(qkv.view(-1, 3 * hidden), o.view(-1, hidden), lse, do.view(-1, hidden), NI, H_ * W_, heads, D,
                           D ** -0.5)
        dxn, dwqkv = _qkv_backward(wqkv, ctx.wdq, xn, dqkv.view(NI, H_, W_, 3 * hidden), ctx.needs_input_grad[2])
        # + dy: the residual branch, added in the LN-backward epilogue
        if _direct_all(gamma):
            dx, _ = K.ln_bwd(x, g, dxn, dy, eps, into=gamma.grad.view(-1))
            _ready(gamma)
            dgamma = None
        else:
            dx, dg = K.ln_bwd(x, g, dxn, dy, eps)
            dgamma = dg.view(ctx.gshape)
        return dx, dgamma, dwqkv, dwout, None


class SpatialAttnBlockFn(_Fn):
    """Residual(PreNorm(SpatialLinearAttention)) (video_net.py:313-347) as one node.
    args: x, gamma, wqkv [3*hidden, C, 1, 1], wout [C, hidden, 1, 1], bout [C], meta."""

    @staticmethod
    def forward(ctx, x, gamma, wqkv, wout, bout, meta):
        x = x.contiguous()
        NI, H_, W_, C = x.shape
        heads, D, eps = meta.heads, meta.dim_head, meta.eps
        hidden = heads * D
        g = gamma.reshape(-1)
        train = _train(ctx)
        xn = K.ln_fwd(x, g, eps)
        qkv = K.igemm(xn, _conv_fwd_weight(meta.cq, wqkv, 3 * hidden, C, 1, train))
        o, ws = K.linattn_fwd(qkv.view(-1, 3 * hidden), NI, H_ * W_, heads, D, D ** -0.5)
        y = K.igemm(o.view(NI, H_, W_, hidden), _conv_fwd_weight(meta.co, wout, C, hidden, 1, train), bias=bout,
                    residual=x)
        ctx.wdq = _conv_dgrad_weights(meta.cq, wqkv, 3 * hidden, C, 0, 1, train)[0]
        ctx.wdo = _conv_dgrad_weights(meta.co, wout, C, hidden, 0, 1, train)[0]
        ctx.save_for_backward(x, g, xn, qkv, o, ws, wqkv, wout, gamma, bout)
        ctx.cfg, ctx.gshape = (heads, D, eps), gamma.shape
        return y

    @staticmethod
    def backward(ctx, dy):
        x, g, xn, qkv, o, ws, wqkv, wout, gamma, bout = ctx.saved_tensors
        heads, D, eps = ctx.cfg
        hidden = heads * D
        NI, H_, W_, C = x.shape
        dy = dy.contiguous()
        do = K.igemm(dy, ctx.wdo)
        need = ctx.needs_input_grad
        dwout = _conv_wgrad(wout, o.view(NI, H_, W_, hidden), None, dy, 1) if need[3] else None
        dbout = None
        if need[4] and _direct_all(bout):
            with _on_side(dy):
                K.colsum(dy, into=bout.grad)
            _ready(bout)
        elif need[4]:
            dbout = K.colsum(dy)
        dqkv = K.linattn_bwd(qkv.view(-1, 3 * hidden), ws, do.view(-1, hidden), NI, H_ * W_, heads, D, D ** -0.5)
        dqkv4 = dqkv.view(NI, H_, W_, 3 * hidden)
        dxn, dwqkv = _qkv_backward(wqkv, ctx.wdq, xn, dqkv4, need[2])
        if _direct_all(gamma):
            dx, _ = K.ln_bwd(x, g, dxn, dy, eps, into=gamma.grad.view(-1))
            _ready(gamma)
            dgamma = None
        else:
            dx, dg = K.ln_bwd(x, g, dxn, dy, eps)
            dgamma = dg.view(ctx.gshape)
        return dx, dgamma, dwqkv, dwout, dbout, None


# ------------------------------------------------------------------------------------------------
# network boundary
# ------------------------------------------------------------------------------------------------
class InputConvFn(_Fn):
    """cat([x, cond_map], dim=1) -> Conv3d(2, C, (1,k,k)) with frame broadcast folded in
    (video_net.py:808-815, model.py:110-121).  x/cond: fp32 [B,1,Fx,H,W]; out: fp16 [B*F,H,W,C].  `keep` (fp32 [B]
    of 0 / 1, or None): batch element b sees the null (all-zero) condition where keep[b] == 0, in the forward, the
    weight gradient and the condition's gradient (classifier-free guidance's condition dropout)."""

    @staticmethod
    def forward(ctx, x, cond, weight, bias, F: int, keep=None):
        """Tensor-core path: fp16 (hi, lo) im2col patches x [w | w | bias] through the tcgen05 implicit GEMM
        (kernels.input_patches / input_weight_pack); the patches are kept for the weight gradient."""
        shapes = (x.shape, cond.shape)
        x, cond = x.contiguous().float(), cond.contiguous().float()
        B, H, W = x.shape[0], x.shape[-2], x.shape[-1]
        ks = weight.shape[-1]
        patches = K.input_patches(x, cond, B, F, H, W, ks, keep=keep)
        out = K.igemm(patches, K.input_weight_pack(weight.detach(), bias.detach()))
        if _train(ctx):
            # the patches serve the weight gradient only
            need_w = ctx.needs_input_grad[2] or ctx.needs_input_grad[3]
            ctx.save_for_backward(patches if need_w else None, weight, bias, keep)
            ctx.dims = (B, F, H, W, x.numel() // (B * H * W), cond.numel() // (B * H * W), shapes)
        return out

    @staticmethod
    def backward(ctx, dy):
        patches, weight, bias, keep = ctx.saved_tensors
        B, F, H, W, f0, f1, shapes = ctx.dims
        ks = weight.shape[-1]
        dy = dy.contiguous()
        need_x, need_c = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        dx = dcond = None
        sink = _COND_GRAD_SINK[0] if need_c else None
        if sink is not None:  # scale * d cond added into the sink's buffer; autograd gets none
            K.input_conv_dgrad(dy, weight.detach(), B, F, H, W, ks, f0, f1, need_x=False, dcond_out=sink[0],
                               scale=sink[1], accumulate=True, keep=keep)
            need_c = False
        if need_x or need_c:
            dx, dcond = K.input_conv_dgrad(dy, weight.detach(), B, F, H, W, ks, f0, f1, need_x=need_x, need_cond=need_c,
                                           keep=keep)
            dx = None if dx is None else dx.view(shapes[0])
            dcond = None if dcond is None else dcond.view(shapes[1])
        if not (ctx.needs_input_grad[2] or ctx.needs_input_grad[3]):
            return dx, dcond, None, None, None, None
        nt = weight[0].numel()  # 2 * ks * ks
        full = K.wgrad(patches, dy)[:, 0, :]                       # fp32 [cout, KPAD]
        dw = (full[:, :nt] + full[:, nt:2 * nt]).view_as(weight)   # hi and lo column blocks see the same dy
        db = full[:, 2 * nt]                                       # the ones column: sum of dy
        if _direct_all(weight, bias):
            weight.grad.add_(dw)
            bias.grad.add_(db)
            _ready(weight, bias)
            return dx, dcond, None, None, None, None
        return dx, dcond, dw, db.contiguous(), None, None


class OutConvFn(_Fn):
    """Conv3d(C, 1, 1) evaluated on the centre frame (video_net.py:763 + model.py:129-130).
    a: fp16 [B*F, H, W, 64] -> fp32 [B, 1, H, W]."""

    @staticmethod
    def forward(ctx, a, weight, bias, B: int, F: int, mid: int):
        a = a.contiguous()
        H, W = a.shape[1], a.shape[2]
        ctx.save_for_backward(a, weight)
        ctx.dims = (B, F, H, W, mid)
        return K.out_conv_fwd(a, weight, bias, B, F, H, W, mid)

    @staticmethod
    def backward(ctx, deps):
        a, weight = ctx.saved_tensors
        B, F, H, W, mid = ctx.dims
        da, dw, db = K.out_conv_bwd(a, weight, deps.contiguous().float(), B, F, H, W, mid)
        return da, dw, db, None, None, None


class SmallLinearFn(_Fn):
    """fp32 y = act(x) W^T + b for the time-embedding MLP and FiLM projections
    (video_net.py:651-656, 238-241); act = SiLU on the input when `act_in`."""

    @staticmethod
    def forward(ctx, x, weight, bias, act_in: bool):
        x = x.contiguous()
        ctx.save_for_backward(x, weight, bias)
        ctx.act_in = act_in
        return K.small_linear_fwd(x, weight, bias, act_in)

    @staticmethod
    def backward(ctx, dy):
        x, weight, bias = ctx.saved_tensors
        if _direct_all(weight, bias):
            dx, _, _ = K.small_linear_bwd(x, weight, dy.contiguous(), ctx.act_in, ctx.needs_input_grad[0],
                                          into=(weight.grad, bias.grad))
            _ready(weight, bias)
            return dx, None, None, None
        dx, dW, db = K.small_linear_bwd(x, weight, dy.contiguous(), ctx.act_in, ctx.needs_input_grad[0])
        return dx, dW, db, None


_FILM_TABLES: dict = {}  # (parameter pointers, grad pointers or None) -> device descriptor table


def _film_table(Ws, bs, direct: bool):
    key = (tuple(w.data_ptr() for w in Ws), tuple(b.data_ptr() for b in bs),
           tuple(w.grad.data_ptr() for w in Ws) + tuple(b.grad.data_ptr() for b in bs) if direct else None)
    tab = _FILM_TABLES.get(key)
    if tab is None:
        if len(_FILM_TABLES) > 16:
            _FILM_TABLES.clear()
        tab = K.film_table(Ws, bs, [w.grad for w in Ws], [b.grad for b in bs]) if direct else K.film_table(Ws, bs)
        _FILM_TABLES[key] = tab
    return tab


class FilmAllFn(_Fn):
    """Every ResnetBlock's FiLM projection SiLU -> Linear(time_dim, 2*dim_out) (video_net.py:238-241) in one
    launch: they all read the same time embedding.  apply(temb, W_0, b_0, W_1, b_1, ...) -> tuple of [B, 2C_i].
    Backward: one launch for all weight / bias gradients and one for d temb (the sum over layers), instead of
    ~45 small launches plus autograd's adds."""

    @staticmethod
    def forward(ctx, temb, *wb):
        x = temb.contiguous()
        Ws, bs = list(wb[0::2]), list(wb[1::2])
        Ns = [w.shape[0] for w in Ws]
        outs = K.film_fwd(x, _film_table(Ws, bs, False), Ns)
        ctx.save_for_backward(x, *wb)
        ctx.Ns = Ns
        return tuple(outs)

    @staticmethod
    def backward(ctx, *dys):
        x, wb = ctx.saved_tensors[0], ctx.saved_tensors[1:]
        Ws, bs = list(wb[0::2]), list(wb[1::2])
        B = x.shape[0]
        dy = torch.cat([(d if d is not None else x.new_zeros(B, n)).reshape(-1) for d, n in zip(dys, ctx.Ns)])
        if _direct_all(*Ws, *bs):
            dx = K.film_bwd(x, _film_table(Ws, bs, True), dy, ctx.Ns, ctx.needs_input_grad[0], accumulate=True)
            _ready(*Ws, *bs)
            return (dx,) + (None,) * len(wb)
        dWs, dbs = [torch.empty_like(w) for w in Ws], [torch.empty_like(b) for b in bs]
        dx = K.film_bwd(x, K.film_table(Ws, bs, dWs, dbs), dy, ctx.Ns, ctx.needs_input_grad[0], accumulate=False)
        grads = [None] * len(wb)
        grads[0::2], grads[1::2] = dWs, dbs
        return (dx,) + tuple(grads)


class MseLossFn(_Fn):
    """F.mse_loss(eps, noise) (model.py:208) with the gradient 2*(eps-noise)/N produced on device."""

    @staticmethod
    def forward(ctx, eps, noise):
        loss, diff = K.mse_fwd(eps.contiguous(), noise.contiguous())
        ctx.save_for_backward(diff)
        return loss

    @staticmethod
    def backward(ctx, g):
        (diff,) = ctx.saved_tensors
        g = g.reshape(1).float().contiguous()
        deps = K.scale_by_scalar(diff, g, 2.0 / diff.numel()) if ctx.needs_input_grad[0] else None
        dnoise = K.scale_by_scalar(diff, g, -2.0 / diff.numel()) if ctx.needs_input_grad[1] else None
        return deps, dnoise


class DiffusionLossFn(_Fn):
    """sum_b w[t_b] * sum (pred - target)^2 / numel with target = c_n[t] noise + c_x[t] x0 (`tgt_coef` [T, 2], None for
    the eps target) and per-timestep weights `weight` [T] (None: uniform).  Differentiable in pred, noise and x0 (the
    target's share; q_sample's share comes through QSampleFn)."""

    @staticmethod
    def forward(ctx, pred, x0, noise, t, tgt_coef, weight):
        T = (tgt_coef if tgt_coef is not None else weight).shape[0]
        loss, diff = K.diffusion_loss_fwd(pred.contiguous(), _c(x0), noise.contiguous(), t.contiguous(), tgt_coef,
                                          weight, T)
        ctx.save_for_backward(diff, t, tgt_coef, weight)
        ctx.T = T
        return loss

    @staticmethod
    def backward(ctx, g):
        diff, t, tgt_coef, weight = ctx.saved_tensors
        need = ctx.needs_input_grad
        need_x0 = need[1] and tgt_coef is not None  # the eps target does not depend on x0
        if not (need[0] or need[2] or need_x0):
            return None, None, None, None, None, None
        g = g.reshape(1).float().contiguous()
        dpred, dnoise, dx0 = K.diffusion_loss_bwd(diff, t, tgt_coef, weight, g, 2.0 / diff.numel(), ctx.T, need[0],
                                                  need[2], need_x0)
        return dpred, dx0, dnoise, None, None, None


class QSampleFn(_Fn):
    """x_t = sqrt_ac[t] x0 + sqrt_1mac[t] noise (model.py:196-201), differentiable in x0 and noise."""

    @staticmethod
    def forward(ctx, x0, noise, t, sqrt_ac, sqrt_1mac):
        ctx.save_for_backward(t, sqrt_ac, sqrt_1mac)
        return K.q_sample(x0, noise, t, sqrt_ac, sqrt_1mac)

    @staticmethod
    def backward(ctx, g):
        t, sqrt_ac, sqrt_1mac = ctx.saved_tensors
        dx0, dnoise = K.q_sample_bwd(g.contiguous().float(), t, sqrt_ac, sqrt_1mac, ctx.needs_input_grad[0],
                                     ctx.needs_input_grad[1])
        return dx0, dnoise, None, None, None


# ------------------------------------------------------------------------------------------------
# layout helpers (network boundary and module-level drop-in calls only)
# ------------------------------------------------------------------------------------------------
def to_cl(x: torch.Tensor) -> Tuple[torch.Tensor, int, int]:
    """[B, C, F, H, W] (any float dtype) -> fp16 [B*F, H, W, C] contiguous, plus (B, F)."""
    B, C, F, H, W = x.shape
    return x.permute(0, 2, 3, 4, 1).reshape(B * F, H, W, C).to(H16).contiguous(), B, F


def from_cl(y: torch.Tensor, B: int, F: int) -> torch.Tensor:
    """fp16 [B*F, H, W, C] -> [B, C, F, H, W] view."""
    n, H, W, C = y.shape
    return y.view(B, F, H, W, C).permute(0, 4, 1, 2, 3)
