"""Thin tensor-level wrappers over the C ABI: validate, take data_ptr()/current stream, call.

Nothing here computes with PyTorch; torch only owns the memory and the stream.
"""
from __future__ import annotations

import ctypes
import numbers
from typing import Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import IgemmArgs

H16 = torch.float16


def _stream() -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _req_cuda(*ts: Optional[torch.Tensor]) -> None:
    for t in ts:
        if t is not None and not t.is_cuda:
            raise _lib.CesmError("cesm_emulator_b200 kernels need CUDA tensors (no CPU fallback)")
        if t is not None and not t.is_contiguous():
            raise _lib.CesmError("cesm_emulator_b200 kernels need contiguous tensors")


def _bytes_meta(*ts, kind=None):
    """Profiler annotation: algorithmic bytes = the tensors a kernel must read or write once."""
    if _lib.PROFILER is None:
        return None
    m = {"bytes": float(sum(t.numel() * t.element_size() for t in ts if t is not None))}
    if kind:
        m["kind"] = kind
    return m


TAPS_3x3 = [(dh, dw) for dh in (-1, 0, 1) for dw in (-1, 0, 1)]
TAPS_1x1 = [(0, 0)]


# ---- pre-zeroed scratch arena -------------------------------------------------------------------
class ZeroArena:
    """One persistent fp32 buffer from which the small accumulate-into scratch tensors of a training step
    (GroupNorm sums, linear-attention workspaces, bias-table gradients) are carved: `begin()` clears it
    with ONE memset and tells the library that scratch arrives zeroed (cesm_set_prezeroed_scratch), so
    the ~70 per-call memsets of a step disappear.  Addresses repeat every step (CUDA-graph safe)."""

    def __init__(self, device, floats: int = 4 << 20):
        self.buf = torch.zeros(floats, dtype=torch.float32, device=device)
        self.off = 0
        self.high = 0

    def begin(self) -> None:
        global _ARENA
        if self.high:
            self.buf[:self.high].zero_()
        self.off = 0
        _ARENA = self
        _lib.load().cesm_set_prezeroed_scratch(1)

    def end(self) -> None:
        global _ARENA
        _ARENA = None
        _lib.load().cesm_set_prezeroed_scratch(0)

    def take(self, shape) -> torch.Tensor:
        n = 1
        for d in shape:
            n *= int(d)
        start = self.off
        self.off = start + (n + 63) // 64 * 64  # 256-byte granules
        if self.off > self.buf.numel():
            # larger batch than the arena was sized for: fall back to an individually zeroed tensor (the
            # library's own memsets are off while the arena is active, so it MUST arrive zeroed)
            self.off = start
            return torch.zeros(tuple(shape), dtype=torch.float32, device=self.buf.device)
        self.high = max(self.high, self.off)
        return self.buf[start:start + n].view(*shape)


_ARENA: Optional[ZeroArena] = None


def zero_scratch(shape, device) -> torch.Tensor:
    """fp32 scratch for a kernel that accumulates into it: from the active arena (already zero) or a fresh
    uninitialised tensor (the library zeroes it)."""
    if _ARENA is not None:
        return _ARENA.take(tuple(shape))
    return torch.empty(tuple(shape), dtype=torch.float32, device=device)


def igemm(a0: torch.Tensor, wt: torch.Tensor, *, taps: Sequence[Tuple[int, int]] = TAPS_1x1,
          a1: Optional[torch.Tensor] = None, stride: int = 1,
          out: Optional[torch.Tensor] = None, out_hw: Optional[Tuple[int, int]] = None,
          out_place: Tuple[int, int, int, int] = (1, 1, 0, 0),
          bias: Optional[torch.Tensor] = None, residual: Optional[torch.Tensor] = None,
          gn_sums: Optional[torch.Tensor] = None, gn_frames: int = 1,
          ln_fold: Optional[Tuple[torch.Tensor, float]] = None):
    """out[n,oh,ow,:] = sum_t A[n, oh*stride+dh_t, ow*stride+dw_t, :] @ wt[:, t, :]^T (+bias)(+residual).

    a0/a1: fp16 [N,H,W,C]; wt: fp16 [cout, len(taps)*(C0+C1)]; out: fp16.  `out_hw` is the iterated output
    grid (defaults to H//stride, W//stride); `out_place` = (o_sh, o_sw, o_h0, o_w0) scatters the
    grid into a larger `out` tensor (transposed-conv phases).

    `ln_fold=(colsum, eps)`: a0 is x [.., 64], residual must be the same x, wt = W * gamma (per input channel) and
    colsum[co] = sum_ci wt[co, ci] (fp32, of the fp16 values): returns x + LayerNorm_channels(x) W^T with the row
    statistics computed in the epilogue (no LayerNorm kernel, no normalised tensor in HBM).
    """
    _req_cuda(a0, a1, wt, out, bias, residual)
    assert a0.dtype == H16 and wt.dtype == H16 and a0.dim() == 4
    n, h, w, c0 = a0.shape
    c1 = 0 if a1 is None else a1.shape[-1]
    cout = wt.shape[0]
    assert wt.shape[1] == len(taps) * (c0 + c1), (wt.shape, len(taps), c0, c1)
    oh, ow = out_hw if out_hw is not None else (h // stride, w // stride)
    o_sh, o_sw, o_h0, o_w0 = out_place
    if out is None:
        assert out_place == (1, 1, 0, 0)
        out = torch.empty((n, oh, ow, cout), dtype=H16, device=a0.device)
    assert out.dtype == H16, out.dtype
    args = IgemmArgs()
    args.a0, args.a1, args.c0, args.c1 = _ptr(a0), _ptr(a1), c0, c1
    args.n, args.h, args.w, args.stride = n, h, w, stride
    args.num_taps = len(taps)
    for i, (dh, dw) in enumerate(taps):
        args.tap_dh[i], args.tap_dw[i] = dh, dw
    args.wt, args.cout = _ptr(wt), cout
    args.oh, args.ow = oh, ow
    args.out, args.ldo = _ptr(out), out.shape[-1]
    args.out_h, args.out_w = out.shape[1], out.shape[2]
    args.o_sh, args.o_sw, args.o_h0, args.o_w0 = o_sh, o_sw, o_h0, o_w0
    args.bias = _ptr(bias)
    args.residual = _ptr(residual)
    args.ldr = 0 if residual is None else residual.shape[-1]
    if gn_sums is not None:
        # fused GroupNorm statistics: gn_sums fp32 [n / gn_frames, groups, 2] (zeroed by the call)
        assert gn_sums.dtype == torch.float32 and gn_sums.dim() == 3 and gn_sums.shape[0] * gn_frames == n
        args.gn_sums, args.gn_groups, args.gn_frames = _ptr(gn_sums), gn_sums.shape[1], gn_frames
    if ln_fold is not None:
        cs, eps = ln_fold
        assert residual is not None and residual.data_ptr() == a0.data_ptr() and c0 == 64 and cout == 64 and a1 is None
        assert cs.dtype == torch.float32 and cs.numel() == cout and cs.is_cuda
        args.ln_colsum, args.ln_eps = _ptr(cs), float(eps)
    if bias is not None:
        assert bias.dtype == torch.float32 and bias.numel() == cout
    if residual is not None:
        assert residual.dtype == H16 and residual.shape[:3] == out.shape[:3]
    meta = None
    if _lib.PROFILER is not None:
        rows = n * oh * ow
        ktot = len(taps) * (c0 + c1)
        meta = {"kind": f"{len(taps)}tap", "flops": 2.0 * rows * cout * ktot,
                "bytes": 2.0 * (rows * (c0 + c1) * stride * stride + rows * cout + cout * ktot)}
    _lib.call("cesm_igemm", ctypes.byref(args), _stream(), _meta=meta)
    return out


def wgrad(x0: torch.Tensor, dy: torch.Tensor, *, taps: Sequence[Tuple[int, int]] = TAPS_1x1,
          x1: Optional[torch.Tensor] = None, stride: int = 1, grid_hw: Optional[Tuple[int, int]] = None,
          dy_place: Tuple[int, int, int, int] = (1, 1, 0, 0), into: Optional[torch.Tensor] = None,
          layout: Optional[Tuple[int, int, Sequence[int]]] = None) -> torch.Tensor:
    """dw[co, t, ci] = sum_pixels dy[n,oh,ow,co] * X[n, oh*stride+dh_t, ow*stride+dw_t, ci]  -> fp32 [cout, T, C0+C1].

    With `into` (an fp32 tensor) and `layout` = (so, si, tap_off) the result is instead ACCUMULATED
    at into.flatten()[co*so + ci*si + tap_off[t]] (e.g. straight into a parameter's .grad)."""
    _req_cuda(x0, x1, dy)
    assert x0.dtype == H16 and dy.dtype == H16 and x0.dim() == 4 and dy.dim() == 4
    n, h, w, c0 = x0.shape
    c1 = 0 if x1 is None else x1.shape[-1]
    cout = dy.shape[-1]
    oh, ow = grid_hw if grid_hw is not None else (h // stride, w // stride)
    a = _lib.WgradArgs()
    if into is not None:
        assert layout is not None and into.dtype == torch.float32 and into.is_contiguous()
        dw_ = into
        a.dw_so, a.dw_si = int(layout[0]), int(layout[1])
        for i, o in enumerate(layout[2]):
            a.dw_tap_off[i] = int(o)
    else:
        dw_ = torch.empty((cout, len(taps), c0 + c1), dtype=torch.float32, device=x0.device)
    a.x0, a.x1, a.c0, a.c1 = _ptr(x0), _ptr(x1), c0, c1
    a.n, a.h, a.w, a.stride = n, h, w, stride
    a.num_taps = len(taps)
    for i, (dh, dw) in enumerate(taps):
        a.tap_dh[i], a.tap_dw[i] = dh, dw
    a.dy, a.cout, a.oh, a.ow = _ptr(dy), cout, oh, ow
    a.y_h, a.y_w = dy.shape[1], dy.shape[2]
    a.y_sh, a.y_sw, a.y_h0, a.y_w0 = dy_place
    a.dw = _ptr(dw_)
    meta = None
    if _lib.PROFILER is not None:
        rows = n * oh * ow
        meta = {"kind": f"{len(taps)}tap", "flops": 2.0 * rows * cout * len(taps) * (c0 + c1),
                "bytes": 2.0 * rows * (c0 + c1 + cout) + 4.0 * cout * len(taps) * (c0 + c1)}
    _lib.call("cesm_wgrad", ctypes.byref(a), _stream(), _meta=meta)
    return dw_


def qkv_bwd(dy: torch.Tensor, x: torch.Tensor, wt: torch.Tensor, dw_into: Optional[torch.Tensor] = None):
    """Fused data + weight gradient of a bias-free C=64 -> cout projection (cesm_qkv_bwd).
    dy: fp16 [..., cout]; x: fp16 [..., 64]; wt: fp16 [64, cout] (W^T).  -> (dx fp16 like x, dw fp32 [cout, 64]);
    with `dw_into` (fp32, contiguous [cout, 64] storage, e.g. a parameter's .grad) dW is ACCUMULATED there."""
    _req_cuda(dy, x, wt, dw_into)
    assert dy.dtype == H16 and x.dtype == H16 and wt.dtype == H16 and dy.is_contiguous() and x.is_contiguous()
    cout, cin = dy.shape[-1], x.shape[-1]
    rows = x.numel() // cin
    assert dy.numel() // cout == rows and tuple(wt.shape) == (cin, cout) and wt.is_contiguous()
    dx = torch.empty_like(x)
    if dw_into is None:
        dw = torch.zeros((cout, cin), dtype=torch.float32, device=x.device)
    else:
        assert dw_into.dtype == torch.float32 and dw_into.is_contiguous() and dw_into.numel() == cout * cin
        dw = dw_into
    meta = None
    if _lib.PROFILER is not None:
        meta = {"kind": "qkv", "flops": 4.0 * rows * cout * cin, "bytes": 2.0 * rows * (cout + 2 * cin)}
    _lib.call("cesm_qkv_bwd", _ptr(dy), _ptr(x), _ptr(wt), _ptr(dx), _ptr(dw), cin, rows, cin, cout, _stream(), _meta=meta)
    return dx, dw


def _tap_array(offs: Sequence[int]):
    arr = (ctypes.c_int32 * _lib.CESM_MAX_TAPS)()
    for i, o in enumerate(offs):
        arr[i] = int(o)
    return arr


def pack_weight(src: torch.Tensor, O: int, T: int, I: int, so: int, si: int, tap_off: Sequence[int],
                out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """dst[o][t][i] (fp16) = src.flatten()[o*so + i*si + tap_off[t]]."""
    _req_cuda(src)
    assert src.dtype == torch.float32
    if out is None:
        out = torch.empty((O, T * I), dtype=H16, device=src.device)
    _lib.call("cesm_pack_weight", _ptr(src), _ptr(out), O, T, I, so, si, _tap_array(tap_off), _stream())
    return out


def unpack_wgrad(src: torch.Tensor, dst: torch.Tensor, O: int, T: int, I: int, so: int, si: int,
                 tap_off: Sequence[int], accumulate: bool = False) -> torch.Tensor:
    _req_cuda(src, dst)
    assert src.dtype == torch.float32 and dst.dtype == torch.float32
    _lib.call("cesm_unpack_wgrad", _ptr(src), _ptr(dst), O, T, I, so, si, _tap_array(tap_off), int(accumulate), _stream())
    return dst


OPT_STATE_FLOATS = 16  # CESM_OPT_STATE_FLOATS; layout in include/cesm_b200.h
OPT_STEP, OPT_NORM, OPT_SCALE, OPT_TRACKER, OPT_FOUND_INF, OPT_SKIPPED, OPT_LR, OPT_WD, OPT_INTERVAL = range(9)


def adamw_step(p: torch.Tensor, g: torch.Tensor, m: torch.Tensor, v: torch.Tensor, partials: torch.Tensor,
               state: torch.Tensor, beta1: float, beta2: float, eps: float, max_norm: Optional[float]) -> None:
    """Loss-scale removal + inf check + global-norm clip + AdamW over flat fp32 buffers, then the scaler update
    (see cesm_adamw_step in include/cesm_b200.h; lr, weight decay and the loss scale live in `state`)."""
    _req_cuda(p, g, m, v, partials, state)
    for t in (p, g, m, v, partials, state):
        assert t.dtype == torch.float32 and t.is_contiguous()
    assert p.numel() == g.numel() == m.numel() == v.numel() and state.numel() >= OPT_STATE_FLOATS
    assert partials.numel() >= _lib.load().cesm_adamw_partials()
    _lib.call("cesm_adamw_step", _ptr(p), _ptr(g), _ptr(m), _ptr(v), p.numel(), _ptr(partials), _ptr(state),
              float(beta1), float(beta2), float(eps), float(max_norm) if max_norm is not None else 0.0, _stream(),
              _meta={"bytes": 28.0 * p.numel()})


def adamw_ema_step(p: torch.Tensor, g: torch.Tensor, m: torch.Tensor, v: torch.Tensor, ema: torch.Tensor,
                   partials: torch.Tensor, state: torch.Tensor, beta1: float, beta2: float, eps: float,
                   max_norm: Optional[float], ema_decay: float, ema_start: int) -> None:
    """adamw_step plus the exponential moving average `ema` of the updated parameters in the same pass (see
    cesm_adamw_ema_step in include/cesm_b200.h): a copy while the step count is <= ema_start, then
    ema += (1 - ema_decay) (p - ema)."""
    _req_cuda(p, g, m, v, ema, partials, state)
    for t in (p, g, m, v, ema, partials, state):
        assert t.dtype == torch.float32 and t.is_contiguous()
    assert p.numel() == g.numel() == m.numel() == v.numel() == ema.numel() and state.numel() >= OPT_STATE_FLOATS
    assert partials.numel() >= _lib.load().cesm_adamw_partials()
    _lib.call("cesm_adamw_ema_step", _ptr(p), _ptr(g), _ptr(m), _ptr(v), _ptr(ema), p.numel(), _ptr(partials),
              _ptr(state), float(beta1), float(beta2), float(eps), float(max_norm) if max_norm is not None else 0.0,
              float(ema_decay), int(ema_start), _stream(), _meta={"bytes": 36.0 * p.numel()})


def colsum(x: torch.Tensor, into: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Column sums of fp16 x[..., C]; with `into` (fp32 [C]) the sums are ADDED to it."""
    _req_cuda(x, into)
    C = x.shape[-1]
    out = torch.empty(C, dtype=torch.float32, device=x.device) if into is None else into
    _lib.call("cesm_colsum", _ptr(x), _ptr(out), x.numel() // C, C, int(into is not None), _stream())
    return out


# ---- GroupNorm / LayerNorm ----------------------------------------------------------------------
def gn_stats(x: torch.Tensor, B: int, G: int) -> torch.Tensor:
    _req_cuda(x)
    C = x.shape[-1]
    P = x.numel() // (B * C)
    sums = torch.empty((B, G, 2), dtype=torch.float32, device=x.device)
    _lib.call("cesm_gn_stats", _ptr(x), _ptr(sums), B, P, C, G, _stream(), _meta=_bytes_meta(x))
    return sums


def gn_apply_fwd(x, sums, gamma, beta, film, residual, B: int, G: int, eps: float) -> torch.Tensor:
    _req_cuda(x, sums, gamma, beta, film, residual)
    C = x.shape[-1]
    P = x.numel() // (B * C)
    out = torch.empty_like(x)
    _lib.call("cesm_gn_apply_fwd", _ptr(x), _ptr(sums), _ptr(gamma), _ptr(beta), _ptr(film), _ptr(residual), _ptr(out),
              B, P, C, G, eps, _stream(), _meta=_bytes_meta(x, residual, out))
    return out


def gn_bwd(x, dout, sums, gamma, beta, film, B: int, G: int, eps: float, conv_bias_grad: bool = False,
           into=None):
    """-> (dx, dgamma, dbeta, dfilm or None[, dconv_bias]).  `dconv_bias` is sum_pixels dx per
    channel, i.e. the bias gradient of the convolution that produced x, obtained from the same
    per-channel sums (no extra pass over dx)."""
    _req_cuda(x, dout, sums, gamma, beta, film)
    C = x.shape[-1]
    P = x.numel() // (B * C)
    dev = x.device
    csum = zero_scratch((B, C, 3), dev)
    dx = torch.empty_like(x)
    if into is not None:  # (dgamma, dbeta, dconv_bias) buffers to ACCUMULATE into (parameter .grad views)
        dgamma, dbeta, dcb = into
    else:
        dgamma = torch.empty(C, dtype=torch.float32, device=dev)
        dbeta = torch.empty(C, dtype=torch.float32, device=dev)
        dcb = torch.empty(C, dtype=torch.float32, device=dev) if conv_bias_grad else None
    dfilm = torch.empty((B, 2 * C), dtype=torch.float32, device=dev) if film is not None else None
    _lib.call("cesm_gn_bwd", _ptr(x), _ptr(dout), _ptr(sums), _ptr(gamma), _ptr(beta), _ptr(film), _ptr(csum), _ptr(dx),
              _ptr(dgamma), _ptr(dbeta), _ptr(dfilm), _ptr(dcb), B, P, C, G, eps, int(into is not None), _stream(),
              _meta=_bytes_meta(x, dout, x, dout, dx))
    if conv_bias_grad:
        return dx, dgamma, dbeta, dfilm, dcb
    return dx, dgamma, dbeta, dfilm


def ln_fwd(x: torch.Tensor, gamma: torch.Tensor, eps: float) -> torch.Tensor:
    _req_cuda(x, gamma)
    C = x.shape[-1]
    out = torch.empty_like(x)
    _lib.call("cesm_ln_fwd", _ptr(x), _ptr(gamma), _ptr(out), x.numel() // C, C, eps, _stream(),
              _meta=_bytes_meta(x, out))
    return out


def ln_bwd(x, gamma, dy, dres, eps: float, into: Optional[torch.Tensor] = None):
    """`into`: fp32 [C] buffer the gain gradient is ADDED to (else a fresh tensor is returned)."""
    _req_cuda(x, gamma, dy, dres, into)
    C = x.shape[-1]
    dx = torch.empty_like(x)
    dgamma = torch.empty(C, dtype=torch.float32, device=x.device) if into is None else into
    _lib.call("cesm_ln_bwd", _ptr(x), _ptr(gamma), _ptr(dy), _ptr(dres), _ptr(dx), _ptr(dgamma), x.numel() // C, C, eps,
              int(into is not None), _stream(), _meta=_bytes_meta(x, dy, dres, dx))
    return dx, dgamma


# ---- attention cores ----------------------------------------------------------------------------
LONG_WINDOW_MAX = 128  # cesm_tattn_long_max_frames(): frames of one pixel column that fit in shared memory


def _bias_to_diag(bias: torch.Tensor) -> torch.Tensor:
    """[H, F, F] Toeplitz relative-position bias (video_net.py:302-310: a function of key - query) -> [H, 2F-1] with
    diag[h][d + F - 1] = bias[h][i][i + d]: first column (d < 0, reversed) then first row (d >= 0)."""
    return torch.cat([bias[:, 1:, 0].flip(1), bias[:, 0, :]], dim=1).contiguous()


def _diag_to_bias_grad(ddiag: torch.Tensor, F: int) -> torch.Tensor:
    """The per-diagonal bias gradient as an [H, F, F] tensor with each diagonal's sum placed on its first element:
    every consumer of d(bias) here sums over a diagonal anyway (the bucket of an entry depends on key - query only),
    so the embedding-table gradient is the same as with the element-wise gradient."""
    H = ddiag.shape[0]
    g = torch.zeros((H, F, F), dtype=ddiag.dtype, device=ddiag.device)
    g[:, 0, :] = ddiag[:, F - 1:]
    g[:, 1:, 0] = ddiag[:, :F - 1].flip(1)
    return g


def tattn_fwd(qkv, bias, cs, sn, B: int, F: int, HW: int, H: int, D: int, scale: float):
    """F <= 4: register-resident kernel, `bias` may be any [H, F, F].  F > 4: the shared-memory / tensor-core flash
    kernel (cesm_tattn_long_fwd), which takes the bias by diagonal: `bias` must be Toeplitz (RelativePositionBias)."""
    _req_cuda(qkv, bias, cs, sn)
    rows = B * F * HW
    out = torch.empty((rows, H * D), dtype=H16, device=qkv.device)
    if 4 < F <= LONG_WINDOW_MAX:
        lse = torch.empty((rows, H), dtype=torch.float32, device=qkv.device)
        _lib.call("cesm_tattn_long_fwd", _ptr(qkv), _ptr(_bias_to_diag(bias)), _ptr(cs), _ptr(sn), _ptr(out), _ptr(lse),
                  B, F, HW, H, D, scale, _stream(),
                  _meta={"kind": f"F{F}", "bytes": float(qkv.numel() * 2 + out.numel() * 2),
                         "flops": 4.0 * rows * H * F * D * 2})
        return out, lse
    # F <= 4: the backward recomputes the softmax, so no log-sum-exp is kept.  F > 128: the streaming kernel.
    lse = torch.empty((rows, H), dtype=torch.float32, device=qkv.device) if F > 4 else None
    _lib.call("cesm_tattn_fwd", _ptr(qkv), _ptr(bias), _ptr(cs), _ptr(sn), _ptr(out), _ptr(lse), B, F, HW, H, D, scale,
              _stream(), _meta=_bytes_meta(qkv, out))
    return out, lse


def tattn_bwd(qkv, bias, cs, sn, out, lse, dout, B: int, F: int, HW: int, H: int, D: int, scale: float):
    _req_cuda(qkv, bias, cs, sn, out, lse, dout)
    dqkv = torch.empty_like(qkv)
    if 4 < F <= LONG_WINDOW_MAX:
        ddiag = zero_scratch((H, 2 * F - 1), qkv.device)
        _lib.call("cesm_tattn_long_bwd", _ptr(qkv), _ptr(_bias_to_diag(bias)), _ptr(cs), _ptr(sn), _ptr(out), _ptr(lse),
                  _ptr(dout), _ptr(dqkv), _ptr(ddiag), B, F, HW, H, D, scale, _stream(),
                  _meta={"kind": f"F{F}", "bytes": float(qkv.numel() * 4 + dout.numel() * 4),
                         "flops": 14.0 * B * F * HW * H * F * D * 2})
        return dqkv, _diag_to_bias_grad(ddiag, F)
    dbias = zero_scratch((H, F, F), qkv.device)
    _lib.call("cesm_tattn_bwd", _ptr(qkv), _ptr(bias), _ptr(cs), _ptr(sn), _ptr(out), _ptr(lse), _ptr(dout), _ptr(dqkv),
              _ptr(dbias), B, F, HW, H, D, scale, _stream(), _meta=_bytes_meta(qkv, dout, dqkv))
    return dqkv, dbias


def tattn_proj_ok(C: int, F: int, HW: int, H: int, D: int) -> bool:
    """Shapes the fused projection + attention forward (csrc/tattn_proj.cu) takes."""
    return C == 64 and 1 <= F <= 3 and HW % 16 == 0 and H == 8 and D == 32


def tattn_proj_fwd(xn, wqkv_packed, bias, cs, sn, B: int, F: int, HW: int, H: int, D: int, scale: float):
    """o = attention(xn Wq^T, xn Wk^T, xn Wv^T) for F <= 3 frames without materialising q|k|v.
    xn: fp16 [B*F*HW, 64]; wqkv_packed: fp16 [768, 64] -> fp16 [B*F*HW, 256]."""
    _req_cuda(xn, wqkv_packed, bias, cs, sn)
    assert xn.dtype == H16 and wqkv_packed.dtype == H16 and tuple(wqkv_packed.shape) == (3 * H * D, 64)
    rows = B * F * HW
    out = torch.empty((rows, H * D), dtype=H16, device=xn.device)
    _lib.call("cesm_tattn_proj_fwd", _ptr(xn), _ptr(wqkv_packed), _ptr(bias), _ptr(cs), _ptr(sn), _ptr(out), B, F, HW, H, D,
              64, scale, _stream(),
              _meta={"kind": "fused", "flops": 2.0 * rows * 64 * 3 * H * D, "bytes": float(rows * (64 + H * D) * 2)})
    return out


def mattn_fwd(qkv, NI: int, n: int, H: int, D: int, scale: float):
    """Full softmax attention over the n pixels of each of NI images (use_mid_attn's bottleneck block).
    qkv: fp16 [NI*n, 3*H*D] -> (out fp16 [NI*n, H*D], lse fp32 [NI*n, H])."""
    _req_cuda(qkv)
    assert qkv.dtype == H16 and qkv.shape == (NI * n, 3 * H * D), (tuple(qkv.shape), NI, n, H, D)
    out = torch.empty((NI * n, H * D), dtype=H16, device=qkv.device)
    lse = torch.empty((NI * n, H), dtype=torch.float32, device=qkv.device)
    _lib.call("cesm_mattn_fwd", _ptr(qkv), _ptr(out), _ptr(lse), NI, n, H, D, scale, _stream(),
              _meta={"kind": "fwd", "flops": 4.0 * NI * H * n * n * D, "bytes": float(qkv.numel() * 2 + out.numel() * 2)})
    return out, lse


def mattn_bwd(qkv, out, lse, dout, NI: int, n: int, H: int, D: int, scale: float):
    """-> dqkv fp16 [NI*n, 3*H*D] (q, k and v gradients; no accumulation, deterministic)."""
    _req_cuda(qkv, out, lse, dout)
    assert qkv.dtype == H16 and out.dtype == H16 and dout.dtype == H16 and lse.dtype == torch.float32
    assert qkv.shape == (NI * n, 3 * H * D) and out.shape == dout.shape == (NI * n, H * D) and lse.numel() == NI * n * H
    dqkv = torch.empty_like(qkv)
    delta = torch.empty((NI * n, H), dtype=torch.float32, device=qkv.device)
    # S and P recomputed twice (dQ pass, dK/dV pass), dP twice, dQ, dK, dV once: 4 + 4 + 2 + 2 + 2 = 14 n^2 D per head
    _lib.call("cesm_mattn_bwd", _ptr(qkv), _ptr(out), _ptr(lse), _ptr(dout), _ptr(dqkv), _ptr(delta), NI, n, H, D, scale,
              _stream(), _meta={"kind": "bwd", "flops": 14.0 * NI * H * n * n * D,
                                "bytes": float(qkv.numel() * 4 + out.numel() * 2 + dout.numel() * 2)})
    return dqkv


def linattn_fwd(qkv, NI: int, n: int, H: int, D: int, scale: float):
    """-> (out fp16 [NI*n, H*D], ws fp32 workspace kept for the backward)."""
    _req_cuda(qkv)
    dev = qkv.device
    ws = zero_scratch((_lib.load().cesm_linattn_ws_floats(NI, H),), dev)
    out = torch.empty((NI * n, H * D), dtype=H16, device=dev)
    _lib.call("cesm_linattn_fwd", _ptr(qkv), _ptr(ws), _ptr(out), NI, n, H, D, scale, _stream(),
              _meta=_bytes_meta(qkv, out))
    return out, ws


def linattn_bwd(qkv, ws, dout, NI: int, n: int, H: int, D: int, scale: float):
    _req_cuda(qkv, ws, dout)
    scratch = zero_scratch((NI * H * D * D + NI * H * D,), qkv.device)
    dqkv = torch.empty_like(qkv)
    _lib.call("cesm_linattn_bwd", _ptr(qkv), _ptr(ws), _ptr(dout), _ptr(scratch), _ptr(dqkv), NI, n, H, D, scale,
              _stream(), _meta=_bytes_meta(qkv, dout, dqkv))
    return dqkv


# ---- boundary convs -----------------------------------------------------------------------------
def gather_windows(cond, tgt, plan, cond_out, x0_out) -> None:
    """cond, tgt: fp32 [T, M, H, W] on the device; plan: int32 [B, 6] on the device (see cesm_gather_windows);
    cond_out: fp32 [B, 1, K, h, w]; x0_out: fp32 [B, 1, h, w] -- both written in place."""
    _req_cuda(cond, tgt, plan, cond_out, x0_out)
    assert cond.dtype == tgt.dtype == cond_out.dtype == x0_out.dtype == torch.float32 and plan.dtype == torch.int32
    assert cond.is_contiguous() and tgt.is_contiguous() and cond_out.is_contiguous() and x0_out.is_contiguous()
    T, M, H, W = cond.shape
    B, _, K, h, w = cond_out.shape
    assert plan.shape == (B, 6) and plan.is_contiguous() and x0_out.shape == (B, 1, h, w) and tgt.shape == cond.shape
    _lib.call("cesm_gather_windows", _ptr(cond), _ptr(tgt), _ptr(plan), _ptr(cond_out), _ptr(x0_out), B, T, M, H, W, K,
              h, w, _stream())


INPUT_KPAD = 256  # columns of the input-conv patch matrix: 2 planes x 49 taps x (hi, lo) + 2 ones + padding


def input_patches(in0, in1, B: int, F: int, H: int, W: int, ks: int) -> torch.Tensor:
    """im2col of the two fp32 input planes (frame broadcast folded in) -> fp16 [B*F, H, W, INPUT_KPAD]."""
    _req_cuda(in0, in1)
    f0, f1 = in0.numel() // (B * H * W), in1.numel() // (B * H * W)
    out = torch.empty((B * F, H, W, INPUT_KPAD), dtype=H16, device=in0.device)
    _lib.call("cesm_input_patches", _ptr(in0), _ptr(in1), f0, f1, _ptr(out), B, F, H, W, ks, INPUT_KPAD, _stream(),
              _meta=_bytes_meta(out))
    return out


def input_weight_pack(w, bias, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """[cout, 2, 1, ks, ks] fp32 + bias -> fp16 [cout, INPUT_KPAD] operand matching `input_patches`."""
    _req_cuda(w, bias)
    cout, ks = w.shape[0], w.shape[-1]
    if out is None:
        out = torch.empty((cout, INPUT_KPAD), dtype=H16, device=w.device)
    _lib.call("cesm_input_weight_pack", _ptr(w), _ptr(bias), _ptr(out), cout, ks, INPUT_KPAD, _stream())
    return out


def input_conv_fwd(in0, in1, w, bias, B: int, F: int, H: int, W: int, ks: int):
    _req_cuda(in0, in1, w, bias)
    cout = w.shape[0]
    f0, f1 = in0.numel() // (B * H * W), in1.numel() // (B * H * W)
    out = torch.empty((B * F, H, W, cout), dtype=H16, device=in0.device)
    _lib.call("cesm_input_conv_fwd", _ptr(in0), _ptr(in1), f0, f1, _ptr(w), _ptr(bias), _ptr(out), B, F, H, W, ks, cout,
              _stream())
    return out


def input_conv_wgrad(in0, in1, dy, B: int, F: int, H: int, W: int, ks: int):
    _req_cuda(in0, in1, dy)
    cout = dy.shape[-1]
    f0, f1 = in0.numel() // (B * H * W), in1.numel() // (B * H * W)
    dw = torch.empty((cout, 2, 1, ks, ks), dtype=torch.float32, device=dy.device)
    db = torch.empty(cout, dtype=torch.float32, device=dy.device)
    _lib.call("cesm_input_conv_wgrad", _ptr(in0), _ptr(in1), f0, f1, _ptr(dy), _ptr(dw), _ptr(db), B, F, H, W, ks, cout,
              _stream())
    return dw, db


def input_conv_dgrad(dy, w, B: int, F: int, H: int, W: int, ks: int, f0: int, f1: int, *, need_x: bool = True,
                     need_cond: bool = True, dx_out: Optional[torch.Tensor] = None,
                     dcond_out: Optional[torch.Tensor] = None, scale: float = 1.0, accumulate: bool = False):
    """Data gradient of the input convolution (cesm_input_conv_dgrad): dy fp16 [B*F, H, W, C] and the fp32 weight
    [C, 2, 1, ks, ks] -> (d_x fp32 [B, 1, f0, H, W] or None, d_cond fp32 [B, 1, f1, H, W] or None).  A side with one
    frame while F > 1 gets the sum over the F frames (the forward's broadcast).  Each result is scale * grad, written
    into `dx_out` / `dcond_out` when given -- or, with `accumulate`, added to them."""
    _req_cuda(dy, w, dx_out, dcond_out)
    assert dy.dtype == H16 and tuple(dy.shape[:3]) == (B * F, H, W) and w.dtype == torch.float32
    cout = dy.shape[-1]
    assert tuple(w.shape) == (cout, 2, 1, ks, ks), tuple(w.shape)
    assert need_x or need_cond
    outs = []
    for need, given, fp in ((need_x, dx_out, f0), (need_cond, dcond_out, f1)):
        if not need:
            outs.append(None)
            continue
        if given is None:
            assert not accumulate, "accumulate needs the output buffers"
            given = torch.empty((B, 1, fp, H, W), dtype=torch.float32, device=dy.device)
        assert given.dtype == torch.float32 and given.numel() == B * fp * H * W, (given.dtype, tuple(given.shape))
        outs.append(given)
    meta = None
    if _lib.PROFILER is not None:
        meta = {"flops": 2.0 * B * F * H * W * cout * ks * ks * (int(need_x) + int(need_cond)),
                "bytes": float(dy.numel() * 2 + sum(o.numel() * 4 for o in outs if o is not None))}
    _lib.call("cesm_input_conv_dgrad", _ptr(dy), _ptr(w), _ptr(outs[0]), _ptr(outs[1]), f0, f1, B, F, H, W, ks, cout,
              float(scale), int(accumulate), _stream(), _meta=meta)
    return outs[0], outs[1]


def out_conv_fwd(a, w, bias, B: int, F: int, H: int, W: int, mid: Optional[int] = None):
    _req_cuda(a, w, bias)
    mid = F // 2 if mid is None else mid
    eps = torch.empty((B, 1, H, W), dtype=torch.float32, device=a.device)
    _lib.call("cesm_out_conv_fwd", _ptr(a), _ptr(w), _ptr(bias), _ptr(eps), B, F, mid, H * W, a.shape[-1], _stream())
    return eps


def out_conv_bwd(a, w, deps, B: int, F: int, H: int, W: int, mid: Optional[int] = None):
    _req_cuda(a, w, deps)
    mid = F // 2 if mid is None else mid
    da = torch.empty_like(a)
    dw = torch.empty_like(w)
    db = torch.empty(1, dtype=torch.float32, device=a.device)
    _lib.call("cesm_out_conv_bwd", _ptr(a), _ptr(w), _ptr(deps), _ptr(da), _ptr(dw), _ptr(db), B, F, mid, H * W,
              a.shape[-1], _stream())
    return da, dw, db


# ---- time embedding / small linears -------------------------------------------------------------
def sinusoidal(t: torch.Tensor, dim: int) -> torch.Tensor:
    _req_cuda(t)
    assert t.dtype == torch.int64
    out = torch.empty((t.numel(), dim), dtype=torch.float32, device=t.device)
    _lib.call("cesm_sinusoidal", _ptr(t), _ptr(out), t.numel(), dim, _stream())
    return out


def small_linear_fwd(x, W, bias, act_silu_in: bool):
    _req_cuda(x, W, bias)
    B, K = x.shape
    N = W.shape[0]
    y = torch.empty((B, N), dtype=torch.float32, device=x.device)
    _lib.call("cesm_small_linear_fwd", _ptr(x), _ptr(W), _ptr(bias), _ptr(y), B, K, N, int(act_silu_in), _stream())
    return y


def small_linear_bwd(x, W, dy, act_silu_in: bool, need_dx: bool, into=None):
    """`into`: (dW, db) buffers to ACCUMULATE into (parameter .grad views)."""
    _req_cuda(x, W, dy)
    B, K = x.shape
    N = W.shape[0]
    if into is not None:
        dW, db = into
    else:
        dW = torch.empty_like(W)
        db = torch.empty(N, dtype=torch.float32, device=x.device)
    dx = torch.empty_like(x) if need_dx else None
    _lib.call("cesm_small_linear_bwd", _ptr(x), _ptr(W), _ptr(dy), _ptr(dx), _ptr(dW), _ptr(db), B, K, N,
              int(act_silu_in), int(into is not None), _stream())
    return dx, dW, db


# ---- all FiLM projections of a pass at once -----------------------------------------------------
def film_table(Ws, bs, dWs=None, dbs=None) -> torch.Tensor:
    """Device table of `cesm_film_desc` for these layers (static pointers only: cache it)."""
    n = len(Ws)
    arr = (_lib.FilmDesc * n)()
    n0 = 0
    for i, d in enumerate(arr):
        d.W, d.bias = Ws[i].data_ptr(), bs[i].data_ptr()
        d.dW = dWs[i].data_ptr() if dWs is not None else 0
        d.db = dbs[i].data_ptr() if dbs is not None else 0
        d.N, d.n0 = Ws[i].shape[0], n0
        n0 += Ws[i].shape[0]
    return torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).to(Ws[0].device)


def film_fwd(x: torch.Tensor, table: torch.Tensor, Ns) -> list:
    """-> per-layer fp32 [B, N_i] views of one packed output buffer."""
    _req_cuda(x, table)
    B, K = x.shape
    n_total = int(sum(Ns))
    y = torch.empty(B * n_total, dtype=torch.float32, device=x.device)
    _lib.call("cesm_film_fwd", _ptr(x), _ptr(table), _ptr(y), len(Ns), n_total, B, K, _stream())
    outs, n0 = [], 0
    for N in Ns:
        outs.append(y[B * n0:B * (n0 + N)].view(B, N))
        n0 += N
    return outs


def film_bwd(x: torch.Tensor, table: torch.Tensor, dy_packed: torch.Tensor, Ns, need_dx: bool, accumulate: bool):
    _req_cuda(x, table, dy_packed)
    B, K = x.shape
    n_total = int(sum(Ns))
    assert dy_packed.numel() == B * n_total and dy_packed.dtype == torch.float32 and dy_packed.is_contiguous()
    dx = zero_scratch(x.shape, x.device) if need_dx else None  # the per-layer blocks add into it
    _lib.call("cesm_film_bwd", _ptr(x), _ptr(table), _ptr(dy_packed), len(Ns), n_total, _ptr(dx), B, K, int(accumulate),
              _stream())
    return dx


# ---- DDPM ---------------------------------------------------------------------------------------
def q_sample(x0, noise, t, sqrt_ac, sqrt_1mac):
    _req_cuda(x0, noise, t, sqrt_ac, sqrt_1mac)
    xt = torch.empty_like(x0)
    B = x0.shape[0]
    _lib.call("cesm_q_sample", _ptr(x0), _ptr(noise), _ptr(t), _ptr(sqrt_ac), _ptr(sqrt_1mac), _ptr(xt), B,
              x0.numel() // B, _stream())
    return xt


def q_sample_bwd(g, t, sqrt_ac, sqrt_1mac, need_x0: bool = True, need_noise: bool = True):
    """Backward of q_sample: (dx0 = sqrt_ac[t] g or None, dnoise = sqrt_1mac[t] g or None) per sample."""
    _req_cuda(g, t, sqrt_ac, sqrt_1mac)
    assert g.dtype == torch.float32 and t.dtype == torch.int64 and (need_x0 or need_noise)
    B = g.shape[0]
    assert t.shape == (B,), (tuple(t.shape), B)
    dx0 = torch.empty_like(g) if need_x0 else None
    dnoise = torch.empty_like(g) if need_noise else None
    _lib.call("cesm_q_sample_bwd", _ptr(g), _ptr(t), _ptr(sqrt_ac), _ptr(sqrt_1mac), _ptr(dx0), _ptr(dnoise), B,
              g.numel() // B, _stream())
    return dx0, dnoise


def mse_fwd(eps, noise):
    _req_cuda(eps, noise)
    diff = torch.empty_like(eps)
    loss = torch.empty((), dtype=torch.float32, device=eps.device)
    _lib.call("cesm_mse_fwd", _ptr(eps), _ptr(noise), _ptr(diff), _ptr(loss), eps.numel(), _stream())
    return loss, diff


def _loss_tables(t, tgt_coef, weight, T: int, B: int) -> None:
    assert t.dtype == torch.int64 and t.shape == (B,), (t.dtype, tuple(t.shape), B)
    assert tgt_coef is None or (tgt_coef.dtype == torch.float32 and tgt_coef.shape == (T, 2) and tgt_coef.is_contiguous())
    assert weight is None or (weight.dtype == torch.float32 and weight.shape == (T,) and weight.is_contiguous())


def diffusion_loss_fwd(pred, x0, noise, t, tgt_coef, weight, T: int):
    """Per sample b: target = c_n[t_b] noise + c_x[t_b] x0 (rows of the fp32 [T, 2] `tgt_coef`; None is the eps target
    and x0 is not read), diff = pred - target, loss = sum_b weight[t_b] sum diff^2 / numel (None weight: 1).
    A t outside [0, T) gives NaN.  -> (0-dim loss, diff)."""
    _req_cuda(pred, x0, noise, t, tgt_coef, weight)
    B = pred.shape[0]
    _loss_tables(t, tgt_coef, weight, T, B)
    assert pred.dtype == noise.dtype == torch.float32 and noise.shape == pred.shape
    assert tgt_coef is None or (x0.dtype == torch.float32 and x0.shape == pred.shape)
    diff = torch.empty_like(pred)
    loss = torch.empty((), dtype=torch.float32, device=pred.device)
    _lib.call("cesm_diffusion_loss_fwd", _ptr(pred), _ptr(x0), _ptr(noise), _ptr(t), _ptr(tgt_coef), _ptr(weight),
              _ptr(diff), _ptr(loss), B, pred.numel() // B, T, _stream())
    return loss, diff


def diffusion_loss_bwd(diff, t, tgt_coef, weight, gscale, factor: float, T: int, need_pred: bool = True,
                       need_noise: bool = False, need_x0: bool = False):
    """Backward of diffusion_loss_fwd in one pass: dpred = factor * gscale * weight[t] * diff, dnoise = -c_n[t] dpred,
    dx0 = -c_x[t] dpred (the target's share).  -> (dpred, dnoise, dx0), None where not requested."""
    _req_cuda(diff, t, tgt_coef, weight, gscale)
    B = diff.shape[0]
    _loss_tables(t, tgt_coef, weight, T, B)
    assert diff.dtype == torch.float32 and (need_pred or need_noise or need_x0)
    dpred, dnoise, dx0 = (torch.empty_like(diff) if n else None for n in (need_pred, need_noise, need_x0))
    _lib.call("cesm_diffusion_loss_bwd", _ptr(diff), _ptr(t), _ptr(tgt_coef), _ptr(weight), _ptr(gscale), factor,
              _ptr(dpred), _ptr(dnoise), _ptr(dx0), B, diff.numel() // B, T, _stream())
    return dpred, dnoise, dx0


def scale_by_scalar(x, gscale, factor: float):
    _req_cuda(x, gscale)
    out = torch.empty_like(x)
    _lib.call("cesm_scale_by_scalar", _ptr(x), _ptr(gscale), factor, _ptr(out), x.numel(), _stream())
    return out


def p_sample(xt, eps, z, t, betas, sqrt_1mac, sqrt_recip_a, post_var):
    _req_cuda(xt, eps, z, t, betas, sqrt_1mac, sqrt_recip_a, post_var)
    out = torch.empty_like(xt)
    B = xt.shape[0]
    _lib.call("cesm_p_sample", _ptr(xt), _ptr(eps), _ptr(z), _ptr(t), _ptr(betas), _ptr(sqrt_1mac), _ptr(sqrt_recip_a),
              _ptr(post_var), _ptr(out), B, xt.numel() // B, _stream())
    return out


def ddim_step(xt, eps, z, t, coef, T: int, out=None, next_t=None, t_out=None):
    """out = A[t]*xt + B[t]*eps + S[t]*z per sample from the fp32 [T, 3] table of `model.ddim_schedule`.
    `out` may be `xt` (in place); `z` may be None when every S is 0.  With `t_out`, next_t[t] is written there
    (a buffer other than `t`)."""
    _req_cuda(xt, eps, z, t, coef, out, next_t, t_out)
    assert coef.dtype == torch.float32 and coef.shape == (T, 3), (coef.dtype, tuple(coef.shape), T)
    assert t.dtype == torch.int64 and xt.dtype == eps.dtype == torch.float32 and eps.shape == xt.shape
    assert z is None or (z.dtype == torch.float32 and z.shape == xt.shape)
    assert (t_out is None) == (next_t is None), "next_t and t_out go together"
    assert next_t is None or (next_t.dtype == torch.int64 and next_t.shape == (T,) and t_out.dtype == torch.int64)
    out = torch.empty_like(xt) if out is None else out
    assert out.dtype == torch.float32 and out.shape == xt.shape
    B = xt.shape[0]
    _lib.call("cesm_ddim_step", _ptr(xt), _ptr(eps), _ptr(z), _ptr(t), _ptr(coef), _ptr(next_t), _ptr(t_out), _ptr(out),
              T, B, xt.numel() // B, _stream())
    return out


def dpm_step(xt, eps, hist, t, coef, T: int, out=None, next_t=None, t_out=None):
    """DPM-Solver++(2M) step per sample from the fp32 [T, 5] table (P, Q, R, K0, K1) of `model.dpm_schedule`:
    x0 = P*xt + Q*eps, out = R*xt + K0*x0 + K1*hist, then hist = x0.  `hist` is read only where K1 != 0 and must
    be a buffer of its own; `out` may be `xt` (in place).  With `t_out`, next_t[t] is written there (a buffer other
    than `t`)."""
    _req_cuda(xt, eps, hist, t, coef, out, next_t, t_out)
    assert coef.dtype == torch.float32 and coef.shape == (T, 5), (coef.dtype, tuple(coef.shape), T)
    assert t.dtype == torch.int64 and xt.dtype == eps.dtype == torch.float32 and eps.shape == xt.shape
    assert hist.dtype == torch.float32 and hist.shape == xt.shape
    assert (t_out is None) == (next_t is None), "next_t and t_out go together"
    assert next_t is None or (next_t.dtype == torch.int64 and next_t.shape == (T,) and t_out.dtype == torch.int64)
    out = torch.empty_like(xt) if out is None else out
    assert out.dtype == torch.float32 and out.shape == xt.shape
    B = xt.shape[0]
    _lib.call("cesm_dpm_step", _ptr(xt), _ptr(eps), _ptr(hist), _ptr(t), _ptr(coef), _ptr(next_t), _ptr(t_out),
              _ptr(out), T, B, xt.numel() // B, _stream())
    return out


# ---- seeded sampling noise ------------------------------------------------------------------------
X_T_DRAW = 0xFFFFFFFF  # draw id of the initial noise x_T; the step leaving timestep t draws with id t
# Saliency draw d (engine.SaliencyEngine) uses draw id SALIENCY_DRAW_BASE + d, d < SALIENCY_MAX_DRAWS: above every
# sampler timestep (T < 2^31) and below X_T_DRAW, so saliency noise never repeats a sampling draw of the same field.
SALIENCY_DRAW_BASE = 0x80000000
SALIENCY_MAX_DRAWS = X_T_DRAW - SALIENCY_DRAW_BASE


def split_seed(seed) -> Tuple[int, int]:
    """A sampling seed (an int in [0, 2^64), not a bool) -> its (low, high) 32-bit words, the Philox key."""
    if isinstance(seed, bool) or not isinstance(seed, numbers.Integral) or not 0 <= int(seed) < 1 << 64:
        raise ValueError(f"seed must be an integer in [0, 2**64), got {seed!r}")
    seed = int(seed)
    return seed & 0xFFFFFFFF, seed >> 32


def field_id_vector(field_ids, B: int, device) -> torch.Tensor:
    """Validate the field ids of a seeded chain -> int64 [B] on `device`.  None means arange(B); ids must be integers
    >= 0, and repeats are allowed (padding rows that regenerate a real field)."""
    if field_ids is None:
        return torch.arange(B, dtype=torch.int64, device=device)
    ids = torch.as_tensor(field_ids)
    if ids.dtype.is_floating_point or ids.dtype.is_complex or ids.dtype == torch.bool:
        raise ValueError(f"field_ids must be integers, got dtype {ids.dtype}")
    if tuple(ids.shape) != (B,):
        raise ValueError(f"field_ids must have shape ({B},), got {tuple(ids.shape)}")
    ids = ids.to(torch.int64)
    if bool((ids < 0).any()):
        raise ValueError("field_ids must be >= 0")
    return ids.to(device)


def _seeded_ids(field_ids: torch.Tensor, B: int) -> None:
    assert field_ids.dtype == torch.int64 and field_ids.shape == (B,), (field_ids.dtype, tuple(field_ids.shape), B)


def field_normal(seed: int, field_ids: torch.Tensor, draw: int, shape=None, out: Optional[torch.Tensor] = None):
    """out[b] = the standard normals of field `field_ids[b]` in draw `draw` under `seed` (counter-based Philox4x32-10,
    see include/cesm_b200.h): the same values whatever the row, batch or device.  Give `out` or the [B, ...] `shape`."""
    lo, hi = split_seed(seed)
    out = torch.empty(shape, dtype=torch.float32, device=field_ids.device) if out is None else out
    _req_cuda(field_ids, out)
    assert out.dtype == torch.float32 and 0 <= int(draw) <= 0xFFFFFFFF
    B = out.shape[0]
    _seeded_ids(field_ids, B)
    _lib.call("cesm_field_normal", lo, hi, _ptr(field_ids), int(draw), _ptr(out), B, out.numel() // B, _stream())
    return out


def p_sample_seeded(xt, eps, seed: int, field_ids, t, betas, sqrt_1mac, sqrt_recip_a, post_var, out=None):
    """p_sample with z = field_normal(seed, field_ids, draw=t[b]) drawn inside the kernel (no z buffer), bit-identical
    to p_sample fed that draw.  `out` may be `xt` (in place).  A t outside [0, T) gives NaN."""
    lo, hi = split_seed(seed)
    _req_cuda(xt, eps, field_ids, t, betas, sqrt_1mac, sqrt_recip_a, post_var, out)
    assert t.dtype == torch.int64 and xt.dtype == eps.dtype == torch.float32 and eps.shape == xt.shape
    out = torch.empty_like(xt) if out is None else out
    assert out.dtype == torch.float32 and out.shape == xt.shape
    B = xt.shape[0]
    _seeded_ids(field_ids, B)
    _lib.call("cesm_p_sample_seeded", _ptr(xt), _ptr(eps), lo, hi, _ptr(field_ids), _ptr(t), _ptr(betas),
              _ptr(sqrt_1mac), _ptr(sqrt_recip_a), _ptr(post_var), _ptr(out), betas.shape[0], B, xt.numel() // B,
              _stream())
    return out


def ddim_step_seeded(xt, eps, seed: int, field_ids, t, coef, T: int, out=None, next_t=None, t_out=None):
    """ddim_step with z = field_normal(seed, field_ids, draw=t[b]) drawn inside the kernel (no z buffer),
    bit-identical to ddim_step fed that draw.  Same `out` / `next_t` / `t_out` contract as ddim_step."""
    lo, hi = split_seed(seed)
    _req_cuda(xt, eps, field_ids, t, coef, out, next_t, t_out)
    assert coef.dtype == torch.float32 and coef.shape == (T, 3), (coef.dtype, tuple(coef.shape), T)
    assert t.dtype == torch.int64 and xt.dtype == eps.dtype == torch.float32 and eps.shape == xt.shape
    assert (t_out is None) == (next_t is None), "next_t and t_out go together"
    assert next_t is None or (next_t.dtype == torch.int64 and next_t.shape == (T,) and t_out.dtype == torch.int64)
    out = torch.empty_like(xt) if out is None else out
    assert out.dtype == torch.float32 and out.shape == xt.shape
    B = xt.shape[0]
    _seeded_ids(field_ids, B)
    _lib.call("cesm_ddim_step_seeded", _ptr(xt), _ptr(eps), lo, hi, _ptr(field_ids), _ptr(t), _ptr(coef),
              _ptr(next_t), _ptr(t_out), _ptr(out), T, B, xt.numel() // B, _stream())
    return out
