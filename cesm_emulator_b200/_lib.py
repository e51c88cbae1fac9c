"""ctypes binding of libcesm_b200.so (the C ABI declared in include/cesm_b200.h).

There is deliberately no fallback: if the shared library is missing, or a call fails, the
caller gets an exception.  Importing this module does not need a GPU; calling a compute entry
point does.
"""
from __future__ import annotations

import ctypes
from ctypes import POINTER, Structure, c_char_p, c_float, c_int32, c_int64, c_void_p
from pathlib import Path

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "libcesm_b200.so"

CESM_MAX_TAPS = 16


class IgemmArgs(Structure):
    """Mirror of `cesm_igemm_args` (include/cesm_b200.h)."""

    _fields_ = [
        ("a0", c_void_p), ("a1", c_void_p),
        ("c0", c_int32), ("c1", c_int32),
        ("n", c_int32), ("h", c_int32), ("w", c_int32),
        ("stride", c_int32),
        ("num_taps", c_int32),
        ("tap_dh", c_int32 * CESM_MAX_TAPS), ("tap_dw", c_int32 * CESM_MAX_TAPS),
        ("wt", c_void_p), ("cout", c_int32),
        ("oh", c_int32), ("ow", c_int32),
        ("out", c_void_p), ("ldo", c_int32),
        ("out_h", c_int32), ("out_w", c_int32),
        ("o_sh", c_int32), ("o_sw", c_int32), ("o_h0", c_int32), ("o_w0", c_int32),
        ("bias", c_void_p), ("residual", c_void_p), ("ldr", c_int32),
        ("gn_sums", c_void_p), ("gn_groups", c_int32), ("gn_frames", c_int32),
        ("ln_colsum", c_void_p), ("ln_eps", ctypes.c_float), ("reserved_", c_int32),
    ]


class WgradArgs(Structure):
    """Mirror of `cesm_wgrad_args` (include/cesm_b200.h)."""

    _fields_ = [
        ("x0", c_void_p), ("x1", c_void_p),
        ("c0", c_int32), ("c1", c_int32),
        ("n", c_int32), ("h", c_int32), ("w", c_int32),
        ("stride", c_int32),
        ("num_taps", c_int32),
        ("tap_dh", c_int32 * CESM_MAX_TAPS), ("tap_dw", c_int32 * CESM_MAX_TAPS),
        ("dy", c_void_p), ("cout", c_int32),
        ("oh", c_int32), ("ow", c_int32),
        ("y_h", c_int32), ("y_w", c_int32),
        ("y_sh", c_int32), ("y_sw", c_int32), ("y_h0", c_int32), ("y_w0", c_int32),
        ("dw", c_void_p),
        ("dw_so", ctypes.c_longlong), ("dw_si", ctypes.c_longlong),
        ("dw_tap_off", c_int32 * CESM_MAX_TAPS),
    ]


class PackDesc(Structure):
    """Mirror of `cesm_pack_desc` (include/cesm_b200.h)."""

    _fields_ = [
        ("src", c_void_p), ("dst", c_void_p),
        ("O", c_int32), ("T", c_int32), ("I", c_int32), ("pad_", c_int32),
        ("so", ctypes.c_longlong), ("si", ctypes.c_longlong),
        ("tap_off", c_int32 * CESM_MAX_TAPS),
    ]


class FilmDesc(Structure):
    """Mirror of `cesm_film_desc` (include/cesm_b200.h)."""

    _fields_ = [("W", c_void_p), ("bias", c_void_p), ("dW", c_void_p), ("db", c_void_p), ("N", c_int32), ("n0", c_int32)]


class CesmError(RuntimeError):
    pass


_lib = None


def load() -> ctypes.CDLL:
    """Load the kernel library, building nothing: a missing .so is a hard error."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise CesmError(
            f"{LIB_PATH} not found: build it with `python -m cesm_emulator_b200.build` "
            "(there is no CPU or PyTorch fallback for the B200 kernels)")
    lib = ctypes.CDLL(str(LIB_PATH))
    lib.cesm_last_error.restype = c_char_p
    lib.cesm_version.restype = c_char_p
    lib.cesm_launch_count.restype = ctypes.c_longlong
    lib.cesm_linattn_ws_floats.restype = ctypes.c_size_t
    lib.cesm_linattn_ws_floats.argtypes = [ctypes.c_int, ctypes.c_int]
    lib.cesm_adamw_partials.restype = ctypes.c_int
    lib.cesm_tattn_long_max_frames.restype = ctypes.c_int
    lib.cesm_set_prezeroed_scratch.restype = None
    lib.cesm_set_prezeroed_scratch.argtypes = [ctypes.c_int]
    _declare(lib)
    _lib = lib
    return lib


# name -> argtypes; every function returns int (cesm_status)
_P, _I, _L, _F, _U = c_void_p, ctypes.c_int, ctypes.c_longlong, c_float, ctypes.c_uint
_SIGNATURES: dict[str, list] = {
    "cesm_igemm": [POINTER(IgemmArgs), _P],
    "cesm_wgrad": [POINTER(WgradArgs), _P],
    "cesm_pack_weight": [_P, _P, _I, _I, _I, _L, _L, POINTER(c_int32), _P],
    "cesm_pack_weights_batched": [_P, _I, _P],
    "cesm_unpack_wgrads_batched": [_P, _I, _P],
    "cesm_unpack_wgrad": [_P, _P, _I, _I, _I, _L, _L, POINTER(c_int32), _I, _P],
    "cesm_adamw_step": [_P, _P, _P, _P, _L, _P, _P, _F, _F, _F, _F, _P],
    "cesm_adamw_ema_step": [_P, _P, _P, _P, _P, _L, _P, _P, _F, _F, _F, _F, ctypes.c_double, _L, _P],
    "cesm_colsum": [_P, _P, _L, _I, _I, _P],
    "cesm_gn_stats": [_P, _P, _I, _L, _I, _I, _P],
    "cesm_gn_apply_fwd": [_P, _P, _P, _P, _P, _P, _P, _I, _L, _I, _I, _F, _P],
    "cesm_gn_bwd": [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _L, _I, _I, _F, _I, _P],
    "cesm_ln_fwd": [_P, _P, _P, _L, _I, _F, _P],
    "cesm_ln_bwd": [_P, _P, _P, _P, _P, _P, _L, _I, _F, _I, _P],
    "cesm_tattn_fwd": [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _F, _P],
    "cesm_tattn_bwd": [_P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _F, _P],
    "cesm_tattn_proj_fwd": [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _F, _P],
    "cesm_tattn_long_fwd": [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _F, _P],
    "cesm_tattn_long_bwd": [_P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _F, _P],
    "cesm_mattn_fwd": [_P, _P, _P, _I, _I, _I, _I, _F, _P],
    "cesm_mattn_bwd": [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _F, _P],
    "cesm_linattn_fwd": [_P, _P, _P, _I, _I, _I, _I, _F, _P],
    "cesm_linattn_bwd": [_P, _P, _P, _P, _P, _I, _I, _I, _I, _F, _P],
    "cesm_film_fwd": [_P, _P, _P, _I, _I, _I, _I, _P],
    "cesm_film_bwd": [_P, _P, _P, _I, _I, _P, _I, _I, _I, _P],
    "cesm_gather_windows": [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _P],
    "cesm_qkv_bwd": [_P, _P, _P, _P, _P, _L, _L, _I, _I, _P],
    "cesm_input_patches": [_P, _P, _I, _I, _P, _I, _I, _I, _I, _I, _I, _P],
    "cesm_input_patches_masked": [_P, _P, _I, _I, _P, _P, _I, _I, _I, _I, _I, _I, _P],
    "cesm_input_weight_pack": [_P, _P, _P, _I, _I, _I, _P],
    "cesm_input_conv_fwd": [_P, _P, _I, _I, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P],
    "cesm_input_conv_wgrad": [_P, _P, _I, _I, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P],
    "cesm_input_conv_dgrad": [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _F, _I, _P],
    "cesm_input_conv_dgrad_masked": [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _F, _I, _P],
    "cesm_out_conv_fwd": [_P, _P, _P, _P, _I, _I, _I, _L, _I, _P],
    "cesm_out_conv_bwd": [_P, _P, _P, _P, _P, _P, _I, _I, _I, _L, _I, _P],
    "cesm_sinusoidal": [_P, _P, _I, _I, _P],
    "cesm_small_linear_fwd": [_P, _P, _P, _P, _I, _I, _I, _I, _P],
    "cesm_small_linear_bwd": [_P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P],
    "cesm_q_sample": [_P, _P, _P, _P, _P, _P, _I, _L, _P],
    "cesm_q_sample_bwd": [_P, _P, _P, _P, _P, _P, _I, _L, _P],
    "cesm_mse_fwd": [_P, _P, _P, _P, _L, _P],
    "cesm_scale_by_scalar": [_P, _P, _F, _P, _L, _P],
    "cesm_diffusion_loss_fwd": [_P, _P, _P, _P, _P, _P, _P, _P, _I, _L, _I, _P],
    "cesm_diffusion_loss_bwd": [_P, _P, _P, _P, _P, _F, _P, _P, _P, _I, _L, _I, _P],
    "cesm_p_sample": [_P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _L, _P],
    "cesm_ddim_step": [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _L, _P],
    "cesm_dpm_step": [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _L, _P],
    "cesm_field_normal": [_U, _U, _P, _U, _P, _I, _L, _P],
    "cesm_p_sample_seeded": [_P, _P, _U, _U, _P, _P, _P, _P, _P, _P, _P, _I, _I, _L, _P],
    "cesm_ddim_step_seeded": [_P, _P, _U, _U, _P, _P, _P, _P, _P, _P, _I, _I, _L, _P],
    "cesm_p_sample_guided": [_P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _L, _F, _P],
    "cesm_ddim_step_guided": [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _L, _F, _P],
    "cesm_dpm_step_guided": [_P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _L, _F, _P],
    "cesm_p_sample_seeded_guided": [_P, _P, _U, _U, _P, _P, _P, _P, _P, _P, _P, _I, _I, _L, _F, _P],
    "cesm_ddim_step_seeded_guided": [_P, _P, _U, _U, _P, _P, _P, _P, _P, _P, _I, _I, _L, _F, _P],
    "cesm_cond_keep": [_U, _U, _P, _L, _F, _P, _I, _P],
}


def _declare(lib: ctypes.CDLL) -> None:
    for name, argtypes in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = ctypes.c_int


def exported_symbols() -> list[str]:
    return ["cesm_last_error", "cesm_version", "cesm_launch_count", "cesm_linattn_ws_floats", "cesm_adamw_partials",
            "cesm_set_prezeroed_scratch", "cesm_tattn_long_max_frames",
            *sorted(_SIGNATURES)]


def launch_count() -> int:
    """Kernels launched by libcesm_b200.so in this process so far."""
    return int(load().cesm_launch_count())


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().cesm_last_error().decode("utf-8", "replace")
        raise CesmError(f"{what} failed (status {rc}): {msg}")


class KernelProfiler:
    """Per-C-ABI-call device timing with CUDA events on the calling stream (bench.py's kernel
    breakdown and roofline pass).  Only usable outside graph capture; every call is bracketed by
    two events, so use it in a dedicated, untimed pass."""

    def __init__(self):
        self.records = []  # (name, meta, start_event, end_event)

    def summary(self):
        """-> {key: {"calls", "ms", "flops", "bytes"}} with key = name or name + '/' + meta['kind']."""
        import torch
        torch.cuda.synchronize()
        out = {}
        for name, meta, e0, e1 in self.records:
            key = name if not meta or "kind" not in meta else f"{name}/{meta['kind']}"
            d = out.setdefault(key, {"calls": 0, "ms": 0.0, "flops": 0.0, "bytes": 0.0})
            d["calls"] += 1
            d["ms"] += e0.elapsed_time(e1)
            if meta:
                d["flops"] += meta.get("flops", 0.0)
                d["bytes"] += meta.get("bytes", 0.0)
        return out


PROFILER = None  # set to a KernelProfiler to time every call
# CESM_NVTX=1: every C-ABI call is wrapped in an NVTX range named after the entry point (plus the profiler
# `kind`, e.g. "cesm_igemm/9tap"), so nsys / ncu --nvtx timelines and `ncu --nvtx-include` filters speak the C ABI's
# vocabulary.  Ranges pushed during CUDA-graph capture annotate the capture, not the replays: profile with
# use_graph=False (bench.py --no-graph) for per-call ranges.
NVTX = bool(int(__import__("os").environ.get("CESM_NVTX", "0")))


def _nvtx_call(lib, name, args, meta):
    from torch.cuda import nvtx
    nvtx.range_push(name if not meta or "kind" not in meta else f"{name}/{meta['kind']}")
    try:
        check(getattr(lib, name)(*args), name)
    finally:
        nvtx.range_pop()


def call(name: str, *args, _meta=None) -> None:
    lib = load()
    prof = PROFILER
    if prof is None:
        if NVTX:
            _nvtx_call(lib, name, args, _meta)
            return
        check(getattr(lib, name)(*args), name)
        return
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    check(getattr(lib, name)(*args), name)
    e1.record()
    prof.records.append((name, _meta, e0, e1))
