"""Training-step and sampling engines: the loop bodies of the reference's train.py / inference.py
on CUDA streams and graphs.

TrainEngine.step is what `train_one_epoch` does per batch (train.py:829-867) -- fp16 forward/backward with
a dynamically scaled loss (autocast + GradScaler, train.py:853-867), unscale + inf check, global-norm clip,
AdamW, scaler update -- with two differences that are deliberate and documented in DESIGN.md:
  * under torch.distributed the gradients really are averaged over ranks (the reference wraps the
    model in DDP, train.py:1076, but calls `.module.loss`, so its reducer never fires): static
    buckets in expected-ready order are all-reduced with NCCL on a side stream as soon as the last
    gradient of a bucket has been produced, overlapping the rest of the backward pass;
  * the whole step (RNG draws, forward, backward, all-reduce, unscale, clip, AdamW, loss-scale update) is
    captured once into a CUDA graph and replayed: the GradScaler logic (found-inf check, skipped step, backoff /
    growth of the scale) runs on the device, so there are no host syncs and no per-kernel launch latency.
"""
from __future__ import annotations

import math
import numbers
from typing import List, Optional

import torch
import torch.distributed as dist

from . import kernels as K
from . import ops


def _ready_order(named_params):
    """Parameters in the order backward is expected to finish them: reverse registration order,
    with the tensors every level feeds (time MLP, relative-position table) and the input stage last."""
    late, normal = [], []
    for name, p in named_params:
        if not p.requires_grad:
            continue
        if ".time_mlp." in name or ".time_rel_pos_bias." in name or ".input_conv." in name or ".input_temp_op." in name:
            late.append((name, p))
        else:
            normal.append((name, p))
    return list(reversed(normal)) + list(reversed(late))


class GradBuckets:
    """All gradients live in one flat fp32 buffer (p.grad are views), cut into `n_buckets`
    contiguous buckets in expected-ready order.  With a process group, each bucket is all-reduced
    on `comm_stream` from the hook of its last-finished parameter."""

    def __init__(self, module: torch.nn.Module, n_buckets: int = 4, process_group=None):
        self.pg = process_group
        self.world = dist.get_world_size(process_group) if (process_group is not None or dist.is_initialized()) else 1
        order = _ready_order(module.named_parameters())
        self.params = [p for _, p in order]
        self._named = order
        self._seen = {}
        # every tensor starts on a 64-byte boundary of the flat buffers (kernels read parameters with
        # 16-byte vector loads); the padding stays zero in the gradient, parameter and moment buffers
        pad = lambda n: (n + 15) // 16 * 16
        total = sum(pad(p.numel()) for p in self.params)
        dev = self.params[0].device
        self.flat = torch.zeros(total, dtype=torch.float32, device=dev)
        off = 0
        self.bounds: List[int] = [0]
        per_bucket = -(-total // max(1, n_buckets))
        self._bucket_of = {}
        self._pending_init: List[int] = []
        self.offsets = {}                     # id(param) -> start of its slice in the flat buffers
        # what the reference's optimizer sees: AdamW(diffusion.parameters()) (train.py:1078) -- EVERY parameter in
        # registration order, including the frozen rotary `freqs` (index 3), which holds an index but never a state
        self.registration_order = list(module.parameters())
        for p in self.params:
            n = p.numel()
            self.offsets[id(p)] = off
            p.grad = self.flat[off:off + n].view_as(p)
            b = len(self.bounds) - 1
            self._bucket_of[p.data_ptr()] = b
            if len(self._pending_init) <= b:
                self._pending_init.append(0)
            self._pending_init[b] += 1
            off += pad(n)
            if off - self.bounds[-1] >= per_bucket and off < total:
                self.bounds.append(off)
        self.bounds.append(total)
        self.n_buckets = len(self.bounds) - 1
        self._pending = list(self._pending_init)
        self.on_cuda = dev.type == "cuda"
        self.comm_stream = torch.cuda.Stream(device=dev) if (self.world > 1 and self.on_cuda) else None
        self._hooks = []
        if self.world > 1:
            for p in self.params:
                self._hooks.append(p.register_post_accumulate_grad_hook(self._on_grad))
        self._owned = {p.data_ptr() for p in self.params}
        # packed fp32 scratch of the multi-tap weight gradients: (param ptr, tap key) -> (tensor, spec)
        self._scratch = {}
        self._unpack_plan = {}   # bucket -> (entry count, device descriptor table)
        ops.set_grad_sink(self)  # weight gradients are accumulated straight into the flat buffer

    # grad-sink protocol (ops._wgrad_to_param)
    def owns(self, p) -> bool:
        return p.data_ptr() in self._owned

    def scratch(self, p, key, spec) -> torch.Tensor:
        """Persistent zeroed fp32 [O, T, I] buffer the tcgen05 weight-gradient kernel accumulates into;
        `unpack_bucket` adds it into p.grad (layout `spec`) and re-zeroes it."""
        k = (p.data_ptr(), key)
        ent = self._scratch.get(k)
        if ent is None:
            O, T, I = spec[0], spec[1], spec[2]
            ent = (torch.zeros((O, T, I), dtype=torch.float32, device=p.device), spec, p,
                   self._bucket_of[p.data_ptr()])
            self._scratch[k] = ent
            self._unpack_plan.clear()
        return ent[0]

    def unpack_bucket(self, b: Optional[int]) -> None:
        """One kernel adds every packed scratch of bucket `b` (all buckets if None) into the flat gradient."""
        from . import _lib
        ents = [e for e in self._scratch.values() if b is None or e[3] == b]
        if not ents:
            return
        plan = self._unpack_plan.get(b)
        if plan is None or plan[0] != len(ents):
            arr = (_lib.PackDesc * len(ents))()
            for d, (buf, spec, p, _) in zip(arr, ents):
                d.src, d.dst = buf.data_ptr(), p.grad.data_ptr()
                d.O, d.T, d.I, d.so, d.si = spec[0], spec[1], spec[2], spec[3], spec[4]
                for i, o in enumerate(spec[5]):
                    d.tap_off[i] = int(o)
            host = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8)
            plan = (len(ents), host.to(self.flat.device))
            self._unpack_plan[b] = plan
        _lib.call("cesm_unpack_wgrads_batched", plan[1].data_ptr(), plan[0], K._stream())

    def ready(self, p) -> None:
        if self.world > 1:
            self._on_grad(p)

    def begin_step(self):
        self.flat.zero_()
        self._pending = list(self._pending_init)
        self._seen = {}

    def _on_grad(self, p):
        # A parameter whose gradient was written directly (ops._direct) reports through ready(); torch ALSO runs
        # its post-accumulate hook (measured on 2 B200s: every direct parameter reported twice, the buckets
        # reached zero after half of their gradients and were all-reduced early -- replicas diverged).  Count
        # each parameter once per step.
        if id(p) in self._seen:
            return
        b = self._bucket_of[p.data_ptr()]
        self._seen[id(p)] = True
        self._pending[b] -= 1
        if self._pending[b] == 0:
            if self.on_cuda and ops._SIDE[0] is not None:
                torch.cuda.current_stream().wait_stream(ops._SIDE[0])   # weight gradients issued on the side stream
            self.unpack_bucket(b)
            bucket = self.flat[self.bounds[b]:self.bounds[b + 1]]
            if not self.on_cuda:  # host tensors (gloo): used by the CPU tests of the bucket logic
                dist.all_reduce(bucket, op=dist.ReduceOp.SUM, group=self.pg)
                return
            cur = torch.cuda.current_stream()
            self.comm_stream.wait_stream(cur)
            with torch.cuda.stream(self.comm_stream):
                dist.all_reduce(bucket, op=dist.ReduceOp.SUM, group=self.pg)

    def finish_step(self):
        if self.on_cuda:
            ops.join_side_stream()
        if self.world == 1:
            self.unpack_bucket(None)
        if self.world > 1:
            # a parameter that produced no gradient leaves its bucket un-reduced and the replicas diverge
            # silently (the reference passes find_unused_parameters=True for this, train.py:1076): fail loudly.
            # Host-side bookkeeping only; during graph capture it is checked once, for the captured step.
            late = [b for b, n in enumerate(self._pending) if n > 0]
            if late:
                names = [n for n, p in self._named if self._bucket_of.get(p.data_ptr()) in late and not self._seen.get(id(p))]
                raise RuntimeError(f"gradient buckets {late} were never all-reduced: no gradient arrived for {names[:8]}"
                                   f"{' ...' if len(names) > 8 else ''}")
        if self.world > 1 and self.on_cuda:
            torch.cuda.current_stream().wait_stream(self.comm_stream)

    def flatten_params_(self) -> torch.Tensor:
        """Re-home every parameter into one flat fp32 buffer laid out like `flat` (same offsets), so the
        optimizer step is one elementwise kernel over four flat arrays.  `p.data` become views: state
        dicts, `load_state_dict` (in-place copies) and the modules themselves see no difference."""
        assert not self._scratch, "flatten the parameters before the first step"
        flat_p = torch.zeros_like(self.flat)
        off = 0
        bucket_of = {}
        for p in self.params:
            n = p.numel()
            view = flat_p[off:off + n].view_as(p)
            view.copy_(p.data)
            b = self._bucket_of[p.data_ptr()]
            p.data = view
            bucket_of[p.data_ptr()] = b  # the sink protocol is keyed on the (new) storage address
            off += (n + 15) // 16 * 16
        self._bucket_of = bucket_of
        self._owned = set(bucket_of)
        return flat_p

    def clip_(self, max_norm: float) -> torch.Tensor:
        """Global-norm clip of every gradient (train.py:865) on the flat buffer: two kernels, no sync."""
        total = torch.linalg.vector_norm(self.flat)
        coef = torch.clamp(max_norm / (total + 1e-6), max=1.0)
        self.flat.mul_(coef)
        return total


def check_ema_args(ema_decay, ema_start):
    """Validated (decay, start) of a weight EMA: decay None (no EMA) or a real number in [0, 1), start an integer >= 0."""
    if ema_decay is not None:
        if isinstance(ema_decay, bool) or not isinstance(ema_decay, numbers.Real):
            raise ValueError(f"ema_decay must be a number in [0, 1) or None, got {ema_decay!r}")
        ema_decay = float(ema_decay)
        if not (math.isfinite(ema_decay) and 0.0 <= ema_decay < 1.0):
            raise ValueError(f"ema_decay must be in [0, 1), got {ema_decay}")
    if isinstance(ema_start, bool) or not isinstance(ema_start, numbers.Integral):
        raise ValueError(f"ema_start must be an integer, got {ema_start!r}")
    if ema_start < 0:
        raise ValueError(f"ema_start must be >= 0, got {ema_start}")
    return ema_decay, int(ema_start)


class FusedAdamW:
    """torch.optim.AdamW (train.py:1078-1083) + torch.amp.GradScaler (train.py:862-867, 1084) + clip_grad_norm_
    (train.py:865) as three launches of the library's own kernels over flat buffers (`cesm_adamw_step`).  Step
    counter, loss scale, growth tracker, learning rate and weight decay live in a small device vector (`state`,
    layout in include/cesm_b200.h) so that a replayed CUDA graph advances / honours them.  Drop-in for what the
    engine and train.py use of an optimizer: `step()`, `state_dict()`, `load_state_dict()`,
    `param_groups[0]["lr"]` (picked up by the next step through `sync_hparams`, also after graph capture).

    With `ema_decay` set, `self.ema` is a flat fp32 exponential moving average of the parameters (same layout as
    `self.p`, starting as a copy of it) that every step updates in the same kernel (`cesm_adamw_ema_step`): a copy
    while the step count is <= `ema_start`, then ema += (1 - ema_decay) (p - ema).  Both are fixed per optimizer.
    The EMA is not optimizer state: `state_dict()` stays torch AdamW's format."""

    def __init__(self, buckets: "GradBuckets", lr, betas, weight_decay, eps, max_grad_norm,
                 init_scale: float = 65536.0, growth_interval: int = 2000, ema_decay: Optional[float] = None,
                 ema_start: int = 0):
        from . import _lib
        self.ema_decay, self.ema_start = check_ema_args(ema_decay, ema_start)
        self._buckets = buckets
        self.g = buckets.flat
        self.p = buckets.flatten_params_()
        self.m = torch.zeros_like(self.p)
        self.v = torch.zeros_like(self.p)
        self.ema = self.p.clone() if self.ema_decay is not None else None
        st = torch.zeros(K.OPT_STATE_FLOATS, dtype=torch.float32)
        st[K.OPT_SCALE], st[K.OPT_INTERVAL] = init_scale, growth_interval  # GradScaler() defaults
        self.state = st.to(self.p.device)
        self.partials = torch.zeros(_lib.load().cesm_adamw_partials(), dtype=torch.float32, device=self.p.device)
        self.param_groups = [dict(lr=lr, betas=tuple(betas), weight_decay=weight_decay, eps=eps)]
        self.max_grad_norm = max_grad_norm
        self._synced = None    # (lr, weight_decay) last written to the device
        self._frozen = None    # (betas, eps, max_norm) baked into the first launch / the captured graph
        self.sync_hparams()

    @property
    def grad_norm(self) -> torch.Tensor:
        return self.state[K.OPT_NORM]

    @property
    def loss_scale(self) -> torch.Tensor:
        """0-dim device view of the current loss scale (multiply the loss by it before backward)."""
        return self.state[K.OPT_SCALE]

    def sync_hparams(self) -> None:
        """Bring the device copy of lr / weight decay up to date with `param_groups` (a 8-byte H2D copy, only when
        they changed; call outside graph capture -- TrainEngine does, before every replay)."""
        hp = self.param_groups[0]
        cur = (float(hp["lr"]), float(hp["weight_decay"]))
        if cur != self._synced:
            if self.p.is_cuda and torch.cuda.is_current_stream_capturing():
                raise RuntimeError("FusedAdamW: lr / weight_decay changed while a CUDA graph is being captured")
            self.state[K.OPT_LR:K.OPT_WD + 1].copy_(torch.tensor(cur, dtype=torch.float32))
            self._synced = cur
        frozen = (tuple(hp["betas"]), float(hp["eps"]), self.max_grad_norm)
        if self._frozen is not None and frozen != self._frozen:
            raise RuntimeError("FusedAdamW: betas / eps / max_grad_norm are fixed after the first step "
                               f"(were {self._frozen}, now {frozen})")

    def step(self) -> None:
        hp = self.param_groups[0]
        if not (self.p.is_cuda and torch.cuda.is_current_stream_capturing()):
            self.sync_hparams()
        self._frozen = (tuple(hp["betas"]), float(hp["eps"]), self.max_grad_norm)
        if self.ema is None:
            K.adamw_step(self.p, self.g, self.m, self.v, self.partials, self.state, hp["betas"][0], hp["betas"][1],
                         hp["eps"], self.max_grad_norm)
        else:
            K.adamw_ema_step(self.p, self.g, self.m, self.v, self.ema, self.partials, self.state, hp["betas"][0],
                             hp["betas"][1], hp["eps"], self.max_grad_norm, self.ema_decay, self.ema_start)
        ops.invalidate_weight_cache()  # the fp16 operand copies are stale now

    def _slices(self):
        """index -> (flat offset, numel, shape) for every TRAINABLE parameter, indexed as a torch optimizer built over
        `module.parameters()` indexes them (the reference's AdamW, train.py:1078: frozen parameters keep their slot)."""
        return {i: (self._buckets.offsets[id(p)], p.numel(), p.shape)
                for i, p in enumerate(self._buckets.registration_order) if id(p) in self._buckets.offsets}

    def state_dict(self) -> dict:
        """torch.optim.AdamW's state-dict format, so that checkpoints interchange with the reference's
        `optimizer.load_state_dict` (train.py:934-939) and with any torch AdamW over the same module."""
        step = self.state[0].detach().clone()
        state = {i: {"step": step.clone(), "exp_avg": self.m[o:o + n].view(shape).clone(),
                     "exp_avg_sq": self.v[o:o + n].view(shape).clone()}
                 for i, (o, n, shape) in self._slices().items()}
        g = self.param_groups[0]
        group = dict(lr=g["lr"], betas=tuple(g["betas"]), eps=g["eps"], weight_decay=g["weight_decay"], amsgrad=False,
                     maximize=False, foreach=None, capturable=False, differentiable=False, fused=None,
                     params=list(range(len(self._buckets.registration_order))))
        # "grad_scaler": torch.amp.GradScaler.state_dict() keys (the reference loads one if present, train.py:940-944)
        scaler = {"scale": float(self.state[K.OPT_SCALE]), "growth_factor": 2.0, "backoff_factor": 0.5,
                  "growth_interval": int(self.state[K.OPT_INTERVAL]), "_growth_tracker": int(self.state[K.OPT_TRACKER])}
        return {"state": state, "param_groups": [group], "grad_scaler": scaler}

    def load_state_dict(self, sd: dict) -> None:
        if "state" in sd:  # torch format (ours, the reference's, or any torch AdamW over module.parameters())
            slices = self._slices()
            steps = []
            for i, (o, n, shape) in slices.items():
                st = sd["state"].get(i)
                if st is None:
                    continue
                self.m[o:o + n].view(shape).copy_(st["exp_avg"])
                self.v[o:o + n].view(shape).copy_(st["exp_avg_sq"])
                steps.append(float(st["step"]))
            if steps:
                self.state[0] = max(steps)
            for g, src in zip(self.param_groups, sd.get("param_groups", [])):
                g.update({k: src[k] for k in ("lr", "betas", "eps", "weight_decay") if k in src})
            sc = sd.get("grad_scaler")
            if sc:
                self.state[K.OPT_SCALE] = float(sc["scale"])
                self.state[K.OPT_TRACKER] = float(sc.get("_growth_tracker", 0))
                self.state[K.OPT_INTERVAL] = float(sc.get("growth_interval", 2000))
            self.sync_hparams()
            return
        self.state[:1].copy_(sd["step"])  # flat format of earlier checkpoints of this repo
        self.m.copy_(sd["exp_avg"])
        self.v.copy_(sd["exp_avg_sq"])
        for g, src in zip(self.param_groups, sd.get("param_groups", [])):
            g.update(src)
        self.sync_hparams()


class TrainEngine:
    """One data-parallel training step of `Diffusion.loss` as a replayable CUDA graph.

    `ema_decay` / `ema_start` (CUDA only) keep an exponential moving average of the weights inside the captured
    optimizer step (FusedAdamW).  It starts as a copy of the weights when the engine is built; loading weights into
    the module afterwards does not touch it -- call `reset_ema()` or `load_ema_state_dict()`.  `ema_state_dict()`
    has the layout of `diffusion.model.state_dict()`.

    `min_snr_gamma` (a real number > 0, or None for uniform weights) trains with Min-SNR-gamma loss weights for the
    diffusion's target (`Diffusion.min_snr_weights`), held in a device buffer the captured step reads.  The weights go
    down to 4e-5 (v, t = 999) and scale a sample's whole backward, which runs in fp16: the step divides the loss
    scale's seed by the batch's largest weight (over all ranks), so the fp16 gradient stream carries the magnitudes
    of an unweighted step, and multiplies the fp32 gradients by it before the optimizer step.

    `cond_drop_prob` = p in [0, 1) (CUDA only; 0 is off) trains for classifier-free guidance: each step, each sample
    sees the null (all-zero) condition with probability p.  The mask is drawn inside the captured step into the device
    buffer `keep` (fp32 [B], 0 = dropped) by `kernels.cond_keep`, counter-based from (key, step, global sample index
    rank * B + b): the same global batch drops the same samples on one GPU or split over ranks, and a replay needs no
    host round trip.  The key comes from torch's default generator when the engine is built (rank 0's under
    torch.distributed), so `torch.manual_seed` fixes it as it fixes t and the noise.  The input convolution reads the
    condition through the mask (ops.InputConvFn); no masked copy of it is made."""

    def __init__(self, diffusion, batch_shape, cond_shape, lr: float = 2e-4, betas=(0.9, 0.999),
                 weight_decay: float = 1e-4, eps: float = 1e-8, max_grad_norm: Optional[float] = 1.0,
                 n_buckets: int = 4, use_graph: bool = True, process_group=None, ema_decay: Optional[float] = None,
                 ema_start: int = 0, min_snr_gamma: Optional[float] = None, cond_drop_prob: float = 0.0):
        from .model import check_cond_drop_prob
        ema_decay, ema_start = check_ema_args(ema_decay, ema_start)
        self.cond_drop_prob = check_cond_drop_prob(cond_drop_prob)
        self.loss_weights = None if min_snr_gamma is None else diffusion.min_snr_weights(min_snr_gamma)
        self.diffusion = diffusion
        dev = next(diffusion.parameters()).device
        if ema_decay is not None and dev.type != "cuda":
            raise RuntimeError("the weight EMA is updated by the CUDA optimizer step; there is none on host tensors")
        if self.cond_drop_prob > 0 and dev.type != "cuda":
            raise RuntimeError("the condition-dropout mask is drawn by a CUDA kernel; there is none on host tensors")
        self.device = dev
        self.world = dist.get_world_size(process_group) if dist.is_initialized() else 1
        self.pg = process_group
        self.keep = None
        if self.cond_drop_prob > 0:
            key = torch.randint(0, 1 << 62, (1,), dtype=torch.int64).to(dev)
            if self.world > 1:
                dist.broadcast(key, src=0, group=process_group)
            self.cond_drop_key = int(key.item())
            self.keep = torch.ones((batch_shape[0],), dtype=torch.float32, device=dev)
            self.keep_step = torch.zeros((), dtype=torch.int64, device=dev)  # advanced by every executed step
            self.first_sample = (dist.get_rank(process_group) if self.world > 1 else 0) * batch_shape[0]
        if self.world > 1:
            for t in list(diffusion.parameters()) + list(diffusion.buffers()):
                dist.broadcast(t.data, src=0, group=process_group)  # what DDP's constructor does
        self.buckets = GradBuckets(diffusion, n_buckets=n_buckets, process_group=process_group)
        self.max_grad_norm = max_grad_norm
        # AdamW as train.py:1078-1083 with the clip of train.py:865 folded in; the step lives inside the graph
        if self.buckets.on_cuda:
            self.opt = FusedAdamW(self.buckets, lr, betas, weight_decay, eps, max_grad_norm, ema_decay=ema_decay,
                                  ema_start=ema_start)
        else:  # host tensors: only the gloo tests of the bucket logic come through here
            self.opt = torch.optim.AdamW(self.buckets.params, lr=lr, betas=betas, weight_decay=weight_decay, eps=eps)
        self.x0 = torch.zeros(batch_shape, dtype=torch.float32, device=dev)
        self.cond = torch.zeros(cond_shape, dtype=torch.float32, device=dev)
        self.loss = torch.zeros((), dtype=torch.float32, device=dev)
        self.grad_norm = torch.zeros((), dtype=torch.float32, device=dev)
        self.use_graph = use_graph
        self.graph: Optional[torch.cuda.CUDAGraph] = None
        self.launches_per_step = 0
        self._warm = 0
        self.arena = K.ZeroArena(dev) if dev.type == "cuda" else None
        # weight gradients on a second stream (ops._on_side)
        self.side_stream = torch.cuda.Stream(device=dev) if dev.type == "cuda" else None

    # the captured region ----------------------------------------------------------------------
    def _step_body(self):
        if self.arena is None:
            return self._step_body_inner()
        try:
            self.arena.begin()  # one memset; the library's per-call scratch memsets are off until end()
            self._step_body_inner()
        finally:
            self.arena.end()
            ops.set_side_stream(None)

    def _step_body_inner(self):
        ops.set_grad_sink(self.buckets)
        ops.set_side_stream(self.side_stream)
        ops.prepack_all()  # one kernel refreshes every fp16 operand copy of the (just updated) weights
        self.buckets.begin_step()
        drop = {}  # condition dropout off: the call of before
        if self.keep is not None:
            drop["keep"] = K.cond_keep(self.cond_drop_key, self.keep_step, self.first_sample, self.cond_drop_prob,
                                       self.keep)
        if self.loss_weights is None:
            loss, wmax = self.diffusion.loss(self.x0, self.cond, **drop), None
        else:
            # the reference's randint draw, made here so that the batch's largest weight is known
            t = torch.randint(0, self.diffusion.T, (self.x0.shape[0],), device=self.x0.device)
            loss = self.diffusion.loss(self.x0, self.cond, t, weights=self.loss_weights, **drop)
            wmax = self.loss_weights[t].max()
            if self.world > 1:
                dist.all_reduce(wmax, op=dist.ReduceOp.MAX, group=self.pg)
        if isinstance(self.opt, FusedAdamW):
            # scaler.scale(loss).backward() (train.py:862); /world turns the bucket SUM into the mean
            seed = self.opt.loss_scale * (1.0 / self.world)
            (loss * (seed if wmax is None else seed / wmax)).backward()
        else:
            scaled = loss / self.world if self.world > 1 else loss
            (scaled if wmax is None else scaled / wmax).backward()
        self.buckets.finish_step()
        if wmax is not None:
            self.buckets.flat.mul_(wmax)
        if isinstance(self.opt, FusedAdamW):
            self.opt.step()
            self.grad_norm.copy_(self.opt.grad_norm)
        else:
            if self.max_grad_norm is not None:
                self.grad_norm.copy_(self.buckets.clip_(self.max_grad_norm))
            self.opt.step()
        self.loss.copy_(loss.detach())

    def _run(self):
        from . import _lib
        if not self.use_graph:
            n0 = _lib.launch_count()
            self._step_body()
            self.launches_per_step = _lib.launch_count() - n0
            return
        if self.graph is None:
            if self._warm < 2:  # eager warm-up: lazy init of optimizer state, NCCL, kernel attributes
                self._warm += 1
                self._step_body()
                return
            torch.cuda.synchronize()
            self.graph = torch.cuda.CUDAGraph()
            n0 = _lib.launch_count()
            # (capturing the critical chain on a higher-priority stream than the weight-gradient stream was tried:
            # 11.37 ms against 10.98 ms with equal priorities -- the interleaving the scheduler picks by itself is better)
            with torch.cuda.graph(self.graph):
                self._step_body()
            self.launches_per_step = _lib.launch_count() - n0
        if isinstance(self.opt, FusedAdamW):
            self.opt.sync_hparams()  # an lr schedule / warm-up changes param_groups between replays
        self.graph.replay()
        # the replayed optimizer step rewrote the parameters behind torch's back: every cached fp16 operand
        # copy / F = 1 fold keyed on (pointer, version, epoch) is stale for any eager or eval use that follows
        ops.invalidate_weight_cache()

    # public -----------------------------------------------------------------------------------
    @property
    def has_ema(self) -> bool:
        return isinstance(self.opt, FusedAdamW) and self.opt.ema is not None

    def _require_ema(self) -> None:
        if not self.has_ema:
            raise RuntimeError("this TrainEngine keeps no weight EMA (build it with ema_decay=...)")

    def _ema_entries(self):
        """(name, module tensor, flat EMA slice or None for a frozen tensor) in diffusion.model.state_dict() order."""
        self._require_ema()
        offsets, e = self.buckets.offsets, self.opt.ema
        out = []
        for name, t in self.diffusion.model.state_dict(keep_vars=True).items():
            o = offsets.get(id(t))
            out.append((name, t, None if o is None else e[o:o + t.numel()].view(t.shape)))
        return out

    def ema_state_dict(self) -> dict:
        """The EMA weights in the layout of `diffusion.model.state_dict()` (a checkpoint's "model"): trainable tensors
        from the EMA, frozen ones (the rotary `freqs`) and buffers copied from the module."""
        return {name: (t if e is None else e).detach().clone() for name, t, e in self._ema_entries()}

    def load_ema_state_dict(self, sd: dict) -> None:
        """Load an `ema_state_dict()`; keys and shapes must match exactly.  Frozen entries are checked, not loaded."""
        entries = self._ema_entries()
        names = [n for n, _, _ in entries]
        missing, unexpected = [n for n in names if n not in sd], [k for k in sd if k not in set(names)]
        if missing or unexpected:
            raise RuntimeError(f"EMA state dict: missing keys {missing}, unexpected keys {unexpected}")
        bad = [n for n, t, _ in entries if tuple(sd[n].shape) != tuple(t.shape)]
        if bad:
            raise RuntimeError(f"EMA state dict: shape mismatch for {bad}")
        with torch.no_grad():
            for n, _, e in entries:
                if e is not None:
                    e.copy_(sd[n])

    def reset_ema(self) -> None:
        """Restart the EMA from the current weights (e.g. after loading weights into the module)."""
        self._require_ema()
        self.opt.ema.copy_(self.opt.p)

    def step_resident(self) -> torch.Tensor:
        """One step on whatever is in the static device buffers `x0` / `cond`."""
        self._run()
        return self.loss

    def step_indices(self, device_ds, indices, augment: bool = True) -> torch.Tensor:
        """One step on samples of a device-resident dataset (`synthetic.DeviceEnsemble`): the batch is
        gathered straight into the static buffers by one kernel; only a 24-byte plan per sample crosses PCIe."""
        device_ds.batch_into(indices, self.cond, self.x0, augment)
        self._run()
        return self.loss

    def step(self, x0: torch.Tensor, cond: torch.Tensor) -> torch.Tensor:
        """One step on a host (ideally pinned) or device batch; returns the device loss scalar."""
        self.x0.copy_(x0, non_blocking=True)
        self.cond.copy_(cond, non_blocking=True)
        self._run()
        return self.loss


class SampleEngine:
    """Ensemble generation (inference.py:217-232 + model.py:186-194): the reverse chain for a batch
    of independent fields, one UNet call + fused p_sample update per step, replayed as a CUDA graph
    whose only per-step inputs are the timestep vector and the fresh noise (device RNG).

    With `ddim_steps=N` the engine runs the strided DDIM chain of `model.ddim_schedule` instead (N UNet calls per
    field; `eta` scales its noise).  The mode is fixed per engine, so there is still one graph: a replay is one UNet
    call, a noise draw only if eta > 0, and one `ddim_step` launch that updates `x` in place and writes the next
    timestep to `t_next`, copied into `t`.  The coefficient and next-timestep tables live in static device buffers,
    which the graph captures by address.

    With `dpm_steps=N` it runs the deterministic DPM-Solver++(2M) chain of `model.dpm_schedule` (N UNet calls per
    field).  A replay is one UNet call and one `dpm_step` launch that updates `x` and the previous-x0 buffer `hist`
    in place and writes `t_next`, copied into `t`: no noise draw, and the same library launches per step as DDIM with
    eta = 0.  The first step does not read `hist`, so a new chain needs no reset of it.

    With `seed` (an int in [0, 2^64)) the noise is counter-based instead of torch's generator: x_T of the field in row
    b is `kernels.field_normal(seed, field_ids[b], X_T_DRAW)` and the step leaving timestep t draws z with id t inside
    the fused `p_sample_seeded` / `ddim_step_seeded` kernel.  A field's chain then depends on (seed, field id) only, not
    on its row, its batch, `batch_size` or the rank it runs on.  The ids live in a static int64 buffer `field_ids`
    that the graph captures by address; a replay has no noise draw and there is no z buffer.

    A v-prediction diffusion (`diffusion.prediction_type == "v"`) runs every mode through tables with the conversion to
    eps folded in; its DDPM chain is the `ddim_step` (or `ddim_step_seeded`) launch with `diffusion.ddpm_coef`, the
    N = T, eta = 1 table, in place of `p_sample`.

    With `guidance` = w > 0 every mode samples with classifier-free guidance.  `x`, `cond` and `t` are the first halves
    of static 2B-row buffers whose second halves hold the same fields with the null (all-zero) condition; a replay
    copies x and t into the second half, makes one UNet call on the 2B rows and one guided update launch that combines
    the two halves of the output, (1 + w) out_cond - w out_null, while it updates the B fields.  Seeded noise is drawn
    for the B fields only.  w = 0 is the unguided engine, unchanged."""

    def __init__(self, diffusion, shape, use_graph: bool = True, ddim_steps: Optional[int] = None, eta: float = 0.0,
                 dpm_steps: Optional[int] = None, seed: Optional[int] = None, guidance: float = 0.0):
        from .model import check_guidance, ddim_schedule, dpm_schedule
        self.guidance = check_guidance(guidance)
        if seed is not None:
            K.split_seed(seed)
        if dpm_steps is not None and ddim_steps is not None:
            raise ValueError("ddim_steps and dpm_steps are mutually exclusive")
        if dpm_steps is not None and float(eta) != 0.0:
            raise ValueError(f"eta applies to DDIM only; the DPM-Solver++(2M) chain is deterministic (got eta={eta})")
        self.diffusion = diffusion
        dev = next(diffusion.parameters()).device
        self.device = dev
        self.shape = tuple(shape)
        B = self.shape[0]
        if self.guidance:  # rows [B, 2B): the same fields with the null condition, which stays zero
            self._x2 = torch.zeros((2 * B, *self.shape[1:]), dtype=torch.float32, device=dev)
            self._c2 = torch.zeros_like(self._x2)
            self._t2 = torch.zeros((2 * B,), dtype=torch.long, device=dev)
            self.x, self.cond, self.t = self._x2[:B], self._c2[:B], self._t2[:B]
        else:
            self.x = torch.zeros(self.shape, dtype=torch.float32, device=dev)
            self.cond = torch.zeros(self.shape, dtype=torch.float32, device=dev)
            self.t = torch.zeros((B,), dtype=torch.long, device=dev)
        self.seed = None if seed is None else int(seed)
        if seed is None:
            self.z = torch.zeros(self.shape, dtype=torch.float32, device=dev)
        else:
            self.field_ids = torch.arange(self.shape[0], dtype=torch.int64, device=dev)
        self.arena = K.ZeroArena(dev) if dev.type == "cuda" else None
        self.use_graph = use_graph
        self.graph: Optional[torch.cuda.CUDAGraph] = None
        self.launches_per_step = 0
        self.ddim_steps, self.eta = ddim_steps, float(eta)
        if ddim_steps is not None:
            self.ddim_taus, coef, next_t = ddim_schedule(diffusion.alphas_cumprod, ddim_steps, eta,
                                                         diffusion.prediction_type)
            self.ddim_coef = coef.to(dev)
            self.ddim_next_t = next_t.to(dev)
            self.t_next = torch.zeros_like(self.t)
        self.dpm_steps = dpm_steps
        if dpm_steps is not None:
            self.dpm_taus, coef, next_t = dpm_schedule(diffusion.alphas_cumprod, dpm_steps, diffusion.prediction_type)
            self.dpm_coef = coef.to(dev)
            self.dpm_next_t = next_t.to(dev)
            self.t_next = torch.zeros_like(self.t)
            self.hist = torch.zeros(self.shape, dtype=torch.float32, device=dev)

    def _body(self):
        if self.arena is None:
            return self._body_inner()
        try:
            self.arena.begin()  # scratch of the step comes zeroed from one arena: one memset, not ~30
            self._body_inner()
        finally:
            self.arena.end()

    def _body_inner(self):
        d = self.diffusion
        w = self.guidance or None
        with torch.no_grad():
            if w is None:
                eps = d.model(self.x, self.cond, self.t)
            else:
                B = self.shape[0]
                self._x2[B:].copy_(self.x)
                self._t2[B:].copy_(self.t)
                eps = d.model(self._x2, self._c2, self._t2)
            if self.ddim_steps is not None:
                z = None
                if self.seed is not None and self.eta > 0:
                    K.ddim_step_seeded(self.x, eps, self.seed, self.field_ids, self.t, self.ddim_coef, d.T, out=self.x,
                                       next_t=self.ddim_next_t, t_out=self.t_next, guidance=w)
                    self.t.copy_(self.t_next)
                    return
                if self.eta > 0:
                    self.z.normal_()
                    z = self.z
                K.ddim_step(self.x, eps, z, self.t, self.ddim_coef, d.T, out=self.x, next_t=self.ddim_next_t,
                            t_out=self.t_next, guidance=w)
                self.t.copy_(self.t_next)
                return
            if self.dpm_steps is not None:
                K.dpm_step(self.x, eps, self.hist, self.t, self.dpm_coef, d.T, out=self.x, next_t=self.dpm_next_t,
                           t_out=self.t_next, guidance=w)
                self.t.copy_(self.t_next)
                return
            if self.seed is not None and d.prediction_type == "v":
                K.ddim_step_seeded(self.x, eps, self.seed, self.field_ids, self.t, d.ddpm_coef, d.T, out=self.x,
                                   guidance=w)
                self.t.sub_(1)
                return
            if self.seed is not None:
                K.p_sample_seeded(self.x, eps, self.seed, self.field_ids, self.t, d.betas,
                                  d.sqrt_one_minus_alphas_cumprod, d.sqrt_recip_alphas, d.posterior_variance,
                                  out=self.x, guidance=w)
                self.t.sub_(1)
                return
            self.z.normal_()  # model.py:181 randn_like; kept in a static buffer so that a caller can read the draw
            if d.prediction_type == "v":
                K.ddim_step(self.x, eps, self.z, self.t, d.ddpm_coef, d.T, out=self.x, guidance=w)
                self.t.sub_(1)
                return
            self.x.copy_(K.p_sample(self.x, eps, self.z, self.t, d.betas, d.sqrt_one_minus_alphas_cumprod,
                                    d.sqrt_recip_alphas, d.posterior_variance, guidance=w))
            self.t.sub_(1)

    def step(self):
        from . import _lib
        if not self.use_graph:
            n0 = _lib.launch_count()
            self._body()
            self.launches_per_step = _lib.launch_count() - n0
            return
        if self.graph is None:
            x_keep, t_keep = self.x.clone(), self.t.clone()
            h_keep = self.hist.clone() if self.dpm_steps is not None else None  # a mid-chain step reads hist
            self._body()  # eager warm-up
            torch.cuda.synchronize()
            self.x.copy_(x_keep)
            self.t.copy_(t_keep)
            if h_keep is not None:
                self.hist.copy_(h_keep)
            self.graph = torch.cuda.CUDAGraph()
            n0 = _lib.launch_count()
            with torch.cuda.graph(self.graph):
                self._body()
            self.launches_per_step = _lib.launch_count() - n0
            self.x.copy_(x_keep)
            self.t.copy_(t_keep)
        self.graph.replay()

    def refresh_operands(self) -> None:
        """Operands derived from the weights (packed fp16 copies, F = 1 folds) are captured by ADDRESS: bring their
        contents up to date with whatever training / load_state_dict did since the graph was captured."""
        ops.prepack_all()
        ops.refresh_folds()

    @torch.no_grad()
    def sample(self, cond: torch.Tensor, steps: Optional[int] = None, field_ids=None) -> torch.Tensor:
        """cond: [B,1,H,W] -> generated field [B,1,H,W] after `steps` (default T) reverse steps.  In DDIM and DPM
        mode the chain is always the engine's N steps, and `steps` must be None.  `field_ids` (B integers >= 0,
        default arange(B), repeats allowed) name the fields of a seeded engine; an unseeded one takes none."""
        T = self.diffusion.T
        if self.seed is None and field_ids is not None:
            raise ValueError("field_ids needs a seeded SampleEngine (SampleEngine(..., seed=...))")
        if self.seed is not None:
            ids = K.field_id_vector(field_ids, self.shape[0], self.device)
        if self.ddim_steps is not None:
            if steps is not None:
                raise ValueError("steps does not apply to a DDIM-mode SampleEngine (its chain is ddim_steps long)")
            steps = len(self.ddim_taus)
        if self.dpm_steps is not None:
            if steps is not None:
                raise ValueError("steps does not apply to a DPM-mode SampleEngine (its chain is dpm_steps long)")
            steps = len(self.dpm_taus)
        steps = T if steps is None else steps
        self.refresh_operands()
        self.cond.copy_(cond, non_blocking=True)
        if self.seed is None:
            self.x.normal_()
        else:
            self.field_ids.copy_(ids)
            K.field_normal(self.seed, self.field_ids, K.X_T_DRAW, out=self.x)
        self.t.fill_(T - 1)
        for _ in range(steps):
            self.step()
        return self.x.clone()


SALIENCY_LOSS_SCALE = 65536.0


def saliency_timesteps(T: int, draws) -> torch.Tensor:
    """Stratified saliency timesteps t_d = floor((d + 1/2) T / D), d = 0..D-1: the midpoint of each of D equal strata
    of [0, T), deterministic and the same for every field.  D must be an integer in [1, T] (distinct timesteps).
    -> int64 [D] on the CPU."""
    if isinstance(draws, bool) or not isinstance(draws, numbers.Integral):
        raise ValueError(f"draws must be an integer, got {draws!r}")
    D = int(draws)
    if not 1 <= D <= T:
        raise ValueError(f"draws must be in [1, {T}], got {D}")
    return torch.tensor([(2 * d + 1) * T // (2 * D) for d in range(D)], dtype=torch.int64)


class SaliencyEngine:
    """Emission saliency of a frozen model: how sensitive the denoising loss is to each pixel and frame of the
    condition.  For field b (target x0_b, condition window cond_b),

        S_b = (1/D) sum_d  d/d cond_b  MSE_b(eps_theta(q_sample(x0_b, t_d, eps_d), cond_b, t_d), eps_d),

    where MSE_b is the mean over field b's own H*W pixels.  `Diffusion.loss` is the mean over the whole batch, so
    its gradient is multiplied by B: a field's saliency does not depend on the batch it is computed in.

    Timesteps: `saliency_timesteps(T, draws)` (stratified, no RNG), or an explicit int64 `timesteps` tensor of shape
    [D] (the same for every field) or [D, B].  Noise: torch's CUDA generator; with `seed` (an int in [0, 2^64)) the
    counter-based normals of `kernels.field_normal(seed, field_id, SALIENCY_DRAW_BASE + d)`, so a field's saliency
    depends on (seed, field id) only -- not on its row, its batch or the rank it runs on.

    One draw is a forward and a backward with frozen weights (no weight-gradient launch), captured once as a CUDA
    graph and replayed D times; the condition gradient is added, scaled by B / D, straight into the output buffer by
    the input convolution's data-gradient kernel.  Every parameter must have requires_grad False
    (`inference.load_diffusion_from_checkpoint` freezes them); the training gradient sink is off while a draw runs,
    so a TrainEngine in the same process never receives saliency gradients.  `launches_per_step` counts the library
    launches of one draw.

    The loss is the eps-MSE for either target.  For a v-model the per-timestep weights ab[t] turn its v-MSE into it:
    at the same x_t, eps_hat - eps = sqrt(ab) (v_hat - v).  Training loss weights (Min-SNR) never enter."""

    def __init__(self, diffusion, x0_shape, cond_shape, draws: int = 16, use_graph: bool = True,
                 seed: Optional[int] = None, timesteps=None):
        trainable = [n for n, p in diffusion.named_parameters() if p.requires_grad]
        if trainable:
            raise ValueError(f"SaliencyEngine needs a frozen model; {len(trainable)} parameters require grad "
                             f"(e.g. {trainable[0]}): call requires_grad_(False) on the model")
        if seed is not None:
            K.split_seed(seed)
        x0_shape, cond_shape = tuple(x0_shape), tuple(cond_shape)
        if len(x0_shape) != 4 or x0_shape[1] != 1:
            raise ValueError(f"x0_shape must be [B, 1, H, W], got {x0_shape}")
        B, _, H, W = x0_shape
        if len(cond_shape) == 4:
            frames = 1
        elif len(cond_shape) == 5:
            frames = cond_shape[2]
        else:
            raise ValueError(f"cond_shape must be [B, 1, H, W] or [B, 1, K, H, W], got {cond_shape}")
        if cond_shape[:2] != (B, 1) or cond_shape[-2:] != (H, W):
            raise ValueError(f"cond_shape {cond_shape} does not match x0_shape {x0_shape}")
        T = diffusion.T
        if timesteps is None:
            tab = saliency_timesteps(T, draws)
        else:
            tab = torch.as_tensor(timesteps)
            if tab.dtype.is_floating_point or tab.dtype.is_complex or tab.dtype == torch.bool:
                raise ValueError(f"timesteps must be integers, got dtype {tab.dtype}")
            if tab.dim() not in (1, 2) or tab.shape[0] < 1 or (tab.dim() == 2 and tab.shape[1] != B):
                raise ValueError(f"timesteps must have shape [D] or [D, {B}], got {tuple(tab.shape)}")
            tab = tab.to("cpu", torch.int64)
            if bool((tab < 0).any()) or bool((tab >= T).any()):
                raise ValueError(f"timesteps must lie in [0, {T})")
        if tab.shape[0] > K.SALIENCY_MAX_DRAWS:
            raise ValueError(f"at most {K.SALIENCY_MAX_DRAWS} draws")
        if tab.dim() == 1:
            tab = tab[:, None].expand(-1, B)
        self.diffusion = diffusion
        dev = next(diffusion.parameters()).device
        if dev.type != "cuda":
            raise ValueError("SaliencyEngine runs on the CUDA kernels; the model is on " + str(dev))
        self.device = dev
        self.x0_shape, self.cond_shape = x0_shape, cond_shape
        self.draws = int(tab.shape[0])
        self.t_table = tab.contiguous().to(dev)
        self.loss_weights = diffusion.alphas_cumprod.float() if diffusion.prediction_type == "v" else None
        # the gradient stream is fp16: like the training step (GradScaler's initial scale), the backward starts
        # from 2^16 instead of 1, and the sink's scale takes it out again
        self.grad_seed = torch.full((), SALIENCY_LOSS_SCALE, dtype=torch.float32, device=dev)
        self.scale = B / (self.draws * SALIENCY_LOSS_SCALE)
        self.x0 = torch.zeros(x0_shape, dtype=torch.float32, device=dev)
        self.cond = torch.zeros(cond_shape, dtype=torch.float32, device=dev, requires_grad=True)
        self.noise = torch.zeros(x0_shape, dtype=torch.float32, device=dev)
        self.t = torch.zeros((B,), dtype=torch.int64, device=dev)
        self.out = torch.zeros((B, 1, frames, H, W), dtype=torch.float32, device=dev)
        self.seed = None if seed is None else int(seed)
        if seed is not None:
            self.field_ids = torch.arange(B, dtype=torch.int64, device=dev)
        self.arena = K.ZeroArena(dev)
        self.use_graph = use_graph
        self.graph: Optional[torch.cuda.CUDAGraph] = None
        self.launches_per_step = 0

    def _draw(self, d: int) -> None:
        """Timesteps and noise of draw d into the static buffers the captured pass reads."""
        self.t.copy_(self.t_table[d])
        if self.seed is None:
            self.noise.normal_()
        else:
            K.field_normal(self.seed, self.field_ids, K.SALIENCY_DRAW_BASE + d, out=self.noise)

    def _body(self) -> None:
        prev = ops._GRAD_SINK[0]
        ops.set_grad_sink(None)
        ops.set_cond_grad_sink(self.out, self.scale)
        self.arena.begin()
        try:
            with torch.enable_grad():
                self.diffusion.loss(self.x0, self.cond, self.t, self.noise, self.loss_weights).backward(self.grad_seed)
        finally:
            self.arena.end()
            ops.set_cond_grad_sink(None)
            ops.set_grad_sink(prev)

    def refresh_operands(self) -> None:
        """Packed fp16 weight copies are captured by address: bring them up to date with the module's weights."""
        ops.prepack_all()
        ops.refresh_folds()

    def saliency(self, x0: torch.Tensor, cond: torch.Tensor, field_ids=None) -> torch.Tensor:
        """x0: [B, 1, H, W] target fields, cond: their condition windows (cond_shape) -> fp32 [B, 1, K, H, W]
        saliency (K = 1 for a 4-D cond).  `field_ids` (B integers >= 0, default arange(B)) name the fields of a
        seeded engine; an unseeded one takes none."""
        from . import _lib
        if tuple(x0.shape) != self.x0_shape or tuple(cond.shape) != self.cond_shape:
            raise ValueError(f"expected x0 {self.x0_shape} and cond {self.cond_shape}, got {tuple(x0.shape)} and "
                             f"{tuple(cond.shape)}")
        if self.seed is None and field_ids is not None:
            raise ValueError("field_ids needs a seeded SaliencyEngine (SaliencyEngine(..., seed=...))")
        ids = K.field_id_vector(field_ids, self.x0_shape[0], self.device) if self.seed is not None else None
        self.refresh_operands()
        with torch.no_grad():
            self.x0.copy_(x0, non_blocking=True)
            self.cond.copy_(cond, non_blocking=True)
            if ids is not None:
                self.field_ids.copy_(ids)
        if self.use_graph and self.graph is None:
            self.t.copy_(self.t_table[0])
            self._body()  # eager warm-up on whatever noise the buffer holds; what it added to `out` is cleared below
            torch.cuda.synchronize()
            ops.prepack_all()  # every operand the warm-up registered is current: the capture re-packs none
            self.graph = torch.cuda.CUDAGraph()
            n0 = _lib.launch_count()
            with torch.cuda.graph(self.graph):
                self._body()
            self._graph_launches = _lib.launch_count() - n0
        self.out.zero_()
        for d in range(self.draws):
            n0 = _lib.launch_count()
            self._draw(d)
            if self.graph is not None:
                self.graph.replay()
                self.launches_per_step = _lib.launch_count() - n0 + self._graph_launches
            else:
                self._body()
                self.launches_per_step = _lib.launch_count() - n0
        return self.out.clone()
