"""Synthetic stand-in for the CESM2-LE NetCDF data and dataset_single_member.py.

`SyntheticEnsemble` generates arrays of the reference's logical shape (member, time, lat, lon,
channel) and exposes them in the layout the reference's loaders produce, `(T, M, 1, H, W)`
float32, globally z-scored (train.py:624-646).  `window(idx)` follows
WindowedAllMembersDataset_random's default "consecutive" indexing (dataset_single_member.py:91-108,
168-196): idx -> (member = idx % M, start = idx // M), K consecutive condition frames, target at
the centre frame, optional time-reversal augmentation and random crop.

The fields are not noise: the condition is a smooth emission pattern growing in time, and the
target is a low-pass response to the cumulative condition plus member-dependent weather noise, so
the diffusion loss has something to learn.  Sharding over ranks is DistributedSampler's
(train.py:1002): a seeded permutation of all indices, rank r takes every world-th starting at r.
"""
from __future__ import annotations

from typing import Optional, Tuple

import numpy as np
import torch


class SyntheticEnsemble:
    def __init__(self, members: int = 34, times: int = 251, lat: int = 192, lon: int = 288, seed: int = 1234,
                 K: int = 3, crop_hw: Optional[Tuple[int, int]] = None, time_reverse_p: float = 0.5):
        if K < 2:
            raise ValueError("K must be >= 2")  # dataset_single_member.py:47
        self.M, self.T, self.H, self.W, self.K = members, times, lat, lon, K
        self.crop_hw = crop_hw
        self.time_reverse_p = time_reverse_p
        rng = np.random.default_rng(seed)
        self._aug = np.random.default_rng(seed + 1)
        yy = np.linspace(-1.0, 1.0, lat, dtype=np.float32)[:, None]
        xx = np.linspace(-1.0, 1.0, lon, dtype=np.float32)[None, :]
        # a few emission "hot spots" (same for all members: emissions are a scenario, not weather)
        blobs = np.zeros((lat, lon), np.float32)
        for _ in range(6):
            cy, cx, s = rng.uniform(-0.8, 0.8), rng.uniform(-0.9, 0.9), rng.uniform(0.05, 0.25)
            blobs += rng.uniform(0.5, 1.5) * np.exp(-((yy - cy) ** 2 + (xx - cx) ** 2) / (2 * s * s))
        growth = np.linspace(0.0, 1.0, times, dtype=np.float32) ** 2
        cond_tm = growth[:, None, None] * blobs[None]                                    # (T, H, W)
        cum = np.cumsum(cond_tm, axis=0) / max(1, times)
        # temperature response: zonal-mean warming + polar amplification + member weather noise
        resp = cum.mean(axis=(1, 2), keepdims=True) * (1.0 + 0.8 * np.abs(yy)[None]) + 0.3 * cum
        # logical layout (member, time, lat, lon, channel)
        self.cond_mtllc = np.broadcast_to(cond_tm[None, ..., None], (members, times, lat, lon, 1))
        noise = rng.standard_normal((members, times, lat, lon, 1), dtype=np.float32)
        tgt = resp[None, ..., None] * 4.0 + 0.5 * noise
        # reference layout (T, M, 1, H, W), globally z-scored (train.py:640-646)
        self.cond, _ = self._z(np.ascontiguousarray(np.transpose(self.cond_mtllc, (1, 0, 4, 2, 3))))
        self.tgt, (mu, sd) = self._z(np.ascontiguousarray(np.transpose(tgt, (1, 0, 4, 2, 3))))
        # the known truth in normalised units: member (t, m) is target_mean[t] + target_noise_std * N(0, 1) noise
        self.target_mean = ((resp.astype(np.float64) * 4.0 - float(mu)) / float(sd)).astype(np.float32)  # (T, H, W)
        self.target_noise_std = 0.5 / float(sd)
        self.num_units = max(1, self.T - self.K + 1)

    @classmethod
    def from_arrays(cls, cond: np.ndarray, tgt: np.ndarray, K: int = 3, crop_hw: Optional[Tuple[int, int]] = None,
                    time_reverse_p: float = 0.5, seed: int = 1234) -> "SyntheticEnsemble":
        """Wrap existing `(T, M, 1, H, W)` arrays (the constructor arguments of the reference's dataset class,
        dataset_single_member.py:30-44) instead of generating fields; the arrays are used as they are."""
        if cond.ndim != 5 or tgt.ndim != 5:
            raise ValueError("Expect (T, M, 1, H, W)")       # dataset_single_member.py:42
        if cond.shape != tgt.shape:
            raise ValueError("cond/tgt shapes must match")   # :43
        if K < 2:
            raise ValueError("K must be >= 2")
        self = cls.__new__(cls)
        self.T, self.M, _, self.H, self.W = cond.shape
        self.K, self.crop_hw, self.time_reverse_p = int(K), crop_hw, float(time_reverse_p)
        self._aug = np.random.default_rng(seed + 1)
        self.cond_mtllc = None
        self.target_mean = self.target_noise_std = None  # unknown for arrays from outside
        self.cond = np.ascontiguousarray(cond, dtype=np.float32)
        self.tgt = np.ascontiguousarray(tgt, dtype=np.float32)
        self.num_units = max(1, self.T - self.K + 1)
        return self

    @staticmethod
    def _z(a: np.ndarray):
        """Global z-score -> (z-scored float32 array, (mean, std + 1e-8) it applied)."""
        a = a.astype(np.float32)
        mu, sd = a.mean(), a.std() + 1e-8
        return (a - mu) / sd, (mu, sd)

    def __len__(self) -> int:
        return self.num_units * self.M

    def out_hw(self) -> Tuple[int, int]:
        if self.crop_hw is None:
            return self.H, self.W
        return min(self.crop_hw[0], self.H), min(self.crop_hw[1], self.W)

    def plan(self, idx: int, augment: bool = True) -> Tuple[int, int, int, int, int, int]:
        """The random decisions of one sample, in the reference's draw order (dataset_single_member.py:
        168-196): -> (member, first frame, target frame, crop row, crop col, time-reverse flag)."""
        m, t0 = idx % self.M, idx // self.M
        anchor = min(t0 + self.K // 2, self.T - 1)
        rev = int(augment and self.time_reverse_p > 0 and self._aug.random() < self.time_reverse_p)
        i = j = 0
        if self.crop_hw is not None:
            h, w = self.out_hw()
            if augment:
                i = 0 if h == self.H else int(self._aug.integers(0, self.H - h + 1))
                j = 0 if w == self.W else int(self._aug.integers(0, self.W - w + 1))
            else:
                i, j = (self.H - h) // 2, (self.W - w) // 2
        return m, t0, anchor, i, j, rev

    def window(self, idx: int, augment: bool = True):
        """-> (cond_win [1,K,h,w], x0 [1,h,w]) float32 torch tensors."""
        m, t0, anchor, i, j, rev = self.plan(idx, augment)
        h, w = self.out_hw()
        times = np.arange(t0, t0 + self.K)
        cond = self.cond[times, m, 0]            # (K, H, W)
        x0 = self.tgt[anchor, m]                 # (1, H, W)
        if rev:
            mid = self.K // 2
            cond = np.concatenate([cond[:mid][::-1], cond[mid:mid + 1], cond[mid + 1:][::-1]], axis=0)
        cond = np.ascontiguousarray(cond[:, i:i + h, j:j + w])[None]
        x0 = np.ascontiguousarray(x0[:, i:i + h, j:j + w])
        return torch.from_numpy(cond), torch.from_numpy(x0)

    def shard_indices(self, epoch: int, rank: int, world: int, seed: int = 0) -> np.ndarray:
        """DistributedSampler(shuffle=True, drop_last=False) semantics (train.py:1002,1107)."""
        g = torch.Generator().manual_seed(seed + epoch)
        perm = torch.randperm(len(self), generator=g).numpy()
        total = -(-len(perm) // world) * world
        perm = np.concatenate([perm, perm[: total - len(perm)]])
        return perm[rank:total:world]

    def to_device(self, device) -> "DeviceEnsemble":
        return DeviceEnsemble(self, device)

    def batch(self, indices, augment: bool = True, pin: bool = False):
        """-> (cond [B,1,K,h,w], x0 [B,1,h,w])."""
        cs, xs = zip(*(self.window(int(i), augment) for i in indices))
        cond, x0 = torch.stack(cs), torch.stack(xs)
        if pin and torch.cuda.is_available():
            cond, x0 = cond.pin_memory(), x0.pin_memory()
        return cond, x0


class DeviceEnsemble:
    """The on-device data path (SURVEY 8(f) rank 3): both (T, M, H, W) arrays live in HBM (1.9 GB each at
    the full CESM2-LE shape) and a batch is assembled by ONE kernel (`cesm_gather_windows`) from a 24-byte
    per-sample plan, instead of numpy gathers on the host plus a 1.7 MB host-to-device copy per step.  The
    plan is drawn on the host by `SyntheticEnsemble.plan`, so the random stream -- and therefore every
    batch -- is identical to the host path's (`tests/test_kernels_gpu.py::test_device_data_path`)."""

    def __init__(self, ds: SyntheticEnsemble, device):
        self.ds = ds
        self.device = torch.device(device)
        self.cond = torch.from_numpy(np.ascontiguousarray(ds.cond[:, :, 0])).to(self.device)   # (T, M, H, W)
        self.tgt = torch.from_numpy(np.ascontiguousarray(ds.tgt[:, :, 0])).to(self.device)
        # pinned host plans in a ring; each slot carries the CUDA event recorded after the H2D copy that read it,
        # and the host waits on that event before rewriting the slot.  The training loop never syncs inside an
        # epoch, so without this the host can run more than a ring ahead of the stream-ordered copies and
        # overwrite a plan that has not been read yet (torn / repeated batches).
        self._plan_ring = []
        self._plan_events = []
        self._plan_dev = None
        self._turn = 0

    def plan(self, indices, augment: bool = True) -> torch.Tensor:
        """int32 [B, 6] plan in pinned host memory (one of 8 rotating buffers)."""
        B = len(indices)
        if not self._plan_ring or self._plan_ring[0].shape[0] != B:
            mk = lambda: torch.empty((B, 6), dtype=torch.int32)
            if self.device.type == "cuda":
                torch.cuda.synchronize(self.device)   # nothing may still be reading the old ring
            self._plan_ring = [mk().pin_memory() if torch.cuda.is_available() else mk() for _ in range(8)]
            self._plan_events = [None] * len(self._plan_ring)
            self._plan_dev = torch.empty((B, 6), dtype=torch.int32, device=self.device)
        slot = self._turn % len(self._plan_ring)
        host = self._plan_ring[slot]
        if self._plan_events[slot] is not None:
            self._plan_events[slot].synchronize()     # the copy issued 8 batches ago has consumed this buffer
        self._turn += 1
        host.copy_(torch.tensor([self.ds.plan(int(i), augment) for i in indices], dtype=torch.int32))
        return host

    def batch_into(self, indices, cond_out: torch.Tensor, x0_out: torch.Tensor, augment: bool = True) -> None:
        """Fill the (static) device buffers cond_out [B,1,K,h,w] / x0_out [B,1,h,w] for these sample indices."""
        from . import kernels as K
        host = self.plan(indices, augment)
        slot = (self._turn - 1) % len(self._plan_ring)
        self._plan_dev.copy_(host, non_blocking=True)
        if self.device.type == "cuda":
            ev = self._plan_events[slot] or torch.cuda.Event()
            ev.record(torch.cuda.current_stream(self.device))
            self._plan_events[slot] = ev
        K.gather_windows(self.cond, self.tgt, self._plan_dev, cond_out, x0_out)
