"""CPU tests of the host-side logic: config overrides, the synthetic ensemble / sharding, and the
gradient-bucket all-reduce (world_size 2 over gloo)."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_config_load_and_overrides():
    sys.path.insert(0, ROOT)
    import utils_conf
    for name, mults, crop, bs in (("baseline", [1, 2, 4], [128, 128], 2), ("more_blocks", [1, 2, 4, 8], [64, 64], 64)):
        cfg = utils_conf.load_config(os.path.join(ROOT, "config", name))  # extension-less JSON (utils_conf.py:8-17)
        assert cfg["unet"]["ch_mults"] == mults and cfg["dataset"]["crop_hw"] == crop
        assert cfg["train"]["batch_size"] == bs and cfg["dataset"]["K"] == 3
        assert cfg["unet"]["base_ch"] == 64 and cfg["unet"]["groups"] == 8
    utils_conf.apply_overrides(cfg, ["train.batch_size=4", "unet.use_checkpoint=false", "train.lr=2.5e-4", "x.y.z=abc",
                                     "train.max_grad_norm=1.0"])
    assert cfg["train"]["batch_size"] == 4 and cfg["unet"]["use_checkpoint"] is False
    assert cfg["x"]["y"]["z"] == "abc" and cfg["train"]["max_grad_norm"] == 1.0
    assert cfg["train"]["lr"] == 2.5e-4
    with pytest.raises(ValueError):
        utils_conf.apply_overrides(cfg, ["novalue"])
    with pytest.raises(FileNotFoundError):
        utils_conf.load_config(os.path.join(ROOT, "config", "nope"))


def test_synthetic_ensemble_shapes_and_windows():
    from cesm_emulator_b200.synthetic import SyntheticEnsemble
    ds = SyntheticEnsemble(members=3, times=7, lat=16, lon=24, seed=1, K=3, crop_hw=(8, 8))
    assert ds.cond_mtllc.shape == (3, 7, 16, 24, 1)                      # (member, time, lat, lon, channel)
    assert ds.cond.shape == ds.tgt.shape == (7, 3, 1, 16, 24)            # reference layout (T, M, 1, H, W)
    assert abs(float(ds.tgt.mean())) < 1e-3 and abs(float(ds.tgt.std()) - 1) < 1e-3   # global z-score
    assert len(ds) == (7 - 3 + 1) * 3                                     # consecutive windows x members
    cond, x0 = ds.window(7, augment=False)                                # idx 7 -> member 1, start 2, anchor 3
    assert cond.shape == (1, 3, 8, 8) and x0.shape == (1, 8, 8) and cond.dtype == torch.float32
    assert np.array_equal(cond[0].numpy(), ds.cond[2:5, 1, 0, 4:12, 8:16])
    assert np.array_equal(x0.numpy(), ds.tgt[3, 1, :, 4:12, 8:16])
    c, x = ds.batch([0, 1, 2, 3])
    assert c.shape == (4, 1, 3, 8, 8) and x.shape == (4, 1, 8, 8)
    with pytest.raises(ValueError):
        SyntheticEnsemble(members=1, times=4, lat=8, lon=8, K=1)
    # DistributedSampler semantics: ranks partition a seeded permutation, padded to equal length
    a, b = ds.shard_indices(3, 0, 2), ds.shard_indices(3, 1, 2)
    assert len(a) == len(b) == 8 and set(a) | set(b) == set(range(15))
    assert not np.array_equal(ds.shard_indices(4, 0, 2), a)


def _bucket_worker(rank, world, port, q):
    import torch.distributed as dist
    from cesm_emulator_b200.engine import GradBuckets
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        torch.manual_seed(0)  # identical weights on every rank
        net = torch.nn.Sequential(torch.nn.Linear(6, 16), torch.nn.Tanh(), torch.nn.Linear(16, 16), torch.nn.Tanh(),
                                  torch.nn.Linear(16, 1))
        buckets = GradBuckets(net, n_buckets=3)
        assert buckets.n_buckets >= 2 and buckets.world == world
        torch.manual_seed(100 + rank)  # different data per rank
        x = torch.randn(5, 6)
        buckets.begin_step()
        # engine mode: a parameter whose gradient is written directly reports through ready() AND torch runs its
        # post-accumulate hook as well (seen on 2 B200s: buckets were all-reduced after half of their gradients).
        # Emulate the double report: a backward hook on the first layer's output calls ready() for the LAST
        # layer's parameters right after autograd accumulated them -- they must be counted once.
        last = list(net[4].parameters())
        def report_again(*_):
            for p in last:
                buckets.ready(p)

        h = net[2].register_full_backward_hook(report_again)
        (net(x).pow(2).mean() / world).backward()   # mean over ranks == sum of (loss / world)
        h.remove()
        assert buckets._pending == [0] * buckets.n_buckets, buckets._pending
        buckets.finish_step()
        norm = buckets.clip_(1e9)
        # the flat buffer pads every tensor to a 64-byte boundary: compare the per-parameter views.  numpy copies:
        # a tensor is passed as a file descriptor that the parent fetches from this process, which may have exited
        q.put((rank, torch.cat([p.grad.reshape(-1) for p in buckets.params]).numpy(), x.numpy(), float(norm)))
    finally:
        dist.destroy_process_group()


def test_grad_buckets_allreduce_world2_gloo():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    procs = [ctx.Process(target=_bucket_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=120) for _ in procs], key=lambda t: t[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    (_, g0, x0, n0), (_, g1, x1, n1) = res
    g0, x0, g1, x1 = (torch.from_numpy(a) for a in (g0, x0, g1, x1))
    assert torch.equal(g0, g1)  # every rank holds the same averaged gradient
    # single-process run over the concatenated batch gives the same gradient (mean over both halves)
    from cesm_emulator_b200.engine import _ready_order
    torch.manual_seed(0)
    net = torch.nn.Sequential(torch.nn.Linear(6, 16), torch.nn.Tanh(), torch.nn.Linear(16, 16), torch.nn.Tanh(),
                              torch.nn.Linear(16, 1))
    (0.5 * net(x0).pow(2).mean() + 0.5 * net(x1).pow(2).mean()).backward()
    ref = torch.cat([p.grad.reshape(-1) for _, p in _ready_order(net.named_parameters())])
    assert torch.allclose(g0, ref, rtol=1e-5, atol=1e-7)
    assert abs(n0 - ref.norm().item()) < 1e-5 * max(1.0, ref.norm().item())


def test_window_plan_and_frame_map_match_the_host_gather():
    """The on-device data path is driven by `SyntheticEnsemble.plan` and a frame map evaluated inside
    cesm_gather_windows; restated here in numpy (same formula as the kernel: left and right halves around
    the centre flipped) it must reproduce `window()` for every K, with and without crops."""
    from cesm_emulator_b200.synthetic import SyntheticEnsemble

    def gather(ds, plan):
        m, t0, ta, i0, j0, rev = plan
        h, w = ds.out_hw()
        K, mid = ds.K, ds.K // 2
        src = [(mid - 1 - k if k < mid else (mid if k == mid else K + mid - k)) if rev else k for k in range(K)]
        cond = np.stack([ds.cond[t0 + s, m, 0, i0:i0 + h, j0:j0 + w] for s in src])[None]
        return cond, ds.tgt[ta, m, :, i0:i0 + h, j0:j0 + w]

    for K, crop in ((2, None), (3, (8, 8)), (4, (6, 10)), (5, None), (7, (8, 12))):
        kw = dict(members=3, times=12, lat=12, lon=16, seed=3, K=K, crop_hw=crop, time_reverse_p=0.6)
        a, b = SyntheticEnsemble(**kw), SyntheticEnsemble(**kw)   # two identical random streams
        flips = 0
        for idx in list(range(len(a)))[::2]:
            plan = a.plan(idx)
            cond, x0 = b.window(idx)
            gc, gx = gather(a, plan)
            assert np.array_equal(cond.numpy(), gc) and np.array_equal(x0.numpy(), gx)
            assert plan[0] == idx % a.M and plan[1] == idx // a.M and plan[2] == min(plan[1] + K // 2, a.T - 1)
            flips += plan[5]
        assert flips > 0
        assert a.plan(5, augment=False)[3:] == (((a.H - a.out_hw()[0]) // 2, (a.W - a.out_hw()[1]) // 2, 0))


# ------------------------------------------------------------------------------------------------
# the data path pinned to the REFERENCE's dataset class (fixture: tests/golden/make_dataset_golden.py)
# ------------------------------------------------------------------------------------------------
def _dataset_fixture():
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "dataset_windows.npz"))
    T, M, H, W = (int(v) for v in g["shape"])
    rng = np.random.default_rng(int(g["seed"]))
    cond = rng.standard_normal((T, M, 1, H, W)).astype(np.float32)
    tgt = rng.standard_normal((T, M, 1, H, W)).astype(np.float32)
    return g, cond, tgt


class _ScriptedDraws:
    """Stands in for the augmentation generator: replays crop origins (and 'never reverse')."""

    def __init__(self, origins):
        self.vals = [int(v) for ij in origins for v in ij]

    def random(self):
        return 1.0

    def integers(self, lo, hi):
        v = self.vals.pop(0)
        assert lo <= v < hi
        return v


def test_windows_match_reference_dataset_class():
    """`SyntheticEnsemble.window` returns what WindowedAllMembersDataset_random (dataset_single_member.py:168-196,
    the class train.py:990 builds) returns for the same arrays: indexing, centre target, centre-preserving time
    reversal, centre / clamped / random crops (the random origins replayed from the reference's own draws)."""
    from cesm_emulator_b200.synthetic import SyntheticEnsemble
    g, cond, tgt = _dataset_fixture()

    def all_windows(ds, augment):
        cs, xs = zip(*(ds.window(i, augment) for i in range(len(ds))))
        return np.stack([c.numpy() for c in cs]), np.stack([x.numpy() for x in xs])

    for K in (3, 4, 5):
        ds = SyntheticEnsemble.from_arrays(cond, tgt, K=K, time_reverse_p=0.0)
        assert len(ds) == g[f"plain_K{K}_cond"].shape[0]
        c, x = all_windows(ds, True)
        assert np.array_equal(c, g[f"plain_K{K}_cond"]) and np.array_equal(x, g[f"plain_K{K}_x0"])
        ds = SyntheticEnsemble.from_arrays(cond, tgt, K=K, time_reverse_p=1.0)
        c, x = all_windows(ds, True)
        assert np.array_equal(c, g[f"rev_K{K}_cond"]) and np.array_equal(x, g[f"rev_K{K}_x0"])
    ds = SyntheticEnsemble.from_arrays(cond, tgt, K=3, crop_hw=(8, 10), time_reverse_p=0.0)
    c, x = all_windows(ds, False)     # augment=False = the reference's crop_mode="center"
    assert np.array_equal(c, g["center_crop_cond"]) and np.array_equal(x, g["center_crop_x0"])
    ds = SyntheticEnsemble.from_arrays(cond, tgt, K=3, crop_hw=(64, 10), time_reverse_p=0.0)
    c, x = all_windows(ds, False)
    assert np.array_equal(c, g["clamped_crop_cond"]) and np.array_equal(x, g["clamped_crop_x0"])
    ds = SyntheticEnsemble.from_arrays(cond, tgt, K=3, crop_hw=(8, 10), time_reverse_p=0.5)
    ds._aug = _ScriptedDraws(g["random_crop_origin"])
    c, x = all_windows(ds, True)
    assert np.array_equal(c, g["random_crop_cond"]) and np.array_equal(x, g["random_crop_x0"])
    with pytest.raises(ValueError):
        SyntheticEnsemble.from_arrays(cond, tgt[:-1])
    with pytest.raises(ValueError):
        SyntheticEnsemble.from_arrays(cond, tgt, K=1)


def test_prediction_netcdf_product(tmp_path):
    """inference.py:260-281: variable name, dims, coordinates and attributes of the output file."""
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from scipy.io import netcdf_file
    from inference import write_prediction_netcdf
    pred = np.random.default_rng(0).standard_normal((3, 2, 4, 6)).astype(np.float32)
    path = str(tmp_path / "out" / "pred.nc")
    write_prediction_netcdf(path, pred, stack_coord=[1850, 1851, 1852], lat=np.linspace(-90, 90, 4),
                            attrs={"cond_var": "CO2_em_anthro"})
    with netcdf_file(path, "r", mmap=False) as f:
        v = f.variables["TREFHT_pred"]
        assert v.dimensions == ("year", "member_id", "lat", "lon")
        assert np.array_equal(v[:], pred)
        assert v.units == b"standardized" and v.cond_var == b"CO2_em_anthro"
        assert list(f.variables["year"][:]) == [1850, 1851, 1852]
        assert np.allclose(f.variables["lat"][:], np.linspace(-90, 90, 4))
        assert list(f.variables["member_id"][:]) == [0, 1] and f.variables["lon"].shape == (6,)
    with pytest.raises(ValueError):
        write_prediction_netcdf(path, pred, lat=[0.0, 1.0])


def test_layernorm_fold_algebra_and_in_place_refresh():
    """ops._fold_f1(gamma=...) builds the operands of the one-kernel one-frame temporal block (cesm_igemm ln_colsum):
    x + LN(x) (W_out W_v)^T  ==  x + rstd (x (W gamma)^T - mean colsum).  The tensors are rebuilt IN PLACE when the
    weights change (their addresses are baked into captured graphs)."""
    import types
    from cesm_emulator_b200 import ops
    torch.manual_seed(0)
    C, hidden, eps = 64, 256, 1e-5
    wqkv = torch.nn.Parameter(torch.randn(3 * hidden, C) * 0.05)
    wout = torch.nn.Parameter(torch.randn(C, hidden) * 0.05)
    gamma = torch.nn.Parameter(1.0 + 0.1 * torch.randn(1, C, 1, 1, 1))
    meta = types.SimpleNamespace()
    wln, colsum = ops._fold_f1(meta, wqkv, wout, hidden, C, gamma=gamma)
    x = torch.randn(50, C) * 1.3 + 0.4

    def want():
        mu, var = x.mean(-1, keepdim=True), x.var(-1, unbiased=False, keepdim=True)
        ln = (x - mu) / (var + eps).sqrt() * gamma.detach().reshape(1, C)
        return x + ln @ (wout.detach() @ wqkv.detach()[2 * hidden:]).t()

    def got():
        mu, var = x.mean(-1, keepdim=True), x.var(-1, unbiased=False, keepdim=True)
        return x + (var + eps).rsqrt() * (x @ wln.float().t() - mu * colsum[None, :])

    assert (got() - want()).abs().max() < 5e-3 * want().abs().max()          # fp16 rounding of W gamma
    assert torch.allclose(colsum, wln.float().sum(1))
    ptrs = (wln.data_ptr(), colsum.data_ptr())
    with torch.no_grad():
        wout.mul_(1.5)                     # in-place update bumps the version -> the fold key changes
    ops.refresh_folds()
    wln2, colsum2 = ops._fold_f1(meta, wqkv, wout, hidden, C, gamma=gamma)
    assert (wln2.data_ptr(), colsum2.data_ptr()) == ptrs
    assert (got() - want()).abs().max() < 5e-3 * want().abs().max()
