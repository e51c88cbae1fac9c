import json, os, sys
import torch, torch.distributed as dist
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
from _parity import BASELINE_KW, rel_err
from cesm_emulator_b200 import ops
from cesm_emulator_b200.engine import TrainEngine
from cesm_emulator_b200.model import Diffusion, UNet
rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local); dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
solo = [dist.new_group([r]) for r in range(world)][rank]
B, K, H, W = 1, 3, 32, 48
g = torch.Generator().manual_seed(100)
x0_all = torch.randn(world * B, 1, H, W, generator=g); cond_all = torch.randn(world * B, 1, K, H, W, generator=g)
t_all = torch.randint(0, 1000, (world * B,), generator=g); noise_all = torch.randn(world * B, 1, H, W, generator=g)
mine = slice(rank * B, (rank + 1) * B)
def grads_of(pg, sl, batch, n_buckets=4, sync=False):
    torch.manual_seed(0)
    m = Diffusion(UNet(**BASELINE_KW)).to(dev); m.train()
    e = TrainEngine(m, (batch, 1, H, W), (batch, 1, K, H, W), lr=0.0, weight_decay=0.0, max_grad_norm=None, use_graph=False, process_group=pg, n_buckets=n_buckets)
    if sync:
        orig = e.buckets._on_grad
        def synced(p):
            torch.cuda.synchronize(); orig(p); torch.cuda.synchronize()
        e.buckets._on_grad = synced
        for h in e.buckets._hooks: h.remove()
        e.buckets._hooks = [p.register_post_accumulate_grad_hook(synced) for p in e.buckets.params]
    plain = m.loss
    t, nz = t_all[sl].to(dev), noise_all[sl].to(dev)
    m.loss = lambda x, c: plain(x, c, t=t, noise=nz)
    e.step(x0_all[sl], cond_all[sl])
    torch.cuda.synchronize()
    S = float(e.opt.loss_scale)
    gr = {k: (p.grad / S).clone() for k, p in m.named_parameters() if p.requires_grad}
    info = {"bounds": e.buckets.bounds, "pending_init": e.buckets._pending_init, "pending_end": e.buckets._pending}
    for h in e.buckets._hooks: h.remove()
    ops.set_grad_sink(None)
    return gr, info
g_one, _ = grads_of(solo, slice(0, world * B), world * B)
for tag, kw in [("default", {}), ("sync", {"sync": True}), ("1bucket", {"n_buckets": 1})]:
    gd, info = grads_of(None, mine, B, **kw)
    errs = {k: rel_err(gd[k], g_one[k]) for k in g_one}
    bad = [k for k in errs if errs[k] > 1e-2]
    zero = [k for k in bad if float(gd[k].norm()) == 0.0]
    if rank == 0:
        print(tag, "bad", len(bad), "zero", len(zero), info, flush=True)
torch.cuda.synchronize(); dist.barrier(); os._exit(0)
