"""GPU tests of the DPM-Solver++(2M) sampler: the fused `dpm_step` kernel against float64 torch and against
`ddim_step`, its history handling and C-ABI argument checks, `SampleEngine(dpm_steps=N)` on an exact Gaussian
eps-predictor against a float64 chain, the real network against the fp32 reference (dpm_oracle.py), the eager
`Diffusion.dpm_sample`, weight freshness of a captured DPM graph, and `inference.py`'s DPM path."""
import numpy as np
import pytest
import torch
from torch import nn

import dpm_oracle as PO
from _parity import BASELINE_KW, rel_err
from oracle import cesm_oracle as O

pytestmark = pytest.mark.gpu

T = 1000


def _sched(steps, device):
    from cesm_emulator_b200.model import dpm_schedule
    taus, coef, next_t = dpm_schedule(O.diffusion_buffers(T)["alphas_cumprod"], steps)
    return taus, coef.to(device), next_t.to(device)


def _ref64(coef, t, x, e, hist):
    """(out, x0) in float64 from the fp32 rows; hist enters only where K1 != 0."""
    c = coef.double()[t].view(-1, 5, *([1] * (x.ndim - 1)))
    x, e = x.double(), e.double()
    x0 = c[:, 0] * x + c[:, 1] * e
    out = c[:, 2] * x + c[:, 3] * x0 + torch.where(c[:, 4] != 0, c[:, 4] * hist.double(), 0.0)
    return out, x0


@pytest.mark.parametrize("shape", [(16, 1, 192, 288), (1, 1, 7, 13), (3, 1, 33, 17)])
def test_dpm_step_kernel_matches_float64(cuda, shape):
    from cesm_emulator_b200 import kernels as K
    g = torch.Generator().manual_seed(shape[0])
    x, e, h = (torch.randn(shape, generator=g).to(cuda) for _ in range(3))
    taus, coef, next_t = _sched(50, cuda)
    pick = torch.randint(0, 50, (shape[0],), generator=g)
    pick[0] = 1                           # a second-order row
    if shape[0] > 2:
        pick[1], pick[2] = 0, 49          # the first-order first and last rows
    t = torch.tensor(taus)[pick].to(cuda)
    ref, ref_x0 = _ref64(coef, t, x, e, h)
    hist = h.clone()
    got = K.dpm_step(x, e, hist, t, coef, T)                             # out of place, no t_out
    for b in range(shape[0]):
        assert rel_err(got[b], ref[b]) < 1e-6, (t[b].item(), rel_err(got[b], ref[b]))
        assert rel_err(hist[b], ref_x0[b]) < 1e-6, (t[b].item(), rel_err(hist[b], ref_x0[b]))
    xi, hist, t_out = x.clone(), h.clone(), torch.full_like(t, -7)
    got = K.dpm_step(xi, e, hist, t, coef, T, out=xi, next_t=next_t, t_out=t_out)   # in place
    assert got.data_ptr() == xi.data_ptr()
    for b in range(shape[0]):
        assert rel_err(xi[b], ref[b]) < 1e-6, (t[b].item(), rel_err(xi[b], ref[b]))
        assert rel_err(hist[b], ref_x0[b]) < 1e-6, (t[b].item(), rel_err(hist[b], ref_x0[b]))
    assert torch.equal(t_out, next_t[t])


def test_first_order_rows_do_not_read_history(cuda):
    """A NaN-filled hist on the K1 = 0 rows (first and last step) gives a finite, correct output."""
    from cesm_emulator_b200 import kernels as K
    taus, coef, _ = _sched(10, cuda)
    g = torch.Generator().manual_seed(3)
    x, e = (torch.randn(2, 1, 24, 40, generator=g).to(cuda) for _ in range(2))
    t = torch.tensor([taus[0], taus[-1]], device=cuda)
    hist = torch.full_like(x, float("nan"))
    ref, ref_x0 = _ref64(coef, t, x, e, torch.zeros_like(x))
    got = K.dpm_step(x, e, hist, t, coef, T)
    assert torch.isfinite(got).all() and torch.isfinite(hist).all()
    for b in range(2):
        assert rel_err(got[b], ref[b]) < 1e-6 and rel_err(hist[b], ref_x0[b]) < 1e-6


def test_first_step_equals_ddim_eta_zero(cuda):
    from cesm_emulator_b200 import kernels as K
    from cesm_emulator_b200.model import ddim_schedule
    for steps in (10, 50):
        taus, coef, _ = _sched(steps, cuda)
        _, dcoef, _ = ddim_schedule(O.diffusion_buffers(T)["alphas_cumprod"], steps, 0.0)
        g = torch.Generator().manual_seed(steps)
        x, e = (torch.randn(4, 1, 64, 96, generator=g).to(cuda) for _ in range(2))
        t = torch.full((4,), taus[0], device=cuda)
        got = K.dpm_step(x, e, torch.empty_like(x), t, coef, T)
        ref = K.ddim_step(x, e, None, t, dcoef.to(cuda), T)
        assert rel_err(got, ref) < 1e-6, (steps, rel_err(got, ref))


def test_dpm_step_rejects_invalid_calls(cuda):
    from cesm_emulator_b200 import _lib
    from cesm_emulator_b200.kernels import _stream
    x, e, h = (torch.zeros(2, 1, 4, 4, device=cuda) for _ in range(3))
    t = torch.full((2,), 999, dtype=torch.long, device=cuda)
    t2 = torch.zeros_like(t)
    _, coef, next_t = _sched(10, cuda)
    p = lambda a: a.data_ptr()  # noqa: E731
    ok = [p(x), p(e), p(h), p(t), p(coef), p(next_t), p(t2), p(x), T, 2, 16, _stream()]
    _lib.call("cesm_dpm_step", *ok)
    bad = {8: 0, 9: 0, 10: 0}                                   # T, B, per_sample <= 0
    bad.update({0: None, 1: None, 2: None, 3: None, 4: None, 7: None})   # null xt, eps, hist, t, coef, out
    for i, v in bad.items():
        args = list(ok)
        args[i] = v
        with pytest.raises(_lib.CesmError):
            _lib.call("cesm_dpm_step", *args)
    for i, v in ((5, None),                                     # t_out without the next_t table
                 (6, p(t))):                                    # t_out aliasing t
        args = list(ok)
        args[i] = v
        with pytest.raises(_lib.CesmError):
            _lib.call("cesm_dpm_step", *args)
    # hist overlapping xt / out, eps, t, t_out, coef or next_t, or starting inside xt
    for v in (p(x), p(e), p(t), p(t2), p(coef), p(next_t), p(x) + 16):
        args = list(ok)
        args[2] = v
        with pytest.raises(_lib.CesmError):
            _lib.call("cesm_dpm_step", *args)


def test_dpm_step_out_of_range_t_writes_nan(cuda):
    from cesm_emulator_b200 import kernels as K
    _, coef, next_t = _sched(10, cuda)
    x = torch.ones(3, 1, 5, 5, device=cuda)
    hist = torch.zeros_like(x)
    t = torch.tensor([-1, 999, T], device=cuda)
    t_out = torch.zeros_like(t)
    y = K.dpm_step(x, x, hist, t, coef, T, next_t=next_t, t_out=t_out)
    assert torch.isnan(y[0]).all() and torch.isnan(y[2]).all() and torch.isfinite(y[1]).all()
    assert torch.isnan(hist[0]).all() and torch.isnan(hist[2]).all() and torch.isfinite(hist[1]).all()
    assert t_out.tolist() == [-1, 899, T]


class _GaussEps(nn.Module):
    """Exact eps-predictor for data ~ N(0, s^2): eps*(x, t) = sqrt(1 - ab_t) x / (ab_t s^2 + 1 - ab_t)."""

    def __init__(self, s: float):
        super().__init__()
        self.s = s
        self.anchor = nn.Parameter(torch.zeros(1))   # gives SampleEngine a device to read
        self.register_buffer("ac", O.diffusion_buffers(T)["alphas_cumprod"].clone())

    def forward(self, x, cond, t):
        a = self.ac[t].view(-1, 1, 1, 1)
        return torch.sqrt(1 - a) * x / (a * self.s * self.s + 1 - a)


@pytest.mark.parametrize("steps", [10, 50])
def test_sample_engine_dpm_on_gaussian_stub_matches_float64_chain(cuda, steps):
    from cesm_emulator_b200.engine import SampleEngine
    from cesm_emulator_b200.model import Diffusion
    s = 2.0
    d = Diffusion(_GaussEps(s)).to(cuda).eval()
    buf = {"alphas_cumprod": d.alphas_cumprod.cpu()}
    shape = (16, 1, 64, 64)
    eng = SampleEngine(d, shape, dpm_steps=steps)
    g = torch.Generator().manual_seed(steps)
    x_T = torch.randn(shape, generator=g)
    eng.x.copy_(x_T)
    eng.t.fill_(T - 1)
    eng.hist.fill_(float("nan"))
    x64, x0 = x_T.double(), None
    ac = d.alphas_cumprod.cpu().double()
    for tt in PO.dpm_timesteps(T, steps):
        eng.step()
        a = ac[tt]
        eps = torch.sqrt(1 - a) * x64 / (a * s * s + 1 - a)
        x64, x0 = PO.dpm_update(buf, x64, eps, torch.full((shape[0],), tt, dtype=torch.long), steps, x0)
    assert (eng.t == -1).all()
    assert rel_err(eng.x, x64) < 1e-5, rel_err(eng.x, x64)


def _make(cuda, kw=BASELINE_KW, seed=0):
    from cesm_emulator_b200.model import Diffusion, UNet
    torch.manual_seed(seed)
    d = Diffusion(UNet(**kw)).to(cuda)
    d.eval()
    return d


def test_sample_engine_dpm_matches_oracle(cuda):
    from cesm_emulator_b200.engine import SampleEngine
    d = _make(cuda)
    sd = {k: v.detach().float().cpu() for k, v in d.model.state_dict().items()}
    cfg, buf = O.OracleConfig.from_unet_kwargs(**BASELINE_KW), O.diffusion_buffers(T)
    g = torch.Generator().manual_seed(9)
    x = torch.randn(2, 1, 32, 32, generator=g)
    cond = torch.randn(2, 1, 32, 32, generator=g)
    h = torch.randn(2, 1, 32, 32, generator=g)
    ddim = SampleEngine(d, (2, 1, 32, 32), ddim_steps=10)
    ddim.cond.copy_(cond); ddim.x.copy_(x); ddim.t.fill_(T - 1)
    ddim.step()
    eng = SampleEngine(d, (2, 1, 32, 32), dpm_steps=10)
    assert eng.dpm_taus == [999, 899, 799, 699, 599, 499, 399, 299, 199, 99]
    # one replayed step at a mixed t vector: a first-order step and a second-order one that reads hist
    eng.cond.copy_(cond); eng.x.copy_(x); eng.t.copy_(torch.tensor([999, 399])); eng.hist.copy_(h)
    eng.step()
    assert eng.graph is not None and eng.t.tolist() == [899, 299]
    with torch.no_grad():
        ref, ref_x0 = PO.dpm_step(sd, cfg, buf, x, cond, torch.tensor([999, 399]), 10, h)
    assert rel_err(eng.x, ref) < 1e-2, rel_err(eng.x, ref)
    assert rel_err(eng.hist, ref_x0) < 1e-2, rel_err(eng.hist, ref_x0)
    # the whole N = 10 chain
    eng.x.copy_(x); eng.t.fill_(T - 1)
    for _ in range(10):
        eng.step()
    assert (eng.t == -1).all()
    ref = PO.dpm_sample(sd, cfg, buf, cond, x, 10)
    assert rel_err(eng.x, ref) < 1e-2, rel_err(eng.x, ref)
    assert eng.launches_per_step == ddim.launches_per_step > 0, (eng.launches_per_step, ddim.launches_per_step)


def test_eager_dpm_sample_matches_engine(cuda):
    from cesm_emulator_b200.engine import SampleEngine
    d = _make(cuda)
    shape = (2, 1, 32, 32)
    cond = torch.randn(shape, generator=torch.Generator().manual_seed(4)).to(cuda)
    # both draw x_T as one normal_ over `shape` on the default CUDA generator
    torch.manual_seed(11)
    y_eager = d.dpm_sample(cond, shape, cuda, steps=10)
    eng = SampleEngine(d, shape, dpm_steps=10)
    torch.manual_seed(11)
    y_eng = eng.sample(cond)
    assert torch.isfinite(y_eng).all() and (eng.t == -1).all()
    assert rel_err(y_eager, y_eng) < 1e-3, rel_err(y_eager, y_eng)
    # a second chain on the same engine must not see the history left in `hist`, even a NaN one (the UNet's
    # reductions are not bitwise reproducible run to run, hence the same bar as above)
    eng.hist.fill_(float("nan"))
    torch.manual_seed(11)
    y2 = eng.sample(cond)
    assert torch.isfinite(y2).all() and rel_err(y2, y_eng) < 1e-3, rel_err(y2, y_eng)
    with pytest.raises(ValueError):
        eng.sample(cond, steps=3)


def test_weights_stay_fresh_in_dpm_mode(cuda):
    """A DPM graph captured with one set of weights must compute with the weights a later load_state_dict wrote:
    one replayed step against the eager module with fresh operands, at a first-order and a second-order row."""
    from cesm_emulator_b200 import kernels as K
    from cesm_emulator_b200.engine import SampleEngine
    tiny = dict(BASELINE_KW, ch_mults=(1, 2))
    d, other = _make(cuda, tiny, seed=0), _make(cuda, tiny, seed=1)
    g = torch.Generator().manual_seed(1)
    x = torch.randn(2, 1, 32, 32, generator=g).to(cuda)
    c = torch.randn(2, 1, 32, 32, generator=g).to(cuda)
    h = torch.randn(2, 1, 32, 32, generator=g).to(cuda)
    t = torch.tensor([999, 499], device=cuda)
    samp = SampleEngine(d, (2, 1, 32, 32), dpm_steps=10)
    samp.sample(c)                                     # captures the graph with the first weights
    for rnd in range(2):
        if rnd == 1:
            d.load_state_dict(other.state_dict())
        samp.refresh_operands()
        samp.x.copy_(x); samp.cond.copy_(c); samp.t.copy_(t); samp.hist.copy_(h)
        samp.step()
        with torch.no_grad():
            fresh = _make(cuda, tiny, seed=5)
            fresh.load_state_dict(d.state_dict())
            eps = fresh.model(x, c, t)
            y_ref = K.dpm_step(x, eps, h.clone(), t, samp.dpm_coef, T)
        assert rel_err(samp.x, y_ref) < 1e-2, (rnd, rel_err(samp.x, y_ref))
    with torch.no_grad():
        e0, e1 = other.model(x, c, t), _make(cuda, tiny, seed=0).model(x, c, t)
    assert rel_err(e1, e0) > 5e-2


def test_inference_dpm_path(cuda):
    import inference
    d = _make(cuda, dict(BASELINE_KW, ch_mults=(1, 2)))
    cond = np.random.default_rng(0).standard_normal((2, 2, 1, 32, 32)).astype(np.float32)
    pred = inference.predict_temperature_from_emissions(d, cond, batch_size=3, dpm_steps=5, device=cuda)
    assert pred.shape == (2, 2, 32, 32) and np.isfinite(pred).all()
