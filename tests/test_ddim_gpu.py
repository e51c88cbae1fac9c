"""GPU tests of the strided DDIM sampler: the fused `ddim_step` kernel against float64 torch and against the DDPM
`p_sample` kernel, its C-ABI argument checks, `SampleEngine(ddim_steps=N)` on an exact Gaussian eps-predictor
against a float64 chain, the real network against the fp32 reference (ddim_oracle.py), the eager
`Diffusion.ddim_sample`, weight freshness of a captured DDIM graph, and `inference.py`'s DDIM path."""
import numpy as np
import pytest
import torch
from torch import nn

import ddim_oracle as DO
from _parity import BASELINE_KW, rel_err
from oracle import cesm_oracle as O

pytestmark = pytest.mark.gpu

T = 1000


def _sched(steps, eta, device):
    from cesm_emulator_b200.model import ddim_schedule
    taus, coef, next_t = ddim_schedule(O.diffusion_buffers(T)["alphas_cumprod"], steps, eta)
    return taus, coef.to(device), next_t.to(device)


def _ref64(coef, t, x, e, z):
    c = coef.double()[t].view(-1, 3, *([1] * (x.ndim - 1)))
    out = c[:, 0] * x.double() + c[:, 1] * e.double()
    return out if z is None else out + c[:, 2] * z.double()


@pytest.mark.parametrize("shape", [(16, 1, 192, 288), (1, 1, 7, 13), (3, 1, 33, 17)])
def test_ddim_step_kernel_matches_float64(cuda, shape):
    from cesm_emulator_b200 import kernels as K
    g = torch.Generator().manual_seed(shape[0])
    x, e, z = (torch.randn(shape, generator=g).to(cuda) for _ in range(3))
    for eta in (0.7, 0.0):
        taus, coef, next_t = _sched(50, eta, cuda)
        t = torch.tensor(taus, device=cuda)[torch.randint(0, 50, (shape[0],), generator=g).to(cuda)]
        zz = z if eta > 0 else None
        ref = _ref64(coef, t, x, e, zz)
        got = K.ddim_step(x, e, zz, t, coef, T)                         # out of place, no t_out
        assert rel_err(got, ref) < 1e-6, (eta, rel_err(got, ref))
        xi, t_out = x.clone(), torch.full_like(t, -7)
        got = K.ddim_step(xi, e, zz, t, coef, T, out=xi, next_t=next_t, t_out=t_out)   # in place
        assert got.data_ptr() == xi.data_ptr()
        assert rel_err(xi, ref) < 1e-6, (eta, rel_err(xi, ref))
        assert torch.equal(t_out, next_t[t])


def test_ddim_step_full_chain_eta_one_matches_p_sample(cuda):
    """N = T, eta = 1 is the DDPM posterior step: same eps and z in, p_sample's output out."""
    from cesm_emulator_b200 import kernels as K
    from cesm_emulator_b200.model import Diffusion
    d = Diffusion(nn.Identity()).to(cuda)
    _, coef, _ = _sched(T, 1.0, cuda)
    g = torch.Generator().manual_seed(1)
    x, e, z = (torch.randn(5, 1, 64, 96, generator=g).to(cuda) for _ in range(3))
    t = torch.tensor([0, 1, 37, 500, 999], device=cuda)
    ref = K.p_sample(x, e, z, t, d.betas, d.sqrt_one_minus_alphas_cumprod, d.sqrt_recip_alphas, d.posterior_variance)
    got = K.ddim_step(x, e, z, t, coef, T)
    for b in range(5):
        assert rel_err(got[b], ref[b]) < 1e-5, (t[b].item(), rel_err(got[b], ref[b]))


def test_ddim_step_rejects_invalid_calls(cuda):
    from cesm_emulator_b200 import _lib
    from cesm_emulator_b200.kernels import _stream
    x = torch.zeros(2, 1, 4, 4, device=cuda)
    t = torch.zeros(2, dtype=torch.long, device=cuda)
    t2 = torch.zeros_like(t)
    _, coef, next_t = _sched(10, 0.0, cuda)
    p = lambda a: a.data_ptr()  # noqa: E731
    ok = [p(x), p(x), None, p(t), p(coef), p(next_t), p(t2), p(x), T, 2, 16, _stream()]
    _lib.call("cesm_ddim_step", *ok)
    bad = {8: 0, 9: 0, 10: 0}                          # T, B, per_sample <= 0
    bad.update({0: None, 1: None, 3: None, 4: None, 7: None})   # null xt, eps, t, coef, out
    for i, v in bad.items():
        args = list(ok)
        args[i] = v
        with pytest.raises(_lib.CesmError):
            _lib.call("cesm_ddim_step", *args)
    args = list(ok)
    args[5] = None                                      # t_out without the next_t table
    with pytest.raises(_lib.CesmError):
        _lib.call("cesm_ddim_step", *args)
    args = list(ok)
    args[6] = p(t)                                      # t_out aliasing t
    with pytest.raises(_lib.CesmError):
        _lib.call("cesm_ddim_step", *args)


def test_ddim_step_out_of_range_t_writes_nan(cuda):
    from cesm_emulator_b200 import kernels as K
    _, coef, next_t = _sched(10, 0.0, cuda)
    x = torch.ones(3, 1, 5, 5, device=cuda)
    t = torch.tensor([-1, 999, T], device=cuda)
    t_out = torch.zeros_like(t)
    y = K.ddim_step(x, x, None, t, coef, T, next_t=next_t, t_out=t_out)
    assert torch.isnan(y[0]).all() and torch.isnan(y[2]).all() and torch.isfinite(y[1]).all()
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
@pytest.mark.parametrize("eta", [0.0, 1.0])
def test_sample_engine_ddim_on_gaussian_stub_matches_float64_chain(cuda, steps, eta):
    from cesm_emulator_b200.engine import SampleEngine
    from cesm_emulator_b200.model import Diffusion
    s = 2.0
    d = Diffusion(_GaussEps(s)).to(cuda).eval()
    buf = {"alphas_cumprod": d.alphas_cumprod.cpu()}
    shape = (16, 1, 64, 64)
    eng = SampleEngine(d, shape, ddim_steps=steps, eta=eta)
    g = torch.Generator().manual_seed(steps)
    x_T = torch.randn(shape, generator=g)
    eng.x.copy_(x_T)
    eng.t.fill_(T - 1)
    x64 = x_T.double()
    ac = d.alphas_cumprod.cpu().double()
    for tt in DO.ddim_timesteps(T, steps):
        eng.step()
        tv = torch.full((shape[0],), tt, dtype=torch.long)
        a = ac[tt]
        eps = torch.sqrt(1 - a) * x64 / (a * s * s + 1 - a)
        tp = eng.ddim_next_t.cpu()[tv]
        x64 = DO.ddim_update(buf, x64, eps, tv, tp, eta, eng.z.cpu().double() if eta > 0 else None)
    assert (eng.t == -1).all()
    assert rel_err(eng.x, x64) < 1e-5, rel_err(eng.x, x64)
    if eta == 0:  # float64 std of the discretised chain: 1.72 (N = 10), 1.94 (N = 50); the data std is s = 2
        assert abs(eng.x.std().item() - x64.std().item()) < 1e-4


def _make(cuda, kw=BASELINE_KW, seed=0):
    from cesm_emulator_b200.model import Diffusion, UNet
    torch.manual_seed(seed)
    d = Diffusion(UNet(**kw)).to(cuda)
    d.eval()
    return d


def test_sample_engine_ddim_matches_oracle(cuda):
    from cesm_emulator_b200.engine import SampleEngine
    d = _make(cuda)
    sd = {k: v.detach().float().cpu() for k, v in d.model.state_dict().items()}
    cfg, buf = O.OracleConfig.from_unet_kwargs(**BASELINE_KW), O.diffusion_buffers(T)
    g = torch.Generator().manual_seed(9)
    x = torch.randn(2, 1, 32, 32, generator=g)
    cond = torch.randn(2, 1, 32, 32, generator=g)
    ddpm = SampleEngine(d, (2, 1, 32, 32))
    ddpm.cond.copy_(cond); ddpm.x.copy_(x); ddpm.t.fill_(T - 1)
    ddpm.step()
    for eta in (1.0, 0.0):
        eng = SampleEngine(d, (2, 1, 32, 32), ddim_steps=10, eta=eta)
        assert eng.ddim_taus == [999, 899, 799, 699, 599, 499, 399, 299, 199, 99]
        # one replayed step at a mixed t vector
        eng.cond.copy_(cond); eng.x.copy_(x); eng.t.copy_(torch.tensor([999, 399]))
        eng.step()
        assert eng.graph is not None and eng.t.tolist() == [899, 299]
        with torch.no_grad():
            ref = DO.ddim_step(sd, cfg, buf, x, cond, torch.tensor([999, 399]), torch.tensor([899, 299]), eta,
                               eng.z.cpu())
        assert rel_err(eng.x, ref) < 1e-2, (eta, rel_err(eng.x, ref))
        # the whole N = 10 chain, the engine's noise handed to the reference
        eng.x.copy_(x); eng.t.fill_(T - 1)
        zs = []
        for _ in range(10):
            eng.step()
            zs.append(eng.z.cpu().clone())
        assert (eng.t == -1).all()
        ref = DO.ddim_sample(sd, cfg, buf, cond, x, 10, eta, zs)
        assert rel_err(eng.x, ref) < 1e-2, (eta, rel_err(eng.x, ref))
        assert 0 < eng.launches_per_step <= ddpm.launches_per_step, (eng.launches_per_step, ddpm.launches_per_step)


def test_eager_ddim_sample_matches_engine(cuda):
    from cesm_emulator_b200.engine import SampleEngine
    d = _make(cuda)
    shape = (2, 1, 32, 32)
    cond = torch.randn(shape, generator=torch.Generator().manual_seed(4)).to(cuda)
    # both draw x_T as one normal_ over `shape` on the default CUDA generator
    torch.manual_seed(11)
    a = torch.randn(shape, device=cuda)
    torch.manual_seed(11)
    assert torch.equal(a, torch.zeros(shape, device=cuda).normal_())
    torch.manual_seed(11)
    y_eager = d.ddim_sample(cond, shape, cuda, steps=10, eta=0.0)
    eng = SampleEngine(d, shape, ddim_steps=10)
    torch.manual_seed(11)
    y_eng = eng.sample(cond)
    assert torch.isfinite(y_eng).all() and (eng.t == -1).all()
    assert rel_err(y_eager, y_eng) < 1e-3, rel_err(y_eager, y_eng)
    with pytest.raises(ValueError):
        eng.sample(cond, steps=3)


def test_weights_stay_fresh_in_ddim_mode(cuda):
    """A DDIM graph captured with one set of weights must compute with the weights a later load_state_dict wrote:
    one replayed step against the eager module with fresh operands, fed the replay's noise."""
    from cesm_emulator_b200 import kernels as K
    from cesm_emulator_b200.engine import SampleEngine
    tiny = dict(BASELINE_KW, ch_mults=(1, 2))
    d, other = _make(cuda, tiny, seed=0), _make(cuda, tiny, seed=1)
    g = torch.Generator().manual_seed(1)
    x = torch.randn(2, 1, 32, 32, generator=g).to(cuda)
    c = torch.randn(2, 1, 32, 32, generator=g).to(cuda)
    t = torch.tensor([999, 499], device=cuda)
    samp = SampleEngine(d, (2, 1, 32, 32), ddim_steps=10, eta=1.0)
    samp.sample(c)                                     # captures the graph with the first weights
    for rnd in range(2):
        if rnd == 1:
            d.load_state_dict(other.state_dict())
        samp.refresh_operands()
        samp.x.copy_(x); samp.cond.copy_(c); samp.t.copy_(t)
        samp.step()
        with torch.no_grad():
            fresh = _make(cuda, tiny, seed=5)
            fresh.load_state_dict(d.state_dict())
            eps = fresh.model(x, c, t)
            y_ref = K.ddim_step(x, eps, samp.z, t, samp.ddim_coef, T)
        assert rel_err(samp.x, y_ref) < 1e-2, (rnd, rel_err(samp.x, y_ref))
    # the two weight sets really differ (same x and z would otherwise give nearly the same step)
    with torch.no_grad():
        e0, e1 = other.model(x, c, t), _make(cuda, tiny, seed=0).model(x, c, t)
    assert rel_err(e1, e0) > 5e-2


def test_inference_ddim_path(cuda):
    import inference
    d = _make(cuda, dict(BASELINE_KW, ch_mults=(1, 2)))
    cond = np.random.default_rng(0).standard_normal((2, 2, 1, 32, 32)).astype(np.float32)
    pred = inference.predict_temperature_from_emissions(d, cond, batch_size=3, ddim_steps=5, device=cuda)
    assert pred.shape == (2, 2, 32, 32) and np.isfinite(pred).all()
    pred1 = inference.predict_temperature_from_emissions(d, cond, batch_size=3, ddim_steps=5, eta=1.0, device=cuda)
    assert pred1.shape == (2, 2, 32, 32) and np.isfinite(pred1).all()
