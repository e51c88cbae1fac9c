"""GPU tests of seeded, shard-invariant ensemble generation: `field_normal` against the numpy Philox oracle, its
invariance to the row and batch and its statistics; the fused `p_sample_seeded` / `ddim_step_seeded` kernels against
the unfused ones fed the same draw, bit for bit, and their C-ABI checks; seeded `SampleEngine` chains on an exact
Gaussian eps-predictor and on the real network (row / batch invariance, graph against eager, torch's generator left
alone, weight freshness); and `inference.py --seed` across batch sizes."""
import numpy as np
import pytest
import torch
from scipy import stats
from torch import nn

import philox_oracle as PO
from _parity import BASELINE_KW, rel_err
from oracle import cesm_oracle as O

pytestmark = pytest.mark.gpu

T = 1000
SEED = 0x5EED_0000_CE5E


def _ids(v, cuda):
    return torch.tensor(v, dtype=torch.int64, device=cuda)


def _diffusion(cuda):
    from cesm_emulator_b200.model import Diffusion
    return Diffusion(nn.Identity()).to(cuda)


# ---- 1-3: the draw itself -------------------------------------------------------------------------
@pytest.mark.parametrize("hw", [(7, 13), (33, 17), (64, 96)])
def test_field_normal_matches_oracle(cuda, hw):
    from cesm_emulator_b200 import kernels as K
    ids = [0, 3, (1 << 32) + 5, (1 << 62) + 12345]
    worst = 0.0
    for seed in (0, 1, SEED, (1 << 64) - 1):
        for draw in (0, 999, PO.X_T_DRAW):
            got = K.field_normal(seed, _ids(ids, cuda), draw, (len(ids), 1, *hw)).cpu().numpy()
            for r, f in enumerate(ids):
                ref = PO.field_normal(seed, f, draw, hw[0] * hw[1])
                worst = max(worst, float(np.abs(got[r].reshape(-1) - ref).max()))
    print(f"field_normal vs float64 oracle at {hw}: max abs diff {worst:.3g}")
    assert worst <= 2e-6, worst


@pytest.mark.parametrize("hw", [(33, 17), (64, 96)])
def test_field_normal_is_row_and_batch_invariant(cuda, hw):
    from cesm_emulator_b200 import kernels as K
    both = K.field_normal(SEED, _ids([5, 9, 2], cuda), 17, (3, 1, *hw))
    for r, f in enumerate([5, 9, 2]):
        alone = K.field_normal(SEED, _ids([f], cuda), 17, (1, 1, *hw))
        assert torch.equal(both[r], alone[0]), f


def test_field_normal_statistics(cuda):
    from cesm_emulator_b200 import kernels as K
    B, H, W = 16, 192, 288
    ids = _ids(list(range(100, 100 + B)), cuda)
    z = K.field_normal(SEED, ids, 500, (B, 1, H, W)).double().view(B, -1)
    zp = K.field_normal(SEED, ids, 499, (B, 1, H, W)).double().view(B, -1)
    n = z.numel()
    assert abs(z.mean().item()) < 5 / n ** 0.5
    assert abs(z.var().item() - 1) < 5 * (2 / n) ** 0.5
    ks = stats.kstest(z.cpu().numpy().reshape(-1), "norm")
    assert ks.pvalue > 1e-3, ks

    def corr(a, b):
        a, b = a - a.mean(), b - b.mean()
        return ((a * b).mean() / (a.std() * b.std())).item()
    bar = lambda m: 5 / m ** 0.5  # noqa: E731
    c_fields = corr(z[:-1].reshape(-1), z[1:].reshape(-1))                  # field b against field b+1
    c_draws = corr(z.reshape(-1), zp.reshape(-1))                            # draw t against draw t-1
    c_adj = corr(z[:, :-1].reshape(-1), z[:, 1:].reshape(-1))                # element e against e+1
    print(f"corr fields {c_fields:.2e} draws {c_draws:.2e} adjacent {c_adj:.2e}; KS p {ks.pvalue:.3f}; "
          f"max |z| {z.abs().max().item():.3f}")
    assert abs(c_fields) < bar((B - 1) * H * W) and abs(c_draws) < bar(n) and abs(c_adj) < bar(B * (H * W - 1))
    assert z.abs().max().item() < 7


# ---- 4: fused against unfused ---------------------------------------------------------------------
def _per_row_draw(seed, ids, t, shape, cuda):
    from cesm_emulator_b200 import kernels as K
    z = torch.empty(shape, device=cuda)
    for b in range(shape[0]):
        K.field_normal(seed, ids[b:b + 1], int(t[b]), out=z[b:b + 1])
    return z


@pytest.mark.parametrize("hw", [(33, 17), (64, 96)])
def test_fused_p_sample_equals_unfused(cuda, hw):
    from cesm_emulator_b200 import kernels as K
    d = _diffusion(cuda)
    g = torch.Generator().manual_seed(3)
    shape = (5, 1, *hw)
    x, e = (torch.randn(shape, generator=g).to(cuda) for _ in range(2))
    t = _ids([0, 1, 37, 500, 999], cuda)
    ids = _ids([7, 7, 1 << 33, 2, 0], cuda)
    z = _per_row_draw(SEED, ids, t.tolist(), shape, cuda)
    tabs = (d.betas, d.sqrt_one_minus_alphas_cumprod, d.sqrt_recip_alphas, d.posterior_variance)
    ref = K.p_sample(x, e, z, t, *tabs)
    got = K.p_sample_seeded(x, e, SEED, ids, t, *tabs)
    assert torch.equal(got, ref)
    xi = x.clone()
    K.p_sample_seeded(xi, e, SEED, ids, t, *tabs, out=xi)                   # in place
    assert torch.equal(xi, ref)
    assert torch.equal(got[0], K.p_sample(x, e, torch.zeros_like(z), t, *tabs)[0])   # t = 0 adds no noise


@pytest.mark.parametrize("hw", [(33, 17), (64, 96)])
def test_fused_ddim_step_equals_unfused(cuda, hw):
    from cesm_emulator_b200 import kernels as K
    from cesm_emulator_b200.model import ddim_schedule
    g = torch.Generator().manual_seed(4)
    shape = (4, 1, *hw)
    x, e = (torch.randn(shape, generator=g).to(cuda) for _ in range(2))
    for steps in (T, 20):
        taus, coef, next_t = ddim_schedule(O.diffusion_buffers(T)["alphas_cumprod"], steps, 1.0)
        coef, next_t = coef.to(cuda), next_t.to(cuda)
        t = _ids([taus[0], taus[len(taus) // 2], taus[-2], taus[-1]], cuda)   # the last one is t = 0 for N = T
        ids = _ids([3, 1 << 40, 3, 11], cuda)
        z = _per_row_draw(SEED, ids, t.tolist(), shape, cuda)
        ref = K.ddim_step(x, e, z, t, coef, T)
        t_ref = next_t[t]
        xi, t_out = x.clone(), torch.full_like(t, -7)
        K.ddim_step_seeded(xi, e, SEED, ids, t, coef, T, out=xi, next_t=next_t, t_out=t_out)
        assert torch.equal(xi, ref) and torch.equal(t_out, t_ref), steps
        assert torch.equal(K.ddim_step_seeded(x, e, SEED, ids, t, coef, T), ref)


def test_seeded_steps_bad_t_give_nan_and_pass_t_through(cuda):
    from cesm_emulator_b200 import kernels as K
    from cesm_emulator_b200.model import ddim_schedule
    d = _diffusion(cuda)
    _, coef, next_t = ddim_schedule(d.alphas_cumprod, 10, 1.0)
    coef, next_t = coef.to(cuda), next_t.to(cuda)
    x = torch.ones(3, 1, 5, 5, device=cuda)
    t = _ids([-1, 999, T], cuda)
    ids = _ids([0, 1, 2], cuda)
    t_out = torch.zeros_like(t)
    y = K.ddim_step_seeded(x, x, 1, ids, t, coef, T, next_t=next_t, t_out=t_out)
    assert torch.isnan(y[0]).all() and torch.isnan(y[2]).all() and torch.isfinite(y[1]).all()
    assert t_out.tolist() == [-1, 899, T]
    y = K.p_sample_seeded(x, x, 1, ids, t, d.betas, d.sqrt_one_minus_alphas_cumprod, d.sqrt_recip_alphas,
                          d.posterior_variance)
    assert torch.isnan(y[0]).all() and torch.isnan(y[2]).all() and torch.isfinite(y[1]).all()


def test_seeded_c_abi_rejects_invalid_calls(cuda):
    from cesm_emulator_b200 import _lib
    from cesm_emulator_b200.kernels import _stream
    d = _diffusion(cuda)
    x = torch.zeros(2, 1, 4, 4, device=cuda)
    t = torch.zeros(2, dtype=torch.long, device=cuda)
    ids, t2 = torch.zeros_like(t), torch.zeros_like(t)
    coef = torch.zeros(T, 3, device=cuda)
    next_t = torch.zeros(T, dtype=torch.long, device=cuda)
    p = lambda a: a.data_ptr()  # noqa: E731

    def check(name, ok, bad):
        _lib.call(name, *ok)
        for i, v in bad:
            args = list(ok)
            args[i] = v
            with pytest.raises(_lib.CesmError):
                _lib.call(name, *args)

    check("cesm_field_normal", [1, 2, p(ids), 5, p(x), 2, 16, _stream()],
          [(2, None), (4, None), (5, 0), (5, 65536), (6, 0), (6, -3)])
    check("cesm_p_sample_seeded",
          [p(x), p(x), 1, 2, p(ids), p(t), p(d.betas), p(d.sqrt_one_minus_alphas_cumprod), p(d.sqrt_recip_alphas),
           p(d.posterior_variance), p(x), T, 2, 16, _stream()],
          [(0, None), (1, None), (4, None), (5, None), (6, None), (7, None), (8, None), (9, None), (10, None),
           (11, 0), (12, 0), (13, 0)])
    check("cesm_ddim_step_seeded",
          [p(x), p(x), 1, 2, p(ids), p(t), p(coef), p(next_t), p(t2), p(x), T, 2, 16, _stream()],
          [(0, None), (1, None), (4, None), (5, None), (6, None), (9, None), (10, 0), (11, 0), (12, 0),
           (7, None),                                    # t_out without the next_t table
           (8, p(t)), (8, p(ids))])                      # t_out aliasing t or field_ids


# ---- 5: exact Gaussian eps-predictor ------------------------------------------------------------------
class _GaussEps(nn.Module):
    """Exact eps-predictor for data ~ N(0, s^2): eps*(x, t) = sqrt(1 - ab_t) x / (ab_t s^2 + 1 - ab_t)."""

    def __init__(self, s: float):
        super().__init__()
        self.s = s
        self.anchor = nn.Parameter(torch.zeros(1))
        self.register_buffer("ac", O.diffusion_buffers(T)["alphas_cumprod"].clone())

    def forward(self, x, cond, t):
        a = self.ac[t].view(-1, 1, 1, 1)
        return torch.sqrt(1 - a) * x / (a * self.s * self.s + 1 - a)


MODES = {"ddpm": dict(), "ddim_eta1": dict(ddim_steps=10, eta=1.0), "dpm": dict(dpm_steps=10)}


@pytest.mark.parametrize("mode", list(MODES))
def test_seeded_field_is_bit_identical_across_rows_and_batches(cuda, mode):
    from cesm_emulator_b200.engine import SampleEngine
    from cesm_emulator_b200.model import Diffusion
    d = Diffusion(_GaussEps(2.0)).to(cuda).eval()
    steps = 50 if mode == "ddpm" else None
    hw = (33, 17)
    a = SampleEngine(d, (4, 1, *hw), seed=SEED, **MODES[mode])
    b = SampleEngine(d, (2, 1, *hw), seed=SEED, **MODES[mode])
    ya = a.sample(torch.zeros(4, 1, *hw, device=cuda), steps=steps, field_ids=[5, 9, 2, 9])
    yb = b.sample(torch.zeros(2, 1, *hw, device=cuda), steps=steps, field_ids=[9, 5])
    assert torch.isfinite(ya).all() and not torch.equal(ya[0], ya[1])
    assert torch.equal(ya[0], yb[1]) and torch.equal(ya[1], yb[0]) and torch.equal(ya[3], yb[0])
    yc = b.sample(torch.zeros(2, 1, *hw, device=cuda), steps=steps)   # default ids arange(B)
    yd = a.sample(torch.zeros(4, 1, *hw, device=cuda), steps=steps, field_ids=[1, 1, 0, 0])
    assert torch.equal(yc[0], yd[2]) and torch.equal(yc[1], yd[0])


def test_seeded_ddpm_chain_equals_ddim_full_eta_one(cuda):
    """DDIM with N = T and eta = 1 is the DDPM posterior step, and both draw z with id t: same chain."""
    from cesm_emulator_b200.engine import SampleEngine
    from cesm_emulator_b200.model import Diffusion
    d = Diffusion(_GaussEps(2.0)).to(cuda).eval()
    shape = (3, 1, 64, 64)
    cond = torch.zeros(shape, device=cuda)
    ddpm = SampleEngine(d, shape, seed=SEED).sample(cond, field_ids=[4, 8, 15])
    ddim = SampleEngine(d, shape, ddim_steps=T, eta=1.0, seed=SEED).sample(cond, field_ids=[4, 8, 15])
    err = rel_err(ddim, ddpm)
    print(f"seeded DDPM vs DDIM(N=T, eta=1): rel err {err:.3g}")
    assert err < 1e-5, err


# ---- 6: the real network --------------------------------------------------------------------------
def _make(cuda, kw=BASELINE_KW, seed=0):
    from cesm_emulator_b200.model import Diffusion, UNet
    torch.manual_seed(seed)
    d = Diffusion(UNet(**kw)).to(cuda)
    d.eval()
    return d


@pytest.mark.parametrize("mode", list(MODES))
def test_real_network_field_does_not_depend_on_row_or_batch(cuda, mode):
    from cesm_emulator_b200.engine import SampleEngine
    d = _make(cuda)
    kw = {"ddpm": dict(), "ddim_eta1": dict(ddim_steps=20, eta=1.0), "dpm": dict(dpm_steps=10)}[mode]
    g = torch.Generator().manual_seed(2)
    c = torch.randn(1, 1, 32, 32, generator=g).to(cuda)
    other = torch.randn(3, 1, 32, 32, generator=g).to(cuda)
    a = SampleEngine(d, (4, 1, 32, 32), seed=SEED, **kw)
    b = SampleEngine(d, (2, 1, 32, 32), seed=SEED, **kw)
    ya = a.sample(torch.cat([other[:2], c, c]), field_ids=[1, 2, 40, 41])
    yb = b.sample(torch.cat([c, other[2:]]), field_ids=[40, 7])
    err = rel_err(ya[2], yb[0])
    spread = rel_err(ya[3], ya[2])
    print(f"{mode}: same field at rows 2 / 0 of batches 4 / 2: rel err {err:.3g}; two ids, same condition: {spread:.3g}")
    assert err < 1e-2, err
    assert spread > 0.5, spread


def test_graph_matches_eager_and_leaves_torch_rng_alone(cuda):
    from cesm_emulator_b200.engine import SampleEngine
    d = _make(cuda)
    shape = (3, 1, 32, 32)
    cond = torch.randn(shape, generator=torch.Generator().manual_seed(4)).to(cuda)
    ids = [11, 1 << 35, 11]
    y_eager = d.ddim_sample(cond, shape, cuda, steps=10, eta=1.0, seed=SEED, field_ids=ids)
    eng = SampleEngine(d, shape, ddim_steps=10, eta=1.0, seed=SEED)
    state = torch.cuda.get_rng_state()
    y_eng = eng.sample(cond, field_ids=ids)                 # captures the graph
    y_eng2 = eng.sample(cond, field_ids=ids)                # replays it
    torch.cuda.synchronize()
    assert torch.equal(torch.cuda.get_rng_state(), state)
    assert eng.graph is not None and (eng.t == -1).all()
    err = rel_err(y_eng, y_eager)
    print(f"seeded DDIM graph vs eager: rel err {err:.3g}")
    assert err < 1e-3, err
    assert rel_err(y_eng2, y_eng) < 1e-3
    y_dpm = d.dpm_sample(cond, shape, cuda, steps=10, seed=SEED, field_ids=ids)
    y_dpm_eng = SampleEngine(d, shape, dpm_steps=10, seed=SEED).sample(cond, field_ids=ids)
    assert rel_err(y_dpm_eng, y_dpm) < 1e-3, rel_err(y_dpm_eng, y_dpm)


def test_eager_ddpm_sample_matches_engine(cuda):
    from cesm_emulator_b200.engine import SampleEngine
    d = _make(cuda, dict(BASELINE_KW, ch_mults=(1, 2)))
    shape = (2, 1, 16, 16)
    cond = torch.randn(shape, generator=torch.Generator().manual_seed(5)).to(cuda)
    y_eager = d.sample(cond, shape, cuda, seed=3, field_ids=[6, 2])
    y_eng = SampleEngine(d, shape, seed=3).sample(cond, field_ids=[6, 2])
    assert rel_err(y_eng, y_eager) < 1e-3, rel_err(y_eng, y_eager)


def test_weights_stay_fresh_in_seeded_graph(cuda):
    from cesm_emulator_b200 import kernels as K
    from cesm_emulator_b200.engine import SampleEngine
    tiny = dict(BASELINE_KW, ch_mults=(1, 2))
    d, other = _make(cuda, tiny, seed=0), _make(cuda, tiny, seed=1)
    g = torch.Generator().manual_seed(1)
    x = torch.randn(2, 1, 32, 32, generator=g).to(cuda)
    c = torch.randn(2, 1, 32, 32, generator=g).to(cuda)
    t = _ids([999, 499], cuda)
    samp = SampleEngine(d, (2, 1, 32, 32), ddim_steps=10, eta=1.0, seed=SEED)
    samp.sample(c, field_ids=[3, 4])                        # captures the graph with the first weights
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
            y_ref = K.ddim_step_seeded(x, eps, SEED, _ids([3, 4], cuda), t, samp.ddim_coef, T)
        assert rel_err(samp.x, y_ref) < 1e-2, (rnd, rel_err(samp.x, y_ref))


# ---- 7: inference.py ------------------------------------------------------------------------------
def test_inference_seed_is_batch_size_invariant(cuda):
    import inference
    d = _make(cuda, dict(BASELINE_KW, ch_mults=(1, 2)))
    cond = np.random.default_rng(0).standard_normal((2, 1, 1, 32, 32)).astype(np.float32)
    cond = np.repeat(cond, 3, axis=1)                       # one condition per year, shared by its members
    kw = dict(ddim_steps=10, eta=1.0, device=cuda, seed=SEED)
    p3 = inference.predict_temperature_from_emissions(d, cond, batch_size=3, **kw)
    p16 = inference.predict_temperature_from_emissions(d, cond, batch_size=16, **kw)
    worst = max(rel_err(torch.from_numpy(p3[t, m]), torch.from_numpy(p16[t, m])) for t in range(2) for m in range(3))
    print(f"inference --seed, batch_size 3 vs 16: worst per-field rel err {worst:.3g}")
    assert worst < 1e-2, worst
    for t in range(2):
        for m in range(3):
            for m2 in range(m):
                assert rel_err(torch.from_numpy(p3[t, m]), torch.from_numpy(p3[t, m2])) > 0.1, (t, m, m2)
