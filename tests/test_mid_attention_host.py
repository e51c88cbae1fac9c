"""CPU checks of use_mid_attn=True (video_net.py:713-719): the oracle's restatement of the block against an
independent formulation of the same spec, and the module tree / state-dict layout the B200 kernels serve."""
import torch
import torch.nn.functional as F

from _parity import BASELINE_KW


def _spec_block(x, gamma, wqkv, wout, heads):
    """The spec written independently of the oracle: channel LayerNorm (gain only, eps 1e-5), bias-free q|k|v
    projection, per frame and head softmax((q 32^-0.5) k^T) v over all h*w pixels (SDPA), bias-free to_out, residual."""
    b, c, f, h, w = x.shape
    xs = x.permute(0, 2, 3, 4, 1).reshape(b * f, h * w, c)
    mean = xs.mean(-1, keepdim=True)
    var = xs.var(-1, unbiased=False, keepdim=True)
    xn = (xs - mean) / torch.sqrt(var + 1e-5) * gamma.reshape(c)
    q, k, v = (t.reshape(b * f, h * w, heads, 32).transpose(1, 2) for t in (xn @ wqkv.t()).chunk(3, dim=-1))
    o = F.scaled_dot_product_attention(q, k, v, scale=32 ** -0.5)
    y = o.transpose(1, 2).reshape(b * f, h * w, heads * 32) @ wout.t()
    return x + y.reshape(b, f, h, w, c).permute(0, 4, 1, 2, 3)


def test_oracle_mid_block_equals_independent_spec():
    from oracle import cesm_oracle as O
    g = torch.Generator().manual_seed(0)
    for (b, c, f, h, w, heads) in [(2, 64, 3, 6, 9, 8), (1, 32, 1, 4, 4, 4), (1, 64, 2, 5, 7, 2)]:
        x = torch.randn(b, c, f, h, w, generator=g)
        gamma = 1 + 0.1 * torch.randn(1, c, 1, 1, 1, generator=g)
        wqkv = torch.randn(3 * heads * 32, c, generator=g) * c ** -0.5
        wout = torch.randn(c, heads * 32, generator=g) * (heads * 32) ** -0.5
        pre = "mid_spatial_attn."
        sd = {pre + "fn.norm.gamma": gamma, pre + "fn.fn.fn.to_qkv.weight": wqkv, pre + "fn.fn.fn.to_out.weight": wout}
        got = O.mid_spatial_attention_block(sd, pre, x, heads)
        ref = _spec_block(x, gamma, wqkv, wout, heads)
        assert got.shape == x.shape
        assert torch.allclose(got, ref, rtol=1e-5, atol=1e-5), (got - ref).abs().max()


def test_mid_attn_state_dict_and_module_tree():
    from oracle import cesm_oracle as O
    from cesm_emulator_b200 import video_net as V
    from cesm_emulator_b200.model import UNet
    kw = dict(BASELINE_KW, use_mid_attn=True)
    torch.manual_seed(0)
    unet = UNet(**kw)
    sd = unet.state_dict()
    pre = "net.mid_spatial_attn."
    assert tuple(sd[pre + "fn.norm.gamma"].shape) == (1, 256, 1, 1, 1)
    assert tuple(sd[pre + "fn.fn.fn.to_qkv.weight"].shape) == (768, 256)
    assert tuple(sd[pre + "fn.fn.fn.to_out.weight"].shape) == (256, 256)
    assert not any(k.startswith(pre) for k in UNet(**BASELINE_KW).state_dict())
    # the wrapper tells the Attention its sequence axis; the temporal attentions keep theirs
    net = unet.net
    assert isinstance(net.mid_spatial_attn.fn.fn, V.EinopsToAndFrom)
    assert net.mid_spatial_attn.fn.fn.fn.seq == "pixels"
    assert net.mid_temporal_attn.fn.fn.fn.seq == "frames"
    assert all(m.seq == "frames" for m in net.modules() if isinstance(m, V.Attention) and m is not net.mid_spatial_attn.fn.fn.fn)
    # the default model is untouched: no mid block
    assert isinstance(UNet(**BASELINE_KW).net.mid_spatial_attn, torch.nn.Identity)

    # the checkpoint loads into the oracle, whose forward then runs the mid block (zeroing its to_out changes the output)
    cfg = O.OracleConfig.from_unet_kwargs(**kw)
    assert cfg.use_mid_attn
    osd = {k: v.detach().float() for k, v in sd.items()}
    g = torch.Generator().manual_seed(1)
    x, cond = torch.randn(1, 1, 16, 16, generator=g), torch.randn(1, 1, 3, 16, 16, generator=g)
    t = torch.tensor([10])
    with torch.no_grad():
        with_mid = O.unet_forward(osd, cfg, x, cond, t)
        osd[pre + "fn.fn.fn.to_out.weight"] = torch.zeros(256, 256)
        without = O.unet_forward(osd, cfg, x, cond, t)
    assert with_mid.shape == (1, 1, 16, 16) and torch.isfinite(with_mid).all()
    assert (with_mid - without).abs().max() > 1e-4

    # the round trip through a second module works in both directions (strict)
    torch.manual_seed(1)
    other = UNet(**kw)
    other.load_state_dict(sd, strict=True)
    assert torch.equal(other.state_dict()[pre + "fn.fn.fn.to_qkv.weight"], sd[pre + "fn.fn.fn.to_qkv.weight"])
