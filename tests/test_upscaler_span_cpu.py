"""CPU tests of the SPAN pieces: the oracle's key layout for nf 48 at 1x / 2x / 4x with and without the input
normalisation, the synthetic state dict, the Conv3XC fusion against the unfused training form and against an
independent composition of the three convs, the activated b5_2 that block_6 returns, that the random init leaves the
output input-dependent, the tiling at 1x / 2x with a SPAN descriptor, and the reversal the node picks for "SPAN"."""
import pytest
import torch
import torch.nn.functional as F

from _span_oracle import Conv3XC, build_span, stale_eval_conv
from oracle import upscaler_oracle as uo


@pytest.mark.parametrize("norm", [True, False])
@pytest.mark.parametrize("s", [1, 2, 4])
def test_span_oracle_key_layout(s, norm):
    from vae_decode_hdr_b200.synthetic import random_span_state_dict
    sd = build_span(0, nf=48, s=s, norm=norm).state_dict()
    assert ("no_norm" in sd) == (not norm)
    assert sd["conv_1.sk.weight"].shape == (48, 3, 1, 1)
    assert sd["conv_1.conv.0.weight"].shape == (6, 3, 1, 1) and sd["conv_1.conv.1.weight"].shape == (96, 6, 3, 3)
    assert sd["conv_1.conv.2.weight"].shape == (48, 96, 1, 1) and sd["conv_1.eval_conv.weight"].shape == (48, 3, 3, 3)
    blocks = sorted({k.split(".")[0] for k in sd if k.startswith("block_")})
    assert blocks == [f"block_{b}" for b in range(1, 7)]
    for b in range(1, 7):
        for c in (1, 2, 3):
            p = f"block_{b}.c{c}_r"
            assert sd[f"{p}.sk.weight"].shape == (48, 48, 1, 1) and sd[f"{p}.conv.1.weight"].shape == (96, 96, 3, 3)
            assert sd[f"{p}.conv.0.bias"].shape == (96,) and sd[f"{p}.conv.2.bias"].shape == (48,)
    assert sd["conv_cat.weight"].shape == (48, 192, 1, 1) and sd["conv_cat.bias"].shape == (48,)
    assert sd["conv_2.sk.weight"].shape == (48, 48, 1, 1)
    assert sd["upsampler.0.weight"].shape == (3 * s * s, 48, 3, 3) and sd["upsampler.0.bias"].shape == (3 * s * s,)
    syn = random_span_state_dict(0, 48, s, norm)
    assert list(syn) == list(sd) and all(syn[k].shape == sd[k].shape for k in sd)


def _fuse(m: Conv3XC):
    """The fusion written out as matrix products in fp64: W = w3 w2 w1 (+ sk at the centre), b = w3 (w2 b1 + b2) + b3 + b_sk."""
    w1, b1 = m.conv[0].weight.double()[:, :, 0, 0], m.conv[0].bias.double()
    w2, b2 = m.conv[1].weight.double(), m.conv[1].bias.double()
    w3, b3 = m.conv[2].weight.double()[:, :, 0, 0], m.conv[2].bias.double()
    w = torch.einsum("om,mjyx,ji->oiyx", w3, w2, w1)
    w[:, :, 1, 1] += m.sk.weight.double()[:, :, 0, 0]
    b = w3 @ (w2.sum((2, 3)) @ b1 + b2) + b3 + m.sk.bias.double()
    return w, b


@pytest.mark.parametrize("cin,cout", [(3, 48), (48, 48), (16, 16)])
def test_conv3xc_fusion(cin, cout):
    torch.manual_seed(cin + cout)
    m = Conv3XC(cin, cout).eval().requires_grad_(False)
    w, b = _fuse(m)
    assert float((m.eval_conv.weight.double() - w).norm() / w.norm()) <= 1e-6
    assert float((m.eval_conv.bias.double() - b).norm() / b.norm()) <= 1e-6
    x = torch.randn(2, cin, 11, 13)
    with torch.no_grad():
        fused = m(x)
        m.train()
        unfused = m(x)
        m.eval()
    # zero padding of x is not zero padding of conv.0(x): the forms agree away from the border
    assert torch.allclose(fused[:, :, 1:-1, 1:-1], unfused[:, :, 1:-1, 1:-1], atol=1e-4, rtol=1e-4)


def test_eval_forward_rebuilds_a_stale_eval_conv():
    net = build_span(2, nf=16, s=2)
    x = torch.rand(1, 3, 12, 10)
    with torch.no_grad():
        want = net(x)
        net.load_state_dict(stale_eval_conv(net))
        assert float(net.conv_1.eval_conv.weight.abs().max()) > 10.0
        got = net(x)
    assert torch.equal(got, want)


def test_block_6_returns_the_activated_out1():
    net = build_span(3, nf=16, s=1)
    x = torch.randn(1, 16, 9, 7)
    with torch.no_grad():
        _, out1, att = net.block_6(x)
        pre = net.block_6.c1_r(x)
    assert torch.allclose(out1, F.silu(pre), atol=1e-6) and float((out1 - pre).abs().max()) > 1e-3
    assert float(att.abs().max()) <= 0.5


@pytest.mark.parametrize("norm", [True, False])
def test_random_init_output_depends_on_the_input(norm):
    """Six gated blocks of PyTorch-default-init Conv3XCs would return their biases; build_span's init does not."""
    net = build_span(4, nf=48, s=2, norm=norm)
    g = torch.Generator().manual_seed(5)
    a, b = torch.rand(2, 3, 16, 16, generator=g).chunk(2)
    with torch.no_grad():
        ya, yb = net(a), net(b)
        f = net.conv_1((a - net.mean) * 255.0 if norm else a)
        b6 = net.block_6(net.block_5(net.block_4(net.block_3(net.block_2(net.block_1(f)[0])[0])[0])[0])[0])[0]
    assert float((ya - yb).std()) > 0.2 * float(ya.std())
    assert float(b6.std()) > 1e-3 * float(f.std())          # the deep blocks still carry signal


@pytest.mark.parametrize("s", [1, 2])
def test_tiling_with_a_span_descriptor(s):
    """oracle.upscale() at 1x / 2x with a SPAN descriptor: the logit reversal, the output shape, finite values."""
    net = build_span(6, nf=8, s=s)
    desc = uo.FakeDescriptor(net, s, "SPAN")
    img = torch.rand(1, 40, 36, 3) * 0.8 + 0.1
    out = uo.upscale(img, desc, False, False, "bilinear")
    assert uo.reversal_kind("SPAN") == "logit"
    assert out.shape == (1, s * 40, s * 36, 3) and bool(torch.isfinite(out).all())


def test_node_picks_logit_for_span():
    from vae_decode_hdr_b200.upscaler import is_compact_state_dict, reversal_for_architecture, rrdbnet_scale
    assert reversal_for_architecture("SPAN") == "logit"
    sd = build_span(0, nf=8, s=2).state_dict()
    assert not is_compact_state_dict(sd) and rrdbnet_scale(sd) is None       # the library decides, by conv_1.sk.weight
