"""CPU tests of the RRDBNet forms besides the 4x one (0 / 1 / 2 upsampling convs, pixel-unshuffle factor 1 / 2 / 4): the
oracle's forward against an independent functional formulation, its key layouts, the synthetic state dict, the host's
scale rule `rrdbnet_scale`, and the node's scale checks that run before any library call."""
import pytest
import torch
import torch.nn.functional as F

import _rrdb_oracle as ro
from oracle import upscaler_oracle as uo

# (n_up, shuffle, scale): every accepted form
FORMS = [(2, 1, 4), (2, 2, 2), (2, 4, 1), (1, 1, 2), (0, 1, 1), (1, 2, 1)]


def _functional(sd, x, nb, n_up, f):
    def conv(name, a):
        return F.conv2d(a, sd[name + ".weight"], sd[name + ".bias"], padding=1)

    h, w = x.shape[-2:]
    if f > 1:
        x = F.pixel_unshuffle(F.pad(x, (0, (f - w % f) % f, 0, (f - h % f) % f), mode="reflect"), f)
    feat = conv("conv_first", x)
    t = feat
    for i in range(nb):
        r_in = t
        for r in (1, 2, 3):
            cat = [t]
            for j in range(1, 5):
                cat.append(F.leaky_relu(conv(f"body.{i}.rdb{r}.conv{j}", torch.cat(cat, 1)), 0.2))
            t = conv(f"body.{i}.rdb{r}.conv5", torch.cat(cat, 1)) * 0.2 + cat[0]
        t = t * 0.2 + r_in
    t = feat + conv("conv_body", t)
    for k in range(n_up):
        t = F.leaky_relu(conv(f"conv_up{k + 1}", F.interpolate(t, scale_factor=2, mode="nearest")), 0.2)
    out = conv("conv_last", F.leaky_relu(conv("conv_hr", t), 0.2))
    s = (1 << n_up) // f
    return out[..., :s * h, :s * w]


@pytest.mark.parametrize("h,w", [(8, 12), (9, 13), (7, 6)])
@pytest.mark.parametrize("n_up,f,s", FORMS)
def test_oracle_forward_vs_functional(n_up, f, s, h, w):
    net = ro.build_upscaler(3 + n_up + f, nb=2, n_up=n_up, shuffle=f)
    assert net.scale == s
    x = torch.randn(2, 3, h, w, generator=torch.Generator().manual_seed(11))
    with torch.no_grad():
        got = net(x)
    want = _functional(net.state_dict(), x, 2, n_up, f)
    assert got.shape == want.shape == (2, 3, s * h, s * w)
    assert torch.allclose(got, want, atol=1e-5, rtol=0), float((got - want).abs().max())


def test_oracle_defaults_are_the_4x_rrdbnet():
    """With the defaults the helper's network is oracle/upscaler_oracle.py's, parameter for parameter, in both layouts."""
    a, b = ro.build_upscaler(5, nb=2), uo.build_upscaler(5, nb=2)
    sa, sb = a.state_dict(), b.state_dict()
    assert list(sa) == list(sb) and all(torch.equal(sa[k], sb[k]) for k in sa)
    assert list(ro.state_dict_old_arch(a)) == list(uo.state_dict_old_arch(b))
    x = torch.randn(1, 3, 10, 14, generator=torch.Generator().manual_seed(2))
    with torch.no_grad():
        assert torch.equal(a(x), b(x))


@pytest.mark.parametrize("n_up,tops", [(2, [0, 3, 6, 8, 10]), (1, [0, 3, 5, 7]), (0, [0, 2, 4]), (3, [0, 3, 6, 9, 11, 13])])
def test_old_arch_top_level_indices(n_up, tops):
    net = ro.build_upscaler(0, nb=1, n_up=n_up)
    keys = list(ro.state_dict_old_arch(net))
    got = sorted({int(k.split(".")[1]) for k in keys if not k.startswith("model.1.")})
    assert got == tops
    assert all(k.startswith("model.1.sub.") for k in keys if k.startswith("model.1."))
    assert "model.1.sub.1.weight" in keys                                      # conv_body follows the nb blocks


@pytest.mark.parametrize("n_up,f", [(n, f) for n, f, _ in FORMS])
def test_synthetic_state_dict_matches_the_oracle(n_up, f):
    from vae_decode_hdr_b200.synthetic import random_upscaler_state_dict
    sd = ro.build_upscaler(0, nb=2, n_up=n_up, shuffle=f).state_dict()
    syn = random_upscaler_state_dict(0, 2, n_up, f)
    assert list(syn) == list(sd) and all(syn[k].shape == sd[k].shape for k in sd)
    assert sd["conv_first.weight"].shape == (64, 3 * f * f, 3, 3)


def test_rrdbnet_scale_accepted_layouts():
    from vae_decode_hdr_b200.synthetic import random_upscaler_state_dict
    from vae_decode_hdr_b200.upscaler import rrdbnet_scale
    for n_up, f, s in FORMS:
        net = ro.build_upscaler(0, nb=1, n_up=n_up, shuffle=f)
        assert rrdbnet_scale(net.state_dict()) == s, (n_up, f)
        assert rrdbnet_scale(ro.state_dict_old_arch(net)) == s, (n_up, f)
        assert rrdbnet_scale(random_upscaler_state_dict(0, 1, n_up, f)) == s
    assert rrdbnet_scale(uo.build_upscaler(0, nb=1).state_dict()) == 4


def test_rrdbnet_scale_rejected_layouts():
    from vae_decode_hdr_b200.synthetic import random_upscaler_state_dict
    from vae_decode_hdr_b200.upscaler import rrdbnet_scale
    eight = ro.build_upscaler(0, nb=1, n_up=3)
    assert rrdbnet_scale(eight.state_dict()) == 8
    assert rrdbnet_scale(ro.state_dict_old_arch(eight)) == 8
    sd = random_upscaler_state_dict(0, 1, 0, 1)
    sd["conv_first.weight"] = torch.zeros(64, 12, 3, 3)                     # f = 2 with u = 0: scale 1/2
    assert rrdbnet_scale(sd) is None
    sd["conv_first.weight"] = torch.zeros(64, 6, 3, 3)                      # 6 input channels
    assert rrdbnet_scale(sd) is None
    old = ro.state_dict_old_arch(ro.build_upscaler(0, nb=1, n_up=1))
    old["model.9.weight"], old["model.9.bias"] = torch.zeros(3, 64, 3, 3), torch.zeros(3)   # conv_last at 9: no u fits
    assert rrdbnet_scale(old) is None
    assert rrdbnet_scale({"foo.weight": torch.zeros(4, 4, 3, 3)}) is None


class _NoLibrary:
    def __init__(self, *a, **k):
        raise AssertionError("the node called the library")


@pytest.mark.parametrize("n_up,f,desc_scale,match", [
    (2, 2, 4, r"descriptor gives scale 4, its weights are a 2x network"),    # RealESRGAN_x2plus weights, descriptor 4
    (0, 1, 2, r"descriptor gives scale 2, its weights are a 1x network"),    # plain 1x weights, descriptor 2
    (3, 1, 8, r"scales 1, 2 and 4.*8x"),                                     # 8x weights
])
def test_node_refuses_before_any_library_call(monkeypatch, n_up, f, desc_scale, match):
    from vae_decode_hdr_b200 import hdr_upscale_with_model as m
    monkeypatch.setattr(m, "HdrUpscalerEngine", _NoLibrary)
    net = ro.build_upscaler(0, nb=1, n_up=n_up, shuffle=f)
    for model in (net, _OldArch(net)):
        with pytest.raises(RuntimeError, match=match):
            m.HDRUpscaleWithModel._new_engine(uo.FakeDescriptor(model, desc_scale, "ESRGAN"), torch.device("cuda", 0))


class _OldArch:
    """A model whose state_dict() is in the old-arch (spandrel / BasicSR) layout."""

    def __init__(self, net):
        self.net = net

    def state_dict(self):
        return ro.state_dict_old_arch(self.net)
