"""GPU tests of the RRDBNet forms besides the 4x one: the pixel-unshuffle form (RealESRGAN_x2plus: f = 2, and f = 4 at 1x)
and the plain form with 1 or 0 upsampling convs.  The library's forward against the fp32 oracle (tests/_rrdb_oracle.py),
the tcgen05 convs against the CUDA-core validation kernel, the two key layouts, everything after the model at 1x and 2x
given the model (including images whose sides pad edge tiles), the node, and the rejections.

Tolerances as for the 4x RRDBNet (tests/test_gpu_upscaler.py): fp16 tensor-core operands, fp32 accumulation, so the model
output is compared at rel-L2 <= 1e-2; everything after the model is fp32 in the reference's operation order."""
import pytest
import torch

import _rrdb_oracle as ro
from oracle import upscaler_oracle as uo
from oracle.make_golden_upscale import make_image

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# (n_up, shuffle, scale): the forms this file covers (the 4x one, (2, 1, 4), is tests/test_gpu_upscaler.py's)
NEW_FORMS = [(2, 2, 2), (2, 4, 1), (1, 1, 2), (0, 1, 1), (1, 2, 1)]


def _rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm())


def _rel_trimmed(a, b, frac):
    e = ((a - b).double() ** 2).sum(dim=-1).flatten()
    k = e.numel() - int(frac * e.numel())
    return float(e.sort().values[:k].sum().sqrt() / b.double().norm())


@pytest.fixture(scope="module")
def rrdb():
    """(n_up, shuffle, nb) -> (oracle net, engine), built on first use and closed at the end of the module."""
    from vae_decode_hdr_b200.upscaler import HdrUpscalerEngine
    cache = {}

    def get(n_up, f, nb):
        if (n_up, f, nb) not in cache:
            net = ro.build_upscaler(10 * n_up + f + 100 * nb, nb=nb, n_up=n_up, shuffle=f)
            cache[(n_up, f, nb)] = (net, HdrUpscalerEngine(net.state_dict(), DEV))
        return cache[(n_up, f, nb)]
    yield get
    for _, eng in cache.values():
        eng.close()


def _oracle(net, x_bhwc, reversal):
    with torch.no_grad():
        y = net(x_bhwc.movedim(-1, 1))
    if reversal != "none":
        y = uo.reversal(y, reversal)
    return y.movedim(1, -1)


@pytest.mark.parametrize("reversal", ["none", "atanh"])
@pytest.mark.parametrize("n,h,w", [(1, 16, 16), (2, 40, 56), (1, 9, 133), (3, 64, 32)])
@pytest.mark.parametrize("nb", [1, 2])
@pytest.mark.parametrize("n_up,f,s", NEW_FORMS)
def test_rrdbnet_forms_forward_vs_oracle(rrdb, n_up, f, s, nb, n, h, w, reversal):
    """atanh: the plain 1x form's output reaches past +-1, where the hook saturates and is ill-conditioned, so the 0.5 %
    worst pixels are set aside there (as in the Compact tests)."""
    net, eng = rrdb(n_up, f, nb)
    assert (eng.scale, eng.blocks) == (s, nb)
    x = make_image(n, h, w, 5 + n, 3.0)
    got = eng.forward(x.to(DEV), reversal).cpu()
    assert got.shape == (n, s * h, s * w, 3)
    ref = _oracle(net, x, reversal)
    err = _rel(got, ref) if reversal == "none" else _rel_trimmed(got, ref, 0.005)
    assert err < 1e-2, err


@pytest.mark.parametrize("n_up,f,s", NEW_FORMS)
def test_rrdbnet_forms_tcgen05_vs_cuda_core_kernel(rrdb, n_up, f, s):
    """Same packed operands through the tcgen05 kernel and the CUDA-core validation kernel (25 x 42: padded for f = 2, 4)."""
    from vae_decode_hdr_b200 import _native as N
    _, eng = rrdb(n_up, f, 1)
    x = make_image(2, 25, 42, 3, 3.0).to(DEV)
    a = eng.forward(x, "none")
    eng.set_conv_impl(N.CONV_DIRECT)
    try:
        b = eng.forward(x, "none")
    finally:
        eng.set_conv_impl(N.CONV_TCGEN05)
    assert a.shape == (2, 25 * s, 42 * s, 3)
    assert _rel(a, b) < 3e-3, _rel(a, b)


@pytest.mark.parametrize("n_up,f,s", NEW_FORMS)
def test_old_arch_state_dict_gives_identical_model(rrdb, n_up, f, s):
    from vae_decode_hdr_b200.upscaler import HdrUpscalerEngine
    net, eng = rrdb(n_up, f, 1)
    eng_old = HdrUpscalerEngine(ro.state_dict_old_arch(net), DEV)
    try:
        assert (eng_old.scale, eng_old.blocks) == (s, 1)
        x = make_image(1, 21, 26, 9, 3.0).to(DEV)
        assert torch.equal(eng.forward(x, "atanh"), eng_old.forward(x, "atanh"))
    finally:
        eng_old.close()


class _GpuModel(torch.nn.Module):
    """The oracle's tiling / recombination driven by the GPU network: isolates everything after the model."""

    def __init__(self, eng):
        super().__init__()
        self.eng = eng

    def forward(self, a):
        return self.eng.forward(a.movedim(1, -1).contiguous().to(DEV), "none").cpu().movedim(-1, 1)


# 531 x 37: the edge tiles (83 rows) and the 37 columns are not multiples of 2 or 4, so they pad
_AFTER_MODEL_CASES = [(1, 530, 24, False, False, "bilinear", "atanh"), (1, 40, 600, True, True, "nearest-exact", "logit"),
                      (1, 520, 520, False, True, "bilinear", "logit"), (1, 531, 37, False, True, "bislerp", "atanh"),
                      (2, 30, 26, True, True, "bicubic", "atanh")]


@pytest.mark.parametrize("B,H,W,blur,fix,method,reversal", _AFTER_MODEL_CASES)
@pytest.mark.parametrize("n_up,f,s", [(2, 2, 2), (1, 1, 2), (2, 4, 1), (0, 1, 1)])
def test_tiling_blend_and_recombination_are_exact_given_the_model(rrdb, n_up, f, s, B, H, W, blur, fix, method, reversal):
    _, eng = rrdb(n_up, f, 1)
    img = make_image(B, H, W, 31, 3.0)
    arch = "ESRGAN" if reversal == "atanh" else "Other"                 # the oracle picks the reversal by name
    want = uo.upscale(img, uo.FakeDescriptor(_GpuModel(eng), s, arch), blur, fix, method)
    got = eng.upscale(img.to(DEV), reversal, blur, fix, method).cpu()
    assert got.shape == want.shape == (B, s * H, s * W, 3)
    err = (got - want).abs()
    # atanhf / logf vs torch differ by an ulp or two; the 3x3 medians can pick an equal-within-ulp other sample
    assert float(err.max()) <= 2e-5 * max(1.0, float(want.abs().max())), float(err.max())


def _node_with(monkeypatch, descriptor, model_path):
    from vae_decode_hdr_b200.hdr_upscale_with_model import HDRUpscaleWithModel
    node = HDRUpscaleWithModel()
    calls = []

    def load(name):
        calls.append(name)
        return descriptor
    monkeypatch.setattr(node, "_load_model_internal", load)
    monkeypatch.setattr(HDRUpscaleWithModel, "_model_path", staticmethod(lambda name: model_path))
    return node, calls


@pytest.mark.parametrize("n_up,f,s,H,W", [(2, 2, 2, 37, 30), (0, 1, 1, 44, 52)])
def test_node_runs_the_form_and_caches_it(monkeypatch, tmp_path, n_up, f, s, H, W):
    from vae_decode_hdr_b200.hdr_upscale_with_model import HDRUpscaleWithModel
    net = ro.build_upscaler(8, nb=2, gain=0.5, n_up=n_up, shuffle=f)      # output within +-0.5: atanh well-conditioned
    desc = uo.FakeDescriptor(net, s, "ESRGAN")
    node, calls = _node_with(monkeypatch, desc, str(tmp_path / "rrdb.pth"))
    img = make_image(1, H, W, 12, 3.0)
    try:
        (a,) = node.upscale(img, "rrdb.pth", False, True, "bislerp")
        (b,) = node.upscale(img, "rrdb.pth", False, True, "bislerp")
        assert len(calls) == 1                                          # the second call hit the engine cache
        assert a.device.type == "cpu" and a.shape == (1, s * H, s * W, 3) and torch.equal(a, b)
        ref = uo.upscale(img, desc, False, True, "bislerp")
        assert _rel(a, ref) < 1e-2, _rel(a, ref)
    finally:
        HDRUpscaleWithModel.release_memory()


def _sd(n_up=2, f=1):
    from vae_decode_hdr_b200.synthetic import random_upscaler_state_dict
    return random_upscaler_state_dict(0, 1, n_up, f)


def test_rejections_name_the_tensor_and_its_shape():
    from vae_decode_hdr_b200.upscaler import HdrUpscalerEngine
    with pytest.raises(RuntimeError, match=r"conv_up3\.weight has shape \[64,64,3,3\].*8x"):
        HdrUpscalerEngine(_sd(3, 1), DEV)
    old8 = ro.state_dict_old_arch(ro.build_upscaler(0, nb=1, n_up=3))
    with pytest.raises(RuntimeError, match=r"model\.9\.weight has shape \[64,64,3,3\].*8x"):
        HdrUpscalerEngine(old8, DEV)
    with pytest.raises(RuntimeError, match=r"conv_first\.weight has shape \[64,12,3,3\].*below 1"):
        HdrUpscalerEngine(_sd(0, 2), DEV)                                            # f = 2 with u = 0: scale 1/2
    sd = _sd()
    sd["conv_first.weight"] = torch.zeros(64, 6, 3, 3)
    with pytest.raises(RuntimeError, match=r"conv_first\.weight has shape \[64,6,3,3\].*3, 12 or 48"):
        HdrUpscalerEngine(sd, DEV)
    sd = _sd()
    sd["conv_up1.weight"], sd["conv_up1.bias"] = torch.zeros(256, 64, 3, 3), torch.zeros(256)   # pixel-shuffle upsampler
    with pytest.raises(RuntimeError, match=r"conv_up1\.weight has the wrong shape \[256,64,3,3\]"):
        HdrUpscalerEngine(sd, DEV)
    old = ro.state_dict_old_arch(ro.build_upscaler(0, nb=1, n_up=1))
    old["model.9.weight"], old["model.9.bias"] = torch.zeros(3, 64, 3, 3), torch.zeros(3)      # conv_last at 9: no u fits
    with pytest.raises(RuntimeError, match=r"model\.9\.weight has shape \[3,64,3,3\]"):
        HdrUpscalerEngine(old, DEV)


def test_tile_side_too_short_for_the_reflect_pad(rrdb):
    _, eng4 = rrdb(2, 4, 1)
    with pytest.raises(RuntimeError, match="tile side of 2 pixels"):
        eng4.forward(make_image(1, 2, 16, 1, 1.0).to(DEV), "none")
    _, eng2 = rrdb(2, 2, 1)
    with pytest.raises(RuntimeError, match="tile side of 1 pixels"):
        eng2.upscale(make_image(1, 1, 40, 1, 1.0).to(DEV), "atanh")
    got = eng2.upscale(make_image(1, 3, 40, 1, 1.0).to(DEV), "atanh")                # 3 rows: a pad of 1 is fine
    assert got.shape == (1, 6, 80, 3) and bool(torch.isfinite(got).all())
