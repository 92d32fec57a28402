"""GPU tests of the SPAN upscaler: the library's forward against the fp32 oracle (tests/_span_oracle.py SPAN) at 1x, 2x
and 4x, nf 48 and 16, with and without the input normalisation; the reversal hooks; HDR-range input; the tcgen05 convs
against the CUDA-core validation kernel; stale eval_conv tensors; everything after the model given the model; the node;
and the rejections of SPAN layouts the library does not run.

Tolerances as for Compact (tests/test_gpu_upscaler_compact.py): fp16 tensor-core operands, fp32 accumulation and an fp32
block stream, so the model output is compared at rel-L2 <= 1e-2; everything after the model is fp32 in the reference's
operation order.  Each comparison prints the error it measured."""
import pytest
import torch

from _metrics import GpuModel, rel_l2, rel_trimmed
from _span_oracle import build_span, stale_eval_conv
from oracle import upscaler_oracle as uo
from oracle.make_golden_upscale import make_image

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def span():
    """(nf, s, norm) -> (oracle net, engine), built on first use and closed at the end of the module."""
    from vae_decode_hdr_b200.upscaler import HdrUpscalerEngine
    cache = {}

    def get(nf, s, norm=True):
        if (nf, s, norm) not in cache:
            net = build_span(nf + s + (0 if norm else 100), nf=nf, s=s, norm=norm)
            cache[(nf, s, norm)] = (net, HdrUpscalerEngine(net.state_dict(), DEV))
        return cache[(nf, s, norm)]
    yield get
    for _, eng in cache.values():
        eng.close()


def _oracle(net, x_bhwc, reversal):
    with torch.no_grad():
        y = net(x_bhwc.movedim(-1, 1))
    if reversal != "none":
        y = uo.reversal(y, reversal)
    return y.movedim(1, -1)


@pytest.mark.parametrize("n,h,w", [(1, 8, 12), (2, 40, 56), (1, 9, 133), (3, 31, 17)])    # 8 x 12: under 128 px, no slab
@pytest.mark.parametrize("norm", [True, False])
@pytest.mark.parametrize("nf", [48, 16])
@pytest.mark.parametrize("s", [1, 2, 4])
def test_span_forward_vs_oracle(span, s, nf, norm, n, h, w):
    net, eng = span(nf, s, norm)
    assert (eng.scale, eng.blocks) == (s, 6)
    x = make_image(n, h, w, 5 + n, 1.0).clamp(0, 1)
    got = eng.forward(x.to(DEV), "none").cpu()
    assert got.shape == (n, s * h, s * w, 3)
    err = rel_l2(got, _oracle(net, x, "none"))
    print(f"span nf {nf} {s}x norm {norm} {n}x{h}x{w}: rel-L2 {err:.2e}")
    assert err < 1e-2, err


@pytest.mark.parametrize("reversal", ["atanh", "logit"])
@pytest.mark.parametrize("s", [1, 2, 4])
def test_span_forward_with_reversal_vs_oracle(span, s, reversal):
    """The reversal hook is ill-conditioned next to its clamps: the 0.5 % worst pixels are set aside."""
    net, eng = span(48, s)
    x = make_image(2, 40, 56, 8, 1.0).clamp(0, 1)
    got = eng.forward(x.to(DEV), reversal).cpu()
    err = rel_trimmed(got, _oracle(net, x, reversal), 0.005)
    print(f"span {s}x {reversal}: trimmed rel-L2 {err:.2e}")
    assert err < 1e-2, err


@pytest.mark.parametrize("norm", [True, False])
def test_span_hdr_range_input(span, norm):
    """Amplitude-16 HDR input, unclamped as in the first pass: the x - mean fp16 operand and the fp32 block stream hold it."""
    net, eng = span(48, 4, norm)
    x = make_image(1, 48, 40, 17, 16.0)
    assert float(x.abs().max()) > 8.0
    got = eng.forward(x.to(DEV), "none").cpu()
    assert bool(torch.isfinite(got).all())
    err = rel_l2(got, _oracle(net, x, "none"))
    print(f"span HDR amplitude 16 norm {norm}: rel-L2 {err:.2e}")
    assert err < 1e-2, err


@pytest.mark.parametrize("nf,s", [(48, 4), (16, 2)])
def test_span_tcgen05_vs_cuda_core_kernel(span, nf, s):
    """Same packed operands through the tcgen05 kernel (64-column SiLU and gate builds, generic builds) and the CUDA-core
    validation kernel: only the fp32 summation order differs (plus the fp16 roundings it flips)."""
    from vae_decode_hdr_b200 import _native as N
    _, eng = span(nf, s)
    x = make_image(2, 24, 40, 3, 1.0).clamp(0, 1).to(DEV)
    a = eng.forward(x, "none")
    eng.set_conv_impl(N.CONV_DIRECT)
    try:
        b = eng.forward(x, "none")
    finally:
        eng.set_conv_impl(N.CONV_TCGEN05)
    err = rel_l2(a, b)
    print(f"span nf {nf} {s}x tcgen05 vs CUDA core: rel-L2 {err:.2e}")
    assert err < 3e-3, err


def test_span_ignores_a_stale_eval_conv():
    from vae_decode_hdr_b200.upscaler import HdrUpscalerEngine
    net = build_span(11, nf=48, s=2)
    a_eng = HdrUpscalerEngine(net.state_dict(), DEV)
    b_eng = HdrUpscalerEngine(stale_eval_conv(net), DEV)
    try:
        x = make_image(1, 24, 40, 4, 1.0).clamp(0, 1).to(DEV)
        assert torch.equal(a_eng.forward(x, "none"), b_eng.forward(x, "none"))
    finally:
        a_eng.close()
        b_eng.close()


_AFTER_MODEL_CASES = [(1, 530, 24, False, False, "bilinear", "atanh"), (1, 40, 600, True, True, "nearest-exact", "logit"),
                      (1, 36, 44, False, True, "bislerp", "logit"), (2, 30, 26, False, True, "bicubic", "logit")]


@pytest.mark.parametrize("B,H,W,blur,fix,method,reversal", _AFTER_MODEL_CASES)
@pytest.mark.parametrize("s", [1, 2, 4])
def test_tiling_blend_and_recombination_are_exact_given_the_model(span, s, B, H, W, blur, fix, method, reversal):
    _, eng = span(16, s)
    img = make_image(B, H, W, 31, 1.0).clamp(0, 1)
    arch = "ESRGAN" if reversal == "atanh" else "SPAN"                # the oracle picks the reversal by name
    want = uo.upscale(img, uo.FakeDescriptor(GpuModel(eng), s, arch), blur, fix, method)
    got = eng.upscale(img.to(DEV), reversal, blur, fix, method).cpu()
    assert got.shape == want.shape == (B, s * H, s * W, 3)
    err = (got - want).abs()
    # atanhf / logf vs torch differ by an ulp or two; the 3x3 medians can pick an equal-within-ulp other sample
    assert float(err.max()) <= 2e-5 * max(1.0, float(want.abs().max())), float(err.max())


def _node_with(monkeypatch, descriptor, model_path=None):
    from vae_decode_hdr_b200.hdr_upscale_with_model import HDRUpscaleWithModel
    node = HDRUpscaleWithModel()
    calls = []

    def load(name):
        calls.append(name)
        return descriptor
    monkeypatch.setattr(node, "_load_model_internal", load)
    if model_path is not None:
        monkeypatch.setattr(HDRUpscaleWithModel, "_model_path", staticmethod(lambda name: model_path))
    return node, calls


def test_node_runs_a_span_model_with_logit_and_its_cache(monkeypatch, tmp_path):
    from vae_decode_hdr_b200 import upscaler as U
    from vae_decode_hdr_b200.hdr_upscale_with_model import HDRUpscaleWithModel
    net = build_span(12, nf=16, s=2)
    desc = uo.FakeDescriptor(net, 2, "SPAN")
    node, calls = _node_with(monkeypatch, desc, str(tmp_path / "span_2x.pth"))
    seen = []
    real = U.HdrUpscalerEngine.upscale

    def spy(self, image, reversal, *a, **k):
        seen.append(reversal)
        return real(self, image, reversal, *a, **k)
    monkeypatch.setattr(U.HdrUpscalerEngine, "upscale", spy)
    img = make_image(1, 20, 28, 12, 1.0).clamp(0, 1)
    try:
        (a,) = node.upscale(img, "span_2x.pth", True, True, "bislerp")
        (b,) = node.upscale(img, "span_2x.pth", True, True, "bislerp")
        assert len(calls) == 1 and seen == ["logit", "logit"]           # the second call hit the engine cache
        assert a.shape == (1, 40, 56, 3) and torch.equal(a, b)
        ref = uo.upscale(img, desc, True, True, "bislerp")
        assert rel_l2(a, ref) < 1e-2, rel_l2(a, ref)
    finally:
        HDRUpscaleWithModel.release_memory()


def test_node_rejects_a_descriptor_scale_the_span_weights_contradict(monkeypatch):
    net = build_span(13, nf=8, s=2)
    node, _ = _node_with(monkeypatch, uo.FakeDescriptor(net, 4, "SPAN"))
    with pytest.raises(RuntimeError, match=r"scale 4.*2x"):
        node.upscale(make_image(1, 16, 16, 1, 1.0), "wrong.pth")


def _span_sd(nf=48, s=2):
    from vae_decode_hdr_b200.synthetic import random_span_state_dict
    return random_span_state_dict(0, nf, s)


def test_span_rejections_name_the_tensor():
    from vae_decode_hdr_b200.upscaler import HdrUpscalerEngine
    sd = _span_sd()
    sd["upsampler.0.weight"], sd["upsampler.0.bias"] = torch.zeros(27, 48, 3, 3), torch.zeros(27)     # a 3x model
    with pytest.raises(RuntimeError, match=r"upsampler\.0\.weight has shape \[27,48,3,3\].*scale 1, 2 or 4"):
        HdrUpscalerEngine(sd, DEV)
    for nf in (52, 96):
        with pytest.raises(RuntimeError, match=rf"conv_1\.sk\.weight has shape \[{nf},3,1,1\].*multiple of 8 in 8\.\.64"):
            HdrUpscalerEngine(_span_sd(nf=nf), DEV)
    sd = _span_sd()
    sd["conv_1.sk.weight"] = torch.zeros(48, 1, 1, 1)                                                # 1 input channel
    with pytest.raises(RuntimeError, match=r"conv_1\.sk\.weight has shape \[48,1,1,1\]"):
        HdrUpscalerEngine(sd, DEV)
    sd = _span_sd()
    del sd["block_4.c2_r.conv.1.bias"]
    with pytest.raises(RuntimeError, match=r"lacks block_4\.c2_r\.conv\.1\.bias \(want shape \[96\]\)"):
        HdrUpscalerEngine(sd, DEV)
    sd = _span_sd()
    for k in [k for k in sd if k.startswith("block_6.")]:
        sd["block_7." + k[len("block_6."):]] = sd[k].clone()
    with pytest.raises(RuntimeError, match=r"block_7\.\S+ has shape \[\d+(,\d+)*\]; SPAN has exactly the blocks"):
        HdrUpscalerEngine(sd, DEV)
    sd = _span_sd()
    sd["block_2.c3_r.conv.2.weight"] = torch.zeros(48, 80, 1, 1)                                      # mismatched Conv3XC
    with pytest.raises(RuntimeError, match=r"block_2\.c3_r\.conv\.2\.weight has shape \[48,80,1,1\]; want \[48,96,1,1\]"):
        HdrUpscalerEngine(sd, DEV)
