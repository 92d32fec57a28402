"""GPU tests of the Real-ESRGAN Compact (SRVGGNetCompact) upscaler: the library's forward against the fp32 oracle
(tests/_compact_oracle.py SRVGGNetCompact) at 1x, 2x and 4x, the tcgen05 convs against the CUDA-core validation kernel,
everything after the model (tiling, feather blend, YCbCr, medians, local fix) at the Compact's scales given the model,
the node with Compact descriptors, and the rejections of what the library does not run.

Tolerances as for RRDBNet (tests/test_gpu_upscaler.py): fp16 tensor-core operands, fp32 accumulation, so the model
output is compared at rel-L2 <= 1e-2; everything after the model is fp32 in the reference's operation order."""
import pytest
import torch

from _compact_oracle import build_compact
from _metrics import GpuModel, rel_l2, rel_trimmed
from oracle import upscaler_oracle as uo
from oracle.make_golden_upscale import make_image

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def compact():
    """(nf, nc, s) -> (oracle net, engine), built on first use and closed at the end of the module."""
    from vae_decode_hdr_b200.upscaler import HdrUpscalerEngine
    cache = {}

    def get(nf, nc, s):
        if (nf, nc, s) not in cache:
            net = build_compact(nf + 10 * nc + s, nf=nf, nc=nc, s=s)
            cache[(nf, nc, s)] = (net, HdrUpscalerEngine(net.state_dict(), DEV))
        return cache[(nf, nc, s)]
    yield get
    for _, eng in cache.values():
        eng.close()


def _oracle(net, x_bhwc, reversal):
    with torch.no_grad():
        y = net(x_bhwc.movedim(-1, 1))
    if reversal != "none":
        y = uo.reversal(y, reversal)
    return y.movedim(1, -1)


@pytest.mark.parametrize("n,h,w", [(1, 8, 12), (2, 40, 56), (1, 9, 133), (3, 64, 32)])    # 8 x 12: under 128 px, no slab
@pytest.mark.parametrize("nc", [0, 4])
@pytest.mark.parametrize("nf", [64, 24])
@pytest.mark.parametrize("s", [1, 2, 4])
def test_compact_forward_vs_oracle(compact, s, nf, nc, n, h, w):
    net, eng = compact(nf, nc, s)
    assert (eng.scale, eng.blocks) == (s, nc)
    x = make_image(n, h, w, 5 + n, 3.0)
    got = eng.forward(x.to(DEV), "none").cpu()
    assert got.shape == (n, s * h, s * w, 3)
    assert rel_l2(got, _oracle(net, x, "none")) < 1e-2


@pytest.mark.parametrize("reversal", ["atanh", "logit"])
@pytest.mark.parametrize("s", [1, 2, 4])
def test_compact_forward_with_reversal_vs_oracle(compact, s, reversal):
    """The reversal hook is ill-conditioned next to its clamps: the 0.5 % worst pixels are set aside."""
    net, eng = compact(64, 4, s)
    x = make_image(2, 40, 56, 8, 3.0)
    got = eng.forward(x.to(DEV), reversal).cpu()
    ref = _oracle(net, x, reversal)
    assert rel_trimmed(got, ref, 0.005) < 1e-2, rel_trimmed(got, ref, 0.005)


def test_compact_full_depth_vs_oracle():
    """realesr-general-x4v3's shape (nf 64, 32 body convs, 4x): error accumulation through the full depth."""
    from vae_decode_hdr_b200.upscaler import HdrUpscalerEngine
    net = build_compact(1, nf=64, nc=32, s=4)
    eng = HdrUpscalerEngine(net.state_dict(), DEV)
    try:
        assert (eng.scale, eng.blocks) == (4, 32)
        x = make_image(1, 48, 40, 17, 3.0)
        got = eng.forward(x.to(DEV), "none").cpu()
        assert rel_l2(got, _oracle(net, x, "none")) < 1e-2, rel_l2(got, _oracle(net, x, "none"))
    finally:
        eng.close()


@pytest.mark.parametrize("nf,nc,s", [(64, 4, 4), (24, 4, 2)])
def test_compact_tcgen05_vs_cuda_core_kernel(compact, nf, nc, s):
    """Same packed operands through the tcgen05 kernel (64-column PReLU build, generic 32-column build) and the CUDA-core
    validation kernel: only the fp32 summation order differs (plus the fp16 roundings it flips)."""
    from vae_decode_hdr_b200 import _native as N
    _, eng = compact(nf, nc, s)
    x = make_image(2, 24, 40, 3, 3.0).to(DEV)
    a = eng.forward(x, "none")
    eng.set_conv_impl(N.CONV_DIRECT)
    try:
        b = eng.forward(x, "none")
    finally:
        eng.set_conv_impl(N.CONV_TCGEN05)
    assert rel_l2(a, b) < 3e-3


_AFTER_MODEL_CASES = [(1, 530, 24, False, False, "bilinear", "atanh"), (1, 40, 600, True, True, "nearest-exact", "logit"),
                      (1, 520, 520, False, True, "bilinear", "logit"), (1, 36, 44, False, True, "area", "atanh"),
                      (2, 30, 26, False, True, "bicubic", "logit"), (1, 36, 44, False, True, "bislerp", "atanh"),
                      (2, 20, 28, True, True, "bislerp", "logit")]


@pytest.mark.parametrize("B,H,W,blur,fix,method,reversal", _AFTER_MODEL_CASES)
@pytest.mark.parametrize("s", [1, 2, 4])
def test_tiling_blend_and_recombination_are_exact_given_the_model(compact, s, B, H, W, blur, fix, method, reversal):
    _, eng = compact(64, 2, s)
    img = make_image(B, H, W, 31, 3.0)
    arch = "ESRGAN" if reversal == "atanh" else "Compact"              # the oracle picks the reversal by name
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


def test_node_runs_a_2x_compact_model(monkeypatch):
    net = build_compact(5, nf=32, nc=3, s=2)
    desc = uo.FakeDescriptor(net, 2, "Compact")
    node, _ = _node_with(monkeypatch, desc)
    img = make_image(1, 24, 20, 11, 3.0)
    (out,) = node.upscale(img, "compact_2x.pth", False, True, "bislerp")
    assert out.device.type == "cpu" and out.dtype == torch.float32 and out.shape == (1, 48, 40, 3)
    ref = uo.upscale(img, desc, False, True, "bislerp")
    assert rel_l2(out, ref) < 1e-2, rel_l2(out, ref)


def test_node_cached_compact_engine(monkeypatch, tmp_path):
    from vae_decode_hdr_b200.hdr_upscale_with_model import HDRUpscaleWithModel
    net = build_compact(6, nf=16, nc=2, s=4)
    desc = uo.FakeDescriptor(net, 4, "Compact")
    node, calls = _node_with(monkeypatch, desc, str(tmp_path / "compact_4x.pth"))
    img = make_image(1, 20, 28, 12, 3.0)
    try:
        (a,) = node.upscale(img, "compact_4x.pth", True, False, "bilinear")
        (b,) = node.upscale(img, "compact_4x.pth", True, False, "bilinear")
        assert len(calls) == 1                                          # the second call hit the engine cache
        assert a.shape == (1, 80, 112, 3) and torch.equal(a, b)
        ref = uo.upscale(img, desc, True, False, "bilinear")
        assert rel_l2(a, ref) < 1e-2, rel_l2(a, ref)
    finally:
        HDRUpscaleWithModel.release_memory()


def test_node_rejects_a_descriptor_scale_the_weights_contradict(monkeypatch):
    net = build_compact(7, nf=16, nc=1, s=2)
    node, _ = _node_with(monkeypatch, uo.FakeDescriptor(net, 4, "Compact"))
    with pytest.raises(RuntimeError, match=r"scale 4.*2x"):
        node.upscale(make_image(1, 16, 16, 1, 1.0), "wrong.pth")


def test_node_rejects_esrgan_2x_naming_its_scale(monkeypatch):
    node, calls = _node_with(monkeypatch, uo.FakeDescriptor(uo.build_upscaler(0, nb=1), 2, "ESRGAN"))
    with pytest.raises(RuntimeError, match="scale 2"):
        node.upscale(make_image(1, 16, 16, 1, 1.0), "esrgan_2x.pth")
    assert calls == ["esrgan_2x.pth"]


def _compact_sd(nf=16, nc=1, s=2):
    from vae_decode_hdr_b200.synthetic import random_compact_state_dict
    return random_compact_state_dict(0, nf, nc, s)


def test_compact_rejections_name_the_tensor():
    from vae_decode_hdr_b200.upscaler import HdrUpscalerEngine
    sd = _compact_sd()
    sd["body.4.weight"], sd["body.4.bias"] = torch.zeros(27, 16, 3, 3), torch.zeros(27)     # 3 x 3^2: a 3x model
    with pytest.raises(RuntimeError, match=r"body\.4\.weight has shape \[27,16,3,3\].*scale 1, 2 or 4"):
        HdrUpscalerEngine(sd, DEV)
    sd = _compact_sd()
    sd["body.0.weight"] = torch.zeros(16, 1, 3, 3)                                        # 1 input channel
    with pytest.raises(RuntimeError, match=r"body\.0\.weight has shape \[16,1,3,3\]"):
        HdrUpscalerEngine(sd, DEV)
    sd = _compact_sd()
    del sd["body.3.weight"]                                                                 # a PReLU slope
    with pytest.raises(RuntimeError, match=r"lacks the PReLU slopes body\.3\.weight"):
        HdrUpscalerEngine(sd, DEV)
    with pytest.raises(RuntimeError, match=r"body\.0\.weight has shape \[96,3,3,3\].*8\.\.64"):
        HdrUpscalerEngine(_compact_sd(nf=96), DEV)
    with pytest.raises(RuntimeError, match="no RRDB blocks.*body.0.weight"):
        HdrUpscalerEngine({"foo.weight": torch.zeros(4, 4, 3, 3)}, DEV)


def test_rrdbnet_engine_reports_scale_4():
    from vae_decode_hdr_b200.upscaler import HdrUpscalerEngine
    eng = HdrUpscalerEngine(uo.build_upscaler(0, nb=1).state_dict(), DEV)
    try:
        assert (eng.scale, eng.blocks) == (4, 1)
    finally:
        eng.close()
