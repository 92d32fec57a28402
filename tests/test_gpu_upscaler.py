"""GPU parity of the HDR upscaler path (libhdrvae.so hdrvae_upscale*) against the CPU oracle
(oracle/upscaler_oracle.py, pinned bit for bit against the unmodified reference node) and its golden vectors.

Tolerances: the RRDB network runs with fp16 tensor-core operands and an fp32 residual stream, so the model output is
compared at rel-L2 <= 1e-2 (the bar BASELINE.json sets for 16-bit paths; measured ~1e-3); everything after the model
(hook, tiling, feather blend, YCbCr, median, local fix) is fp32 in the reference's operation order and is compared
at 1e-6 given the same model outputs."""
import os

import numpy as np
import pytest
import torch

from _metrics import GpuModel, rel_l2, rel_trimmed
from oracle import upscaler_oracle as uo
from oracle.make_golden_upscale import CASES, make_image

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def nets():
    from vae_decode_hdr_b200.upscaler import HdrUpscalerEngine
    out = {}
    for nb, gain in ((1, 1.0), (2, 1.0), (2, 40.0)):
        net = uo.build_upscaler(0, nb=nb, gain=gain)
        out[(nb, gain)] = (net, HdrUpscalerEngine(net.state_dict(), DEV))
    return out


@pytest.mark.parametrize("n,h,w", [(1, 16, 16), (2, 40, 56), (1, 9, 133), (3, 64, 32)])
@pytest.mark.parametrize("reversal", ["none", "atanh"])
def test_rrdbnet_forward_vs_oracle(nets, n, h, w, reversal):
    net, eng = nets[(2, 1.0)]
    assert eng.blocks == 2
    x = make_image(n, h, w, 5 + n, 3.0)
    with torch.no_grad():
        ref = net(x.movedim(-1, 1))
        if reversal == "atanh":
            ref = uo.reversal(ref, "atanh")
    got = eng.forward(x.to(DEV), reversal)
    assert got.shape == (n, 4 * h, 4 * w, 3)
    assert rel_l2(got.cpu(), ref.movedim(1, -1)) < 1e-2


def test_rrdbnet_tcgen05_vs_cuda_core_kernel(nets):
    """Same packed operands through the tcgen05 kernel and the CUDA-core validation kernel: only the fp32 summation
    order differs (plus the fp16 roundings it flips)."""
    from vae_decode_hdr_b200 import _native as N
    net, eng = nets[(1, 1.0)]
    x = make_image(2, 24, 40, 3, 3.0).to(DEV)
    a = eng.forward(x, "none")
    eng.set_conv_impl(N.CONV_DIRECT)
    try:
        b = eng.forward(x, "none")
    finally:
        eng.set_conv_impl(N.CONV_TCGEN05)
    assert rel_l2(a, b) < 3e-3


def test_old_arch_state_dict_gives_identical_model(nets):
    from vae_decode_hdr_b200.upscaler import HdrUpscalerEngine
    net, eng = nets[(2, 1.0)]
    eng_old = HdrUpscalerEngine(uo.state_dict_old_arch(net), DEV)
    x = make_image(1, 20, 24, 9, 3.0).to(DEV)
    assert torch.equal(eng.forward(x, "atanh"), eng_old.forward(x, "atanh"))
    eng_old.close()


def test_wrong_architecture_fails_loudly():
    from vae_decode_hdr_b200.upscaler import HdrUpscalerEngine
    net = uo.build_upscaler(0, nb=1)
    sd = dict(net.state_dict())
    sd["body.0.rdb1.conv1.weight"] = torch.zeros(16, 64, 3, 3)
    with pytest.raises(RuntimeError, match=r"body\.0\.rdb1\.conv1\.weight has shape \[16,64,3,3\]; want \[32,64,3,3\]"):
        HdrUpscalerEngine(sd, DEV)
    with pytest.raises(RuntimeError, match="no RRDB blocks"):
        HdrUpscalerEngine({"foo.weight": torch.zeros(4, 4, 3, 3)}, DEV)


@pytest.mark.parametrize("B,H,W,blur,fix,method", [(1, 24, 20, False, False, "bilinear"), (1, 530, 24, False, False, "bilinear"),
                                                   (1, 40, 600, True, True, "nearest-exact"), (2, 20, 28, True, True, "bilinear"),
                                                   (1, 520, 520, False, True, "bilinear"), (1, 36, 44, False, True, "area"),
                                                   (2, 30, 26, False, True, "bicubic"), (1, 36, 44, False, True, "bislerp"),
                                                   (2, 20, 28, True, True, "bislerp")])
def test_tiling_blend_and_recombination_are_exact_given_the_model(nets, B, H, W, blur, fix, method):
    net, eng = nets[(1, 1.0)] if max(H, W) > 512 else nets[(2, 40.0)]
    img = make_image(B, H, W, 31, 3.0)
    want = uo.upscale(img, uo.FakeDescriptor(GpuModel(eng)), blur, fix, method)
    got = eng.upscale(img.to(DEV), "atanh", blur, fix, method).cpu()
    assert got.shape == want.shape
    err = (got - want).abs()
    # atanhf vs torch.atanh differ by an ulp or two; everything else is the same fp32 operation sequence.  The 3x3
    # medians can pick a different (equal-within-ulp) sample, which is still an ulp-level difference.
    assert float(err.max()) <= 2e-5 * max(1.0, float(want.abs().max())), float(err.max())


@pytest.mark.parametrize("case", sorted(CASES))
def test_upscale_vs_reference_golden(nets, golden_dir, case):
    g = dict(np.load(os.path.join(golden_dir, case + ".npz"), allow_pickle=False))
    b, h, w, seed, gain, nb, last_gain, blur, fix, method = CASES[case]
    net, eng = nets[(nb, last_gain)]
    img = torch.from_numpy(g["image"])
    got = eng.upscale(img.to(DEV), "atanh", blur, fix, method).cpu()
    ref = torch.from_numpy(g["output"])
    if last_gain > 1.0:
        # conv_last x 40 drives the model output into the +-1 saturation of atanh(clamp(.)): ill-conditioned like the
        # decoder's logit modes, so the 0.5 % worst pixels are set aside
        assert rel_trimmed(got, ref, 0.005) < 1e-2, rel_trimmed(got, ref, 0.005)
    else:
        assert rel_l2(got, ref) < 1e-2, rel_l2(got, ref)


def test_node_surface_and_call(nets, golden_dir, monkeypatch):
    from vae_decode_hdr_b200 import NODE_CLASS_MAPPINGS, NODE_DISPLAY_NAME_MAPPINGS
    from vae_decode_hdr_b200.hdr_upscale_with_model import HDRUpscaleWithModel
    assert NODE_CLASS_MAPPINGS["HDRUpscaleWithModel"] is HDRUpscaleWithModel
    assert NODE_DISPLAY_NAME_MAPPINGS["HDRUpscaleWithModel"] == "HDR Upscale with Model"
    it = HDRUpscaleWithModel.INPUT_TYPES()["required"]
    assert list(it) == ["image", "model_name", "small_blur", "local_fix", "upscale_method"]
    assert it["upscale_method"][0] == ["nearest-exact", "bilinear", "area", "bicubic", "bislerp"]
    assert (HDRUpscaleWithModel.RETURN_TYPES, HDRUpscaleWithModel.FUNCTION, HDRUpscaleWithModel.CATEGORY) == \
        (("IMAGE",), "upscale", "HDR/Upscale")
    net, _ = nets[(2, 1.0)]
    node = HDRUpscaleWithModel()
    monkeypatch.setattr(node, "_load_model_internal", lambda name: uo.FakeDescriptor(net, 4, "ESRGAN"))
    g = dict(np.load(os.path.join(golden_dir, "up_a_single_tile.npz"), allow_pickle=False))
    (out,) = node.upscale(torch.from_numpy(g["image"]), "fake.pth", False, False, "bislerp")
    assert out.device.type == "cpu" and out.dtype == torch.float32 and out.shape == g["output"].shape
    assert rel_l2(out, torch.from_numpy(g["output"])) < 1e-2
    # the node's own defaults with local_fix ticked (ADVICE r1): bislerp is implemented, an unknown method is a ValueError
    (fixed,) = node.upscale(torch.from_numpy(g["image"]), "fake.pth", False, True, "bislerp")
    ref_fixed = uo.upscale(torch.from_numpy(g["image"]), uo.FakeDescriptor(net, 4, "ESRGAN"), False, True, "bislerp")
    assert rel_l2(fixed, ref_fixed) < 1e-2, rel_l2(fixed, ref_fixed)
    with pytest.raises(ValueError):
        node.upscale(torch.from_numpy(g["image"]), "fake.pth", False, True, "lanczos")


def test_c5_pipeline_decode_upscale_pack(nets):
    """Config C5 in small: HDR decode -> 4x HDR upscale -> half packing, all on the GPU through the node-level calls,
    against the oracle chain (reference decode math, reference upscaler math, numpy astype(float16))."""
    from oracle import hdr_oracle as ho
    from oracle.flux_decoder import build_decoder, make_latent
    from vae_decode_hdr_b200.engine import HdrVaeEngine, pack_half
    dec = build_decoder(0)
    eng = HdrVaeEngine(dec.state_dict(), DEV)
    net, up = nets[(2, 1.0)]
    z = make_latent(1, 8, 8, seed=77)
    img, _ = eng.decode(z.to(DEV), "moderate")
    big = up.upscale(img, "atanh")
    half = pack_half(big)
    assert half.dtype == torch.float16 and half.shape == (1, 256, 256, 3)
    assert np.array_equal(half.cpu().numpy(), big.cpu().numpy().astype(np.float16))        # the cast itself is bit-exact
    ref_img, _, _ = ho.simple_hdr_decode(dec, z, "moderate", 1.0)
    ref_big = uo.upscale(ref_img, uo.FakeDescriptor(net))
    ref_half = torch.from_numpy(ref_big.numpy().astype(np.float16)).float()
    assert rel_l2(half.float().cpu(), ref_half) < 1e-2, rel_l2(half.float().cpu(), ref_half)
    eng.close()


def test_rrdbnet_full_depth_nb23_vs_oracle():
    """The C5 model size (23 RRDBs = 69 dense blocks, 347 convs): error accumulation of the fp16-operand / fp32-stream
    plan through the full depth, on a small image so that the fp32 CPU oracle runs in seconds."""
    from vae_decode_hdr_b200.upscaler import HdrUpscalerEngine
    net = uo.build_upscaler(0, nb=23)
    eng = HdrUpscalerEngine(net.state_dict(), DEV)
    assert eng.blocks == 23
    x = make_image(1, 48, 40, 17, 3.0)
    with torch.no_grad():
        ref = net(x.movedim(-1, 1)).movedim(1, -1)
    got = eng.forward(x.to(DEV), "none").cpu()
    assert rel_l2(got, ref) < 1e-2, rel_l2(got, ref)
    eng.close()
