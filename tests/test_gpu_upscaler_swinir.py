"""GPU tests of the SwinIR upscaler: the library's forward against the fp32 oracle (tests/_swinir_oracle.py) for every
upsampler form at each of its scales, 1conv / 3conv, patch_norm on / off, embed_dim 60 and 180, padded and unpadded tiles,
tiles under 128 pixels and n > 1, and one full-depth SwinIR-M; the reversal hooks; HDR-range input; the tcgen05 convs
against the CUDA-core validation kernel; the LayerNorm and window-attention entries against fp64; everything after the
model given the model; the node; and the rejections.

The model output is compared at rel-L2 <= 1e-2 (fp16 operands, fp32 accumulation, an fp32 residual stream); everything
after the model is fp32 in the reference's operation order.  Each comparison prints the error it measured."""
import math

import pytest
import torch

from _metrics import GpuModel, rel_l2, rel_trimmed
from _swinir_oracle import build_swinir, region_mask, rel_index
from oracle import upscaler_oracle as uo
from oracle.make_golden_upscale import make_image

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
FORMS = [("pixelshuffle", 2), ("pixelshuffle", 4), ("pixelshuffledirect", 2), ("pixelshuffledirect", 4),
         ("nearest+conv", 2), ("nearest+conv", 4), ("", 1)]


@pytest.fixture(scope="module")
def swin():
    """(C, depths, heads, upsampler, s, resi, patch_norm) -> (oracle net on the GPU, engine), built on first use."""
    from vae_decode_hdr_b200.upscaler import HdrUpscalerEngine
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    cache = {}

    def get(C=60, depths=(2, 2), heads=6, upsampler="pixelshuffle", s=4, resi="1conv", pn=True):
        key = (C, depths, heads, upsampler, s, resi, pn)
        if key not in cache:
            net = build_swinir(len(cache) + 7, C, depths, heads, 2.0, upsampler, s, resi, pn)
            cache[key] = (net.to(DEV), HdrUpscalerEngine(net.state_dict(), DEV))
        return cache[key]
    yield get
    for _, eng in cache.values():
        eng.close()


def _oracle(net, x_bhwc, reversal):
    with torch.no_grad():
        y = net(x_bhwc.to(DEV).movedim(-1, 1))
    if reversal != "none":
        y = uo.reversal(y, reversal)
    return y.movedim(1, -1).cpu()


# multiples of 8; padded (not multiples of 8, both sides); below 128 pixels; n > 1
SHAPES = [(1, 16, 24), (2, 21, 13), (1, 8, 12), (3, 9, 17)]


@pytest.mark.parametrize("n,h,w", SHAPES)
@pytest.mark.parametrize("upsampler,s", FORMS)
def test_swinir_forward_vs_oracle(swin, upsampler, s, n, h, w):
    net, eng = swin(upsampler=upsampler, s=s)
    assert (eng.scale, eng.blocks) == (s, 2)
    x = make_image(n, h, w, 5 + n, 1.0).clamp(0, 1)
    got = eng.forward(x.to(DEV), "none").cpu()
    assert got.shape == (n, s * h, s * w, 3)
    err = rel_l2(got, _oracle(net, x, "none"))
    print(f"swinir C60 {upsampler or 'none'} {s}x {n}x{h}x{w}: rel-L2 {err:.2e}")
    assert err < 1e-2, err


@pytest.mark.parametrize("C,heads", [(180, 6), (60, 6)])
@pytest.mark.parametrize("resi,pn", [("3conv", False), ("1conv", False), ("3conv", True)])
@pytest.mark.parametrize("upsampler,s", [("nearest+conv", 4), ("pixelshuffledirect", 2)])
def test_swinir_variants_vs_oracle(swin, C, heads, resi, pn, upsampler, s):
    net, eng = swin(C, (2, 1), heads, upsampler, s, resi, pn)
    x = make_image(2, 21, 30, 9, 1.0).clamp(0, 1)
    got = eng.forward(x.to(DEV), "none").cpu()
    err = rel_l2(got, _oracle(net, x, "none"))
    print(f"swinir C{C} {resi} patch_norm {pn} {upsampler} {s}x: rel-L2 {err:.2e}")
    assert err < 1e-2, err


def test_full_depth_swinir_m_vs_oracle(swin):
    net, eng = swin(180, (6,) * 6, 6, "pixelshuffle", 4, "1conv", True)
    assert eng.blocks == 6
    x = make_image(1, 64, 64, 21, 1.0).clamp(0, 1)
    got = eng.forward(x.to(DEV), "none").cpu()
    err = rel_l2(got, _oracle(net, x, "none"))
    print(f"swinir-M 6x6 blocks 4x 64x64: rel-L2 {err:.2e}")
    assert err < 1e-2, err


@pytest.mark.parametrize("reversal", ["atanh", "logit"])
def test_swinir_forward_with_reversal_vs_oracle(swin, reversal):
    """The reversal hook is ill-conditioned next to its clamps: the 0.5 % worst pixels are set aside."""
    net, eng = swin(upsampler="pixelshuffle", s=2)
    x = make_image(2, 40, 56, 8, 1.0).clamp(0, 1)
    got = eng.forward(x.to(DEV), reversal).cpu()
    err = rel_trimmed(got, _oracle(net, x, reversal), 0.005)
    print(f"swinir 2x {reversal}: trimmed rel-L2 {err:.2e}")
    assert err < 1e-2, err


def test_swinir_hdr_range_input(swin):
    net, eng = swin(upsampler="nearest+conv", s=4)
    x = make_image(1, 48, 40, 17, 16.0)
    assert float(x.abs().max()) > 8.0
    got = eng.forward(x.to(DEV), "none").cpu()
    assert bool(torch.isfinite(got).all())
    err = rel_l2(got, _oracle(net, x, "none"))
    print(f"swinir HDR amplitude 16: rel-L2 {err:.2e}")
    assert err < 1e-2, err


@pytest.mark.parametrize("C,upsampler,s", [(180, "pixelshuffle", 4), (60, "", 1)])
def test_swinir_tcgen05_vs_cuda_core_kernel(swin, C, upsampler, s):
    from vae_decode_hdr_b200 import _native as N
    _, eng = swin(C, (2, 1), 6, upsampler, s, "3conv" if C == 60 else "1conv", True)
    x = make_image(2, 24, 40, 3, 1.0).clamp(0, 1).to(DEV)
    a = eng.forward(x, "none")
    eng.set_conv_impl(N.CONV_DIRECT)
    try:
        b = eng.forward(x, "none")
    finally:
        eng.set_conv_impl(N.CONV_TCGEN05)
    err = rel_l2(a, b)
    print(f"swinir C{C} {s}x tcgen05 vs CUDA core: rel-L2 {err:.2e}")
    assert err < 3e-3, err


# ---- the two new kernels through their entries, against fp64 -------------------------------------------------------
@pytest.fixture(scope="module")
def ctx():
    import ctypes as C
    from vae_decode_hdr_b200 import _native as N
    lib = N.load_library()
    c = C.c_void_p()
    N.check(lib.hdrvae_create(C.byref(c), 0), "hdrvae_create")
    yield lib, c
    lib.hdrvae_destroy(c)


@pytest.mark.parametrize("C,yc,f16", [(180, 184, True), (60, 64, True), (180, 180, False), (256, 256, True)])
def test_layernorm_entry_vs_fp64(ctx, C, yc, f16):
    from vae_decode_hdr_b200 import _native as N
    lib, c = ctx
    g = torch.Generator().manual_seed(C + yc)
    P = 3 * 37 * 11
    x = (torch.randn(P, C, generator=g) * 3 + torch.randn(P, 1, generator=g) * 5).to(DEV)
    gamma = (1 + 0.3 * torch.randn(C, generator=g)).to(DEV)
    beta = (0.2 * torch.randn(C, generator=g)).to(DEV)
    y = torch.full((P, yc if f16 else C), float("nan"), dtype=torch.float16 if f16 else torch.float32, device=DEV)
    N.check(lib.hdrvae_layernorm(c, x.data_ptr(), P, C, gamma.data_ptr(), beta.data_ptr(), y.data_ptr(),
                                 N.F16 if f16 else N.F32, yc, torch.cuda.current_stream().cuda_stream), "hdrvae_layernorm")
    torch.cuda.synchronize()
    xd = x.double()
    want = (xd - xd.mean(1, keepdim=True)) / torch.sqrt(xd.var(1, unbiased=False, keepdim=True) + 1e-5) * gamma.double() + beta.double()
    got = y[:, :C].double()
    # fp32 statistics: a few ulp of the normalised value; fp16 output: half an ulp
    bound = 2.0 ** -19 * (want.abs() + gamma.double().abs() * 4 + 1) + (want.abs() * 2.0 ** -11 + 2.0 ** -24 if f16 else 0)
    ratio = float(((got - want).abs() / bound).max())
    print(f"layernorm C {C} {'fp16' if f16 else 'fp32'}: max err/bound {ratio:.3f}")
    assert ratio <= 1.0
    if f16 and yc > C:
        assert bool((y[:, C:] == 0).all()), "pad channels of the fp16 output must be zero"


def _attention_fp64(qkv, table, heads, H, W, shift):
    """SwinIR's window attention in fp64 from the kernel's operands (q pre-scaled, heads padded to 32)."""
    B = qkv.shape[0]
    t = qkv.double().view(B, H, W, 3, heads, 32)
    if shift:
        t = torch.roll(t, shifts=(-shift, -shift), dims=(1, 2))
    win = t.view(B, H // 8, 8, W // 8, 8, 3, heads, 32).permute(0, 1, 3, 5, 6, 2, 4, 7).reshape(-1, 3, heads, 64, 32)
    q, k, v = win[:, 0], win[:, 1], win[:, 2]
    s = q @ k.transpose(-1, -2) + table.double()[rel_index().view(-1)].view(64, 64, heads).permute(2, 0, 1)
    if shift:
        nW = (H // 8) * (W // 8)
        s = (s.view(B, nW, heads, 64, 64) + region_mask(H, W, shift).double().to(s.device)[None, :, None]).view(-1, heads, 64, 64)
    p = s.softmax(-1)
    o = p @ v
    mag = p @ v.abs()                                                     # for the bound
    def back(z):
        z = z.view(B, H // 8, W // 8, heads, 8, 8, 32).permute(0, 1, 4, 2, 5, 3, 6).reshape(B, H, W, heads * 32)
        return torch.roll(z, shifts=(shift, shift), dims=(1, 2)) if shift else z
    return back(o), back(mag)


@pytest.mark.parametrize("B,H,W,heads,shift", [(1, 16, 24, 6, 0), (1, 16, 24, 6, 4), (2, 24, 16, 3, 4), (3, 8, 8, 2, 4),
                                               (2, 32, 40, 8, 0)])
def test_window_attention_entry_vs_fp64(ctx, B, H, W, heads, shift):
    from vae_decode_hdr_b200 import _native as N
    lib, c = ctx
    g = torch.Generator().manual_seed(B * 100 + H + W + heads + shift)
    qkv = torch.randn(B, H, W, 3, heads, 32, generator=g)
    qkv[..., 30:] = 0                                                    # a head dimension of 30 padded to 32
    qkv[:, :, :, 0] *= 30 ** -0.5
    qkv = qkv.to(torch.float16).view(B, H, W, -1).to(DEV)
    table = torch.randn(225, heads, generator=g).to(DEV)
    o = torch.full((B, H, W, heads * 32), float("nan"), dtype=torch.float16, device=DEV)
    N.check(lib.hdrvae_window_attention(c, qkv.data_ptr(), B, H, W, heads, table.data_ptr(), shift, o.data_ptr(),
                                        torch.cuda.current_stream().cuda_stream), "hdrvae_window_attention")
    torch.cuda.synchronize()
    want, mag = _attention_fp64(qkv, table, heads, H, W, shift)
    # P rounded to fp16 before P V (2^-11 relative on each weight), fp32 accumulation and exp, fp16 output rounding
    bound = 2.0 ** -10 * mag + 2.0 ** -11 * want.abs() + 2.0 ** -20
    ratio = float(((o.double() - want).abs() / bound).max())
    print(f"window attention B{B} {H}x{W} heads {heads} shift {shift}: max err/bound {ratio:.3f}")
    assert ratio <= 1.0
    assert bool((o.view(B, H, W, heads, 32)[..., 30:] == 0).all())


# ---- after the model, node, rejections -------------------------------------------------------------------------------
_AFTER_MODEL_CASES = [(1, 530, 24, False, False, "bilinear", "atanh"), (1, 36, 44, False, True, "bislerp", "logit"),
                      (2, 30, 26, True, True, "bicubic", "atanh")]


@pytest.mark.parametrize("B,H,W,blur,fix,method,reversal", _AFTER_MODEL_CASES)
@pytest.mark.parametrize("upsampler,s", [("", 1), ("pixelshuffledirect", 2), ("pixelshuffle", 4)])
def test_tiling_blend_and_recombination_are_exact_given_the_model(swin, upsampler, s, B, H, W, blur, fix, method, reversal):
    _, eng = swin(24, (2,), 3, upsampler, s)
    img = make_image(B, H, W, 31, 1.0).clamp(0, 1)
    arch = "SwinIR" if reversal == "atanh" else "SPAN"                # the oracle picks the reversal by name
    want = uo.upscale(img, uo.FakeDescriptor(GpuModel(eng), s, arch), blur, fix, method)
    got = eng.upscale(img.to(DEV), reversal, blur, fix, method).cpu()
    assert got.shape == want.shape == (B, s * H, s * W, 3)
    err = (got - want).abs()
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


def test_node_runs_a_swinir_model_with_atanh_and_its_cache(monkeypatch, tmp_path):
    from vae_decode_hdr_b200 import upscaler as U
    from vae_decode_hdr_b200.hdr_upscale_with_model import HDRUpscaleWithModel
    net = build_swinir(12, 24, (2,), 3, 2.0, "pixelshuffle", 2)
    desc = uo.FakeDescriptor(net, 2, "SwinIR")
    node, calls = _node_with(monkeypatch, desc, str(tmp_path / "swinir_2x.pth"))
    seen = []
    real = U.HdrUpscalerEngine.upscale

    def spy(self, image, reversal, *a, **k):
        seen.append(reversal)
        return real(self, image, reversal, *a, **k)
    monkeypatch.setattr(U.HdrUpscalerEngine, "upscale", spy)
    img = make_image(1, 20, 28, 12, 1.0).clamp(0, 1)
    try:
        (a,) = node.upscale(img, "swinir_2x.pth", True, True, "bislerp")
        (b,) = node.upscale(img, "swinir_2x.pth", True, True, "bislerp")
        assert len(calls) == 1 and seen == ["atanh", "atanh"]
        assert a.shape == (1, 40, 56, 3) and torch.equal(a, b)
        ref = uo.upscale(img, desc, True, True, "bislerp")
        assert rel_l2(a, ref) < 1e-2, rel_l2(a, ref)
    finally:
        HDRUpscaleWithModel.release_memory()


def test_node_rejects_a_descriptor_scale_the_swinir_weights_contradict(monkeypatch):
    net = build_swinir(13, 24, (1,), 3, 2.0, "pixelshuffle", 4)
    node, _ = _node_with(monkeypatch, uo.FakeDescriptor(net, 2, "SwinIR"))
    with pytest.raises(RuntimeError, match=r"scale 2.*4x"):
        node.upscale(make_image(1, 16, 16, 1, 1.0), "wrong.pth")


def _sd(**k):
    from vae_decode_hdr_b200.synthetic import random_swinir_state_dict
    a = dict(seed=0, embed_dim=24, depths=(2,), heads=3, mlp_ratio=2.0, upsampler="pixelshuffle", s=2)
    a.update(k)
    return random_swinir_state_dict(**a)


def _rejects(sd, pattern):
    from vae_decode_hdr_b200.upscaler import HdrUpscalerEngine
    with pytest.raises(RuntimeError, match=pattern):
        HdrUpscalerEngine(sd, DEV)


def test_swinir_rejections_name_the_tensor():
    sd = _sd()
    sd["layers.0.residual_group.blocks.0.conv_block.cab.0.weight"] = torch.zeros(8, 24, 3, 3)
    _rejects(sd, r"conv_block\.cab\.0\.weight has shape \[8,24,3,3\]: a HAT model")
    sd = _sd()
    sd["upsample.0.weight"], sd["upsample.0.bias"] = torch.zeros(576, 64, 3, 3), torch.zeros(576)          # 3x
    _rejects(sd, r"upsample\.0\.weight has shape \[576,64,3,3\]; want \[256,64,3,3\]")
    sd = _sd(s=4)
    sd["upsample.4.weight"], sd["upsample.4.bias"] = torch.zeros(256, 64, 3, 3), torch.zeros(256)          # 8x
    _rejects(sd, r"upsample\.4\.weight has shape \[256,64,3,3\]: a third 2x stage")
    sd = _sd(upsampler="pixelshuffledirect")
    sd["upsample.0.weight"], sd["upsample.0.bias"] = torch.zeros(27, 24, 3, 3), torch.zeros(27)            # 3x direct
    _rejects(sd, r"upsample\.0\.weight has shape \[27,24,3,3\]; want \[3\*scale\^2,24,3,3\] with scale 2 or 4")
    sd = _sd()
    for k in [k for k in sd if k.endswith("relative_position_bias_table")]:
        sd[k] = torch.zeros(169, 3)                                                                       # window 7
    _rejects(sd, r"relative_position_bias_table has shape \[169,3\]; want \[225,heads\]")
    _rejects(_sd(embed_dim=66, heads=2), r"has shape \[225,2\]: embed_dim 66 over 2 heads")               # hd 33
    sd = _sd()
    sd["conv_first.weight"] = torch.zeros(24, 1, 3, 3)                                                    # in_chans 1
    _rejects(sd, r"conv_first\.weight has shape \[24,1,3,3\]; want \[embed_dim,3,3,3\]")
    sd = _sd()
    sd["absolute_pos_embed"] = torch.zeros(1, 64, 24)
    _rejects(sd, r"absolute_pos_embed has shape \[1,64,24\]")
    sd = _sd()
    del sd["layers.0.residual_group.blocks.1.mlp.fc2.bias"]
    _rejects(sd, r"lacks layers\.0\.residual_group\.blocks\.1\.mlp\.fc2\.bias \(want shape \[24\]\)")
    sd = _sd()
    sd["layers.0.residual_group.blocks.1.attn.proj.weight"] = torch.zeros(24, 20)
    _rejects(sd, r"blocks\.1\.attn\.proj\.weight has shape \[24,20\]; want \[24,24\]")


def test_swinir_refuses_a_tile_side_too_short_for_the_reflect_pad(swin):
    _, eng = swin(upsampler="", s=1)
    with pytest.raises(RuntimeError, match=r"tile side of 3 pixels is too short for the reflect pad of 5 pixels"):
        eng.forward(torch.rand(1, 3, 16, 3, device=DEV), "none")
