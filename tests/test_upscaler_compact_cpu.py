"""CPU tests of the Real-ESRGAN Compact (SRVGGNetCompact) pieces: the oracle's key layout for the published model shapes,
its forward against an independent functional formulation, the synthetic state dict, the feather-blended tiling at the
Compact's 1x / 2x scales, and the node's scale checks that run before any GPU work."""
import os

import pytest
import torch
import torch.nn.functional as F

from _compact_oracle import build_compact
from oracle import upscaler_oracle as uo


@pytest.mark.parametrize("nc,n_convs,n_slopes", [(32, 34, 33), (16, 18, 17)])     # realesr-general-x4v3, animevideov3
def test_compact_oracle_key_layout(nc, n_convs, n_slopes):
    from vae_decode_hdr_b200.synthetic import random_compact_state_dict
    sd = build_compact(0, nf=64, nc=nc, s=4).state_dict()
    convs = [k for k, v in sd.items() if k.endswith(".weight") and v.dim() == 4]
    slopes = [k for k, v in sd.items() if k.endswith(".weight") and v.dim() == 1]
    assert len(convs) == n_convs and len(slopes) == n_slopes
    assert all(sd[k[:-len("weight")] + "bias"].shape == (sd[k].shape[0],) for k in convs)
    assert convs == [f"body.{2 * m}.weight" for m in range(nc + 2)]
    assert slopes == [f"body.{2 * k + 1}.weight" for k in range(nc + 1)]
    assert sd["body.0.weight"].shape == (64, 3, 3, 3)
    assert sd[f"body.{2 * nc + 2}.weight"].shape == (48, 64, 3, 3) and sd[f"body.{2 * nc + 2}.bias"].shape == (48,)
    assert all(sd[k].shape == (64,) for k in slopes)
    assert not any(k.startswith("conv_first") for k in sd)
    # the synthetic state dict (tools, benchmarks) has exactly the oracle's keys and shapes
    syn = random_compact_state_dict(0, 64, nc, 4)
    assert list(syn) == list(sd) and all(syn[k].shape == sd[k].shape for k in sd)


def test_compact_oracle_slopes_are_random_per_channel():
    net = build_compact(3, nf=16, nc=2, s=2)
    w = net.body[1].weight
    assert float(w.min()) < 0.0 < float(w.max()) and len(set(w.tolist())) == 16


@pytest.mark.parametrize("nf,nc,s", [(16, 2, 4), (24, 0, 2), (8, 3, 1)])
def test_compact_oracle_forward_vs_functional(nf, nc, s):
    net = build_compact(7, nf=nf, nc=nc, s=s)
    sd = net.state_dict()
    g = torch.Generator().manual_seed(11)
    x = torch.randn(2, 3, 9, 13, generator=g)
    h = x
    for i in range(2 * nc + 3):
        if i % 2:
            h = F.prelu(h, sd[f"body.{i}.weight"])
        else:
            h = F.conv2d(h, sd[f"body.{i}.weight"], sd[f"body.{i}.bias"], padding=1)
    want = F.pixel_shuffle(h, s) + x.repeat_interleave(s, dim=2).repeat_interleave(s, dim=3)
    with torch.no_grad():
        got = net(x)
    assert got.shape == (2, 3, 9 * s, 13 * s)
    assert torch.allclose(got, want, atol=1e-6, rtol=0)


@pytest.mark.parametrize("s", [1, 2])
def test_tiled_scale_at_compact_scales_is_exact_resampling(s):
    """For a function without spatial context the feather-blended result equals the untiled one, at 1x and 2x too."""
    x = torch.rand(1, 3, 70, 45)
    f = lambda a: F.interpolate(a, scale_factor=s, mode="nearest") * 0.5 + 0.25   # noqa: E731
    tiled = uo.tiled_scale(x, f, tile_x=32, tile_y=32, overlap=8, upscale_amount=s)
    assert tiled.shape == (1, 3, 70 * s, 45 * s)
    assert torch.allclose(tiled, f(x), atol=1e-6)


def test_compact_layout_detection():
    from vae_decode_hdr_b200.synthetic import random_compact_state_dict, random_upscaler_state_dict
    from vae_decode_hdr_b200.upscaler import is_compact_state_dict
    assert is_compact_state_dict(random_compact_state_dict(0, 16, 1, 2))
    assert not is_compact_state_dict(random_upscaler_state_dict(0, 1))
    assert not is_compact_state_dict(uo.state_dict_old_arch(uo.build_upscaler(0, nb=1)))


def test_scale_query_fails_without_a_model():
    from vae_decode_hdr_b200 import _native
    if not os.path.isfile(_native.LIB_PATH):
        _native.build_library()
    lib = _native.load_library()
    assert lib.hdrvae_upscaler_scale(None) < 0 and b"not loaded" in lib.hdrvae_last_error()


def test_node_rejects_rrdbnet_of_another_scale_before_gpu_work():
    """ESRGAN 2x: the node names the scale and raises before a library call (there is no device here)."""
    from vae_decode_hdr_b200.hdr_upscale_with_model import HDRUpscaleWithModel
    desc = uo.FakeDescriptor(uo.build_upscaler(0, nb=1), 2, "ESRGAN")
    with pytest.raises(RuntimeError, match="scale 2"):
        HDRUpscaleWithModel._new_engine(desc, torch.device("cuda", 0))
