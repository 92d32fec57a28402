"""CPU tests of the SwinIR upscaler's host side and its fp32 oracle (tests/_swinir_oracle.py): the synthetic state dict's
keys and shapes, the oracle's Swin transformer layer against torchvision's independent SwinTransformerBlock, the region
mask on a padded non-square tile, key-layout detection, the node's pre-checks and reversal, and the oracle's tiling."""
import pytest
import torch

from _swinir_oracle import SwinLayer, build_swinir, region_mask
from oracle import upscaler_oracle as uo
from oracle.make_golden_upscale import make_image
from vae_decode_hdr_b200 import synthetic as S
from vae_decode_hdr_b200.upscaler import (SWIN_KEY, is_compact_state_dict, is_swinir_state_dict,
                                          reversal_for_architecture)

FORMS = [("pixelshuffle", 2), ("pixelshuffle", 4), ("pixelshuffledirect", 2), ("pixelshuffledirect", 4),
         ("nearest+conv", 2), ("nearest+conv", 4), ("", 1)]


@pytest.mark.parametrize("upsampler,s", FORMS)
@pytest.mark.parametrize("resi", ["1conv", "3conv"])
def test_synthetic_state_dict_has_the_oracle_keys_and_shapes(upsampler, s, resi):
    sd = S.random_swinir_state_dict(0, 60, (2, 1), 6, 2.0, upsampler, s, resi, True)
    net = build_swinir(0, 60, (2, 1), 6, 2.0, upsampler, s, resi, True)
    ref = net.state_dict()
    assert list(sd) == [k for k, _ in S.swinir_param_shapes(60, (2, 1), 6, 2.0, upsampler, s, resi, True)]
    assert set(sd) == set(ref)
    for k, v in sd.items():
        assert tuple(v.shape) == tuple(ref[k].shape), k
    assert torch.equal(sd["layers.0.residual_group.blocks.0.attn.relative_position_index"],
                       ref["layers.0.residual_group.blocks.0.attn.relative_position_index"])
    assert torch.equal(sd["layers.0.residual_group.blocks.1.attn_mask"], region_mask(64, 64, 4))
    assert "layers.0.residual_group.blocks.0.attn_mask" not in sd                     # even blocks do not shift
    tail = {"pixelshuffle": ["conv_before_upsample.0.weight", "upsample.0.weight", "conv_last.weight"],
            "pixelshuffledirect": ["upsample.0.weight"], "nearest+conv": ["conv_up1.weight", "conv_hr.weight"],
            "": ["conv_last.weight"]}[upsampler]
    assert all(k in sd for k in tail)
    assert ("upsample.2.weight" in sd) == (upsampler == "pixelshuffle" and s == 4)
    assert ("conv_up2.weight" in sd) == (upsampler == "nearest+conv" and s == 4)
    assert ("layers.1.conv.2.weight" in sd) == (resi == "3conv")
    assert "patch_embed.norm.weight" not in S.random_swinir_state_dict(0, 60, (1,), 6, 2.0, upsampler, s, resi, False)


def _torchvision_block(layer, dim, heads, shift):
    from torchvision.models.swin_transformer import SwinTransformerBlock
    tv = SwinTransformerBlock(dim, heads, [8, 8], [shift, shift], mlp_ratio=layer.mlp.fc1.out_features / dim,
                              norm_layer=torch.nn.LayerNorm)
    with torch.no_grad():
        tv.norm1.load_state_dict(layer.norm1.state_dict())
        tv.norm2.load_state_dict(layer.norm2.state_dict())
        tv.attn.qkv.load_state_dict(layer.attn.qkv.state_dict())
        tv.attn.proj.load_state_dict(layer.attn.proj.state_dict())
        tv.attn.relative_position_bias_table.copy_(layer.attn.relative_position_bias_table)
        tv.mlp[0].load_state_dict(layer.mlp.fc1.state_dict())
        tv.mlp[3].load_state_dict(layer.mlp.fc2.state_dict())
    return tv.eval()


@pytest.mark.parametrize("shift", [0, 4])
@pytest.mark.parametrize("dim,heads", [(180, 6), (60, 6)])          # head dim 30 and 10
@pytest.mark.parametrize("H,W", [(16, 24), (32, 16)])
def test_oracle_swin_layer_matches_torchvision(shift, dim, heads, H, W):
    g = torch.Generator().manual_seed(dim + shift + H)
    layer = SwinLayer(dim, heads, 2 * dim, shift)
    with torch.no_grad():
        for p in layer.parameters():
            p.copy_(torch.randn(p.shape, generator=g) * (0.5 if p.dim() == 1 else 1.0 / p.shape[-1] ** 0.5))
    layer.eval()
    tv = _torchvision_block(layer, dim, heads, shift)
    x = torch.randn(2, H, W, dim, generator=g)
    with torch.no_grad():
        want = tv(x)
        got = layer(x.reshape(2, H * W, dim), H, W).view(2, H, W, dim)
    err = float((got - want).norm() / want.norm())
    assert err <= 1e-5, err


def test_region_mask_on_a_padded_non_square_tile():
    """A 21 x 13 tile pads to 24 x 16: the rolled image's last 8 rows / columns split at 4 into regions 1 and 2."""
    H, W = 24, 16
    m = region_mask(H, W, 4)
    assert m.shape == (6, 64, 64)
    lab = torch.zeros(H, W, dtype=torch.long)
    for y in range(H):
        for x in range(W):
            lab[y, x] = 3 * (0 if y < H - 8 else 1 if y < H - 4 else 2) + (0 if x < W - 8 else 1 if x < W - 4 else 2)
    win = lab.view(3, 8, 2, 8).permute(0, 2, 1, 3).reshape(6, 64)
    want = torch.where(win[:, :, None] == win[:, None, :], 0.0, -100.0)
    assert torch.equal(m, want)
    assert bool((m[0] == 0).all()) and bool((m[-1] != 0).any())      # an interior window is one region, the corner is not


def test_detection():
    sw = S.random_swinir_state_dict(0, 60, (1,), 6, 2.0, "", 1, "1conv", False)
    assert is_swinir_state_dict(sw) and not is_compact_state_dict(sw)
    assert not is_swinir_state_dict(S.random_upscaler_state_dict(0, nb=1))
    assert not is_swinir_state_dict(S.random_compact_state_dict(0, nf=16, nc=1, s=2))
    assert not is_swinir_state_dict(S.random_span_state_dict(0, nf=16, s=2))
    for mark in ("layers.0.residual_group.blocks.0.conv_block.cab.0.weight",
                 "layers.0.residual_group.overlap_attn.qkv.weight", "relative_position_index_SA"):
        hat = dict(sw)
        hat[mark] = torch.zeros(4)
        assert SWIN_KEY in hat and not is_swinir_state_dict(hat)


def test_node_skips_the_rrdbnet_precheck_and_picks_atanh(monkeypatch):
    from vae_decode_hdr_b200 import hdr_upscale_with_model as M
    sd = S.random_swinir_state_dict(0, 60, (1,), 6, 2.0, "pixelshuffle", 4, "1conv", True)
    called = []
    monkeypatch.setattr(M, "rrdbnet_scale", lambda d: called.append(1) or 1)

    class Stop(Exception):
        pass

    class FakeEngine:
        def __init__(self, state_dict, device):
            raise Stop()
    monkeypatch.setattr(M, "HdrUpscalerEngine", FakeEngine)
    with pytest.raises(Stop):
        M.HDRUpscaleWithModel._new_engine(uo.FakeDescriptor(build_swinir(0, 60, (1,), 6), 4, "SwinIR"), "cpu")
    assert called == []
    assert reversal_for_architecture("SwinIR") == "atanh"


@pytest.mark.parametrize("upsampler,s", [("", 1), ("pixelshuffledirect", 2), ("pixelshuffle", 4)])
def test_oracle_upscale_tiles_a_swinir_descriptor(upsampler, s):
    net = build_swinir(3, 24, (2,), 3, 2.0, upsampler, s)
    img = make_image(1, 20, 28, 3, 1.0).clamp(0, 1)
    out = uo.upscale(img, uo.FakeDescriptor(net, s, "SwinIR"), False, False, "bilinear")
    assert out.shape == (1, s * 20, s * 28, 3) and bool(torch.isfinite(out).all())
