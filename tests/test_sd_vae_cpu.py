"""SD1.x / SDXL VAEs without a GPU: the synthetic weights and the oracle agree on the 4-channel decoder, the oracle's SD
first stage applies post_quant_conv before the decoder, the node collects post_quant_conv from the VAE object, and the
library exports the latent-channel query."""
import os

import pytest
import torch
import torch.nn.functional as F
from torch import nn

from oracle.flux_decoder import build_decoder

from _sd_oracle import FakeComfySDVAE, SDFirstStage, build_sd_decoder, make_sd_latent


def test_synthetic_sd_shapes_equal_the_oracle():
    from vae_decode_hdr_b200.synthetic import decoder_param_shapes, random_decoder_state_dict
    sd_oracle = build_sd_decoder(0)
    ref = sd_oracle.decoder.state_dict()
    assert {k: tuple(v.shape) for k, v in ref.items()} == dict(decoder_param_shapes(4))
    assert tuple(ref["conv_in.weight"].shape) == (512, 4, 3, 3)
    sd = random_decoder_state_dict(0, z_channels=4)
    assert {k: tuple(v.shape) for k, v in sd.items()} == dict(decoder_param_shapes(z_channels=4))
    # Flux's 49 545 475 minus the 12 input channels of conv_in (12 * 9 * 512); post_quant_conv adds 4 * 4 + 4
    assert sum(v.numel() for v in sd.values()) == 49_490_179 == 49_545_475 - 12 * 9 * 512
    assert sum(p.numel() for p in sd_oracle.post_quant_conv.parameters()) == 20
    assert sum(p.numel() for p in sd_oracle.parameters()) == 49_490_179 + 20
    # the defaults stay the Flux decoder
    assert dict(decoder_param_shapes()) == {k: tuple(v.shape) for k, v in build_decoder(0).state_dict().items()}


def test_sd_fake_vae_decode_applies_post_quant_conv_first():
    m = build_sd_decoder(1)
    with torch.no_grad():
        m.post_quant_conv.bias.add_(0.25)          # a bias that would show if it were skipped
    vae = FakeComfySDVAE(m)
    z = make_sd_latent(1, 3, 5, seed=11)
    assert vae.first_stage_model.post_quant_conv is m.post_quant_conv and vae.first_stage_model.decoder is m.decoder
    got = vae.decode(z)
    with torch.no_grad():
        y = m.decoder(F.conv2d(z, m.post_quant_conv.weight, m.post_quant_conv.bias))
        plain = m.decoder(z)
    want = torch.clamp((y + 1.0) / 2.0, 0.0, 1.0).movedim(1, -1)
    assert got.shape == (1, 24, 40, 3)
    assert torch.equal(got, want)
    assert not torch.equal(got, torch.clamp((plain + 1.0) / 2.0, 0.0, 1.0).movedim(1, -1))
    with torch.no_grad():
        assert torch.equal(m.features(z), m.decoder.features(m.post_quant_conv(z)))
    assert m.conv_out is m.decoder.conv_out


class _Stage:
    pass


@pytest.mark.parametrize("case", ["conv", "absent", "none", "identity"])
def test_node_collects_post_quant_conv(case):
    from vae_decode_hdr_b200.hdr_vae_decode import _engine_state_dict, _post_quant_conv_of, _weights_key
    from vae_decode_hdr_b200.synthetic import SyntheticVAE
    dec = build_decoder(0)
    vae = SyntheticVAE({}, device="cpu")
    stage = _Stage()
    stage.decoder = dec
    pqc = nn.Conv2d(4, 4, 1)
    if case == "conv":
        stage.post_quant_conv = pqc
    elif case == "none":
        stage.post_quant_conv = None
    elif case == "identity":
        stage.post_quant_conv = nn.Identity()
    vae.first_stage_model = stage
    got = _post_quant_conv_of(vae)
    sd = _engine_state_dict(dec, got)
    key0 = _weights_key(dec, got)
    if case == "conv":
        assert got is pqc
        assert torch.equal(sd["post_quant_conv.weight"], pqc.weight) and torch.equal(sd["post_quant_conv.bias"], pqc.bias)
        assert len(sd) == len(dec.state_dict()) + 2
        with torch.no_grad():
            pqc.weight.mul_(2.0)                   # an in-place change of post_quant_conv alone must change the key
        assert _weights_key(dec, got) != key0
        assert _weights_key(dec, got)[0] == id(dec)
    else:
        assert got is None
        assert not any(k.startswith("post_quant_conv") for k in sd) and len(sd) == len(dec.state_dict())
        assert key0 == _weights_key(dec)


def test_bias_less_post_quant_conv_sends_zero_bias():
    from vae_decode_hdr_b200.hdr_vae_decode import _engine_state_dict
    pqc = nn.Conv2d(4, 4, 1, bias=False)
    sd = _engine_state_dict(build_decoder(0), pqc)
    assert torch.equal(sd["post_quant_conv.bias"], torch.zeros(4))


def test_synthetic_vae_carries_post_quant_conv():
    from vae_decode_hdr_b200.hdr_vae_decode import _post_quant_conv_of
    from vae_decode_hdr_b200.synthetic import SyntheticVAE
    pqc = nn.Conv2d(4, 4, 1)
    assert _post_quant_conv_of(SyntheticVAE({}, device="cpu", post_quant_conv=pqc)) is pqc
    assert _post_quant_conv_of(SyntheticVAE({}, device="cpu")) is None
    assert not hasattr(SyntheticVAE({}, device="cpu").first_stage_model, "post_quant_conv")


def test_library_exports_latent_channels():
    from vae_decode_hdr_b200 import _native
    if not os.path.isfile(_native.LIB_PATH):
        _native.build_library()
    lib = _native.load_library()
    assert hasattr(lib, "hdrvae_latent_channels")
    assert "hdrvae_latent_channels" in _native.SIGNATURES
    # before any weights are loaded (here: no context at all) the query fails with a message instead of guessing
    assert lib.hdrvae_latent_channels(None) < 0 and b"not loaded" in lib.hdrvae_last_error()


def test_sd_first_stage_is_an_oracle_decoder():
    """hdr_oracle.simple_hdr_decode and the test metrics read .features, .conv_out and the parameters' device / dtype."""
    from oracle import hdr_oracle as ho
    m = build_sd_decoder(0)
    assert isinstance(m, SDFirstStage)
    z = make_sd_latent(1, 2, 2, seed=3)
    out, st, pre = ho.simple_hdr_decode(m, z, "conservative", 1.0)
    assert out.shape == (1, 16, 16, 3) and pre.shape == (1, 128, 16, 16)
    with torch.no_grad():
        assert torch.equal(pre, m.decoder.features(m.post_quant_conv(z)))
