"""The oracle against the committed outputs of the unmodified reference node
(tests/golden/*.npz, generator oracle/make_golden.py) — no GPU needed."""
import glob
import os

import numpy as np
import pytest
import torch

from oracle import hdr_oracle as ho
from oracle.flux_decoder import FakeComfyVAE, build_decoder, weight_fingerprint
from oracle.make_golden import apply_variant
from oracle.ref_loader import load_reference_node, reference_available

MODES = list(ho.HDR_MODES)
CASES = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.npz"))
               if not os.path.basename(p).startswith("up_"))


def _load(golden_dir, name):
    return dict(np.load(os.path.join(golden_dir, name + ".npz"), allow_pickle=False))


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a))


def _bhwc_view_of_nchw(a):
    """ComfyUI returns decode().movedim(1,-1): BHWC view over NCHW storage (SURVEY.md §3.2)."""
    return _t(a).movedim(-1, 1).contiguous().movedim(1, -1)


def test_cases_present():
    assert {"a_b1_4x4", "b_b2_4x6", "c_nohdr_b1_4x4", "d_nonorm_b1_4x4"} <= set(CASES)


@pytest.mark.parametrize("case", CASES)
def test_analysis_stats_match_reference(golden_dir, case):
    g = _load(golden_dir, case)
    an = ho.analyze(_t(g["pre_conv_out"]), _t(g["conv_w"]), _t(g["conv_b"]))
    st = an["stats"]
    for grp, keys in (("pre", ("min", "max", "mean", "std")), ("post", ("min", "max", "mean", "std")),
                      ("conv", ("min", "max", "mean"))):
        for k in keys:
            ref = float(g[f"{grp}_stats.{k}"])
            assert st[f"{grp}_{k}"] == pytest.approx(ref, rel=2e-6, abs=2e-7), (grp, k)
    want = {"SIGMOID": ho.NORM_SIGMOID, "TANH": ho.NORM_TANH, "": ho.NORM_NONE}[str(g["norm_function"])]
    assert st["norm_function"] == want
    np.testing.assert_allclose(an["standard"].numpy(), g["final_result"], rtol=0, atol=2e-7)


@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("mode", MODES)
def test_intelligent_matches_reference(golden_dir, case, mode):
    g = _load(golden_dir, case)
    pre = _t(g["pre_conv_out"])
    # feed the reference's own final_result/stats so only the restated HDR math is under test
    st = {"pre_min": float(g["pre_stats.min"]), "pre_max": float(g["pre_stats.max"]),
          "pre_mean": float(g["pre_stats.mean"]),
          "norm_function": {"SIGMOID": 1, "TANH": 2, "": 0}[str(g["norm_function"])]}
    out, ost = ho.intelligent(_bhwc_view_of_nchw(g["final_result"]), pre, st, mode)
    key = f"intelligent.{mode}"
    if key in g:
        np.testing.assert_array_equal(out.numpy(), g[key])   # same ops, same order: bit-exact
    else:
        # reference raised (TypeError: torch.max(1.0)) -> bypass; our documented rule: linear LDR image
        assert str(g[key + ".error"]) == "TypeError" and ost["has_hdr"] == 0
        np.testing.assert_array_equal(out.numpy(), ho.srgb_to_linear(_t(g["final_result"])).numpy())


@pytest.mark.parametrize("case", [c for c in CASES if c.startswith(("a_", "b_"))])
@pytest.mark.parametrize("mode", MODES)
def test_node_output_matches_reference(golden_dir, case, mode):
    g = _load(golden_dir, case)
    for key in [k for k in g if k.startswith(f"node.{mode}.x")]:
        mult = float(key.split(".x", 1)[1])
        out, st = ho.hdr_epilogue(_t(g["pre_conv_out"]), _t(g["conv_w"]), _t(g["conv_b"]), mode, mult)
        assert st["accepted"] == 1
        assert out.dtype == torch.float32 and out.is_contiguous() and out.shape[-1] == 3
        ref = g[key]
        # conv_out is recomputed here (thread-count dependent summation order) and logit amplifies
        # 1-ulp differences near saturation, hence rel-L2 / max-abs-over-max-ref, not per-element.
        err = np.linalg.norm(out.numpy() - ref) / np.linalg.norm(ref)
        assert err < 1e-6, err
        assert np.abs(out.numpy() - ref).max() / np.abs(ref).max() < 1e-5


@pytest.mark.parametrize("case", ["a_b1_4x4", "b_b2_4x6"])
def test_decoder_restatement_reproduces_golden_activations(golden_dir, case):
    """Seeded weights + seeded latent -> the hooked pre_conv_out the reference captured."""
    g = _load(golden_dir, case)
    dec = apply_variant(build_decoder(0), str(g["variant"]))
    assert weight_fingerprint(dec) == pytest.approx(float(g["weight_fingerprint"]), rel=1e-12)
    with torch.no_grad():
        pre = dec.features(_t(g["latent"]))
    ref = g["pre_conv_out"]
    assert np.linalg.norm(pre.numpy() - ref) / np.linalg.norm(ref) < 1e-5


def test_decoder_matches_independent_implementation(golden_dir):
    """Cross-check the restated decoder against an independent implementation of the BFL Flux.1 AE decoder
    (torchtitan.experiments.flux.model.autoencoder.Decoder) with the same weights: against its output stored in
    tests/golden/bfl_decoder_seed3.npy (torchtitan 0.1.0, torch 2.11, CPU), and live where torchtitan is installed."""
    mine = build_decoder(0)
    z = torch.randn(1, 16, 4, 4, generator=torch.Generator().manual_seed(3))
    with torch.no_grad():
        a = mine(z)
    stored = _t(np.load(os.path.join(golden_dir, "bfl_decoder_seed3.npy")))
    assert (a - stored).norm() / stored.norm() < 1e-5
    assert sum(p.numel() for p in mine.parameters()) == 49_545_475   # SURVEY.md §8 a3
    try:
        from torchtitan.experiments.flux.model import autoencoder as ae
    except ImportError:
        return
    other = ae.Decoder(ch=128, out_ch=3, ch_mult=[1, 2, 4, 4], num_res_blocks=2, in_channels=3,
                       resolution=256, z_channels=16).eval()
    missing, unexpected = other.load_state_dict(mine.state_dict(), strict=True)
    assert not missing and not unexpected
    with torch.no_grad():
        b = other(z)
    assert (a - b).norm() / b.norm() < 1e-5


def test_maxpool_and_argmax_are_exact():
    g = torch.Generator().manual_seed(0)
    x = torch.randn(2, 128, 5, 7, generator=g)
    x[0, 126:, :, :] = 100.0          # channels 126/127 must be ignored
    x[1, 3, 0, 0] = x[1, 40, 0, 0] = 50.0   # tie -> first index
    p3 = ho.channel_maxpool3(x)
    am = ho.channel_argmax3(x)
    assert p3.shape == (2, 5, 7, 3) and p3.max() < 100.0
    assert am[1, 0, 0, 0] == 3
    gathered = torch.gather(x.movedim(1, -1), -1, am.long())
    assert torch.equal(gathered, p3)


def test_mode_aliases():
    assert ho.resolve_mode("moderate") == ("conservative", 3.0)
    assert ho.resolve_mode("Aggressive") == ("mathematical_recovery", 1.0)
    assert ho.resolve_mode("exposure") == ("exposure", 1.0)
    with pytest.raises(ValueError):
        ho.resolve_mode("bogus")


@pytest.mark.skipif(not reference_available(), reason="reference tree not mounted (GPU box)")
def test_live_reference_agrees_with_oracle_fresh_seed():
    """Where /root/reference is mounted: run the unmodified node live on a fresh seed."""
    dec = build_decoder(0)
    vae = FakeComfyVAE(dec)
    z = torch.randn(1, 16, 3, 5, generator=torch.Generator().manual_seed(99))
    node = load_reference_node()
    (ref,) = node.simple_hdr_decode({"samples": z}, vae, hdr_mode="exposure", conservative_ev_multiplier=1.5)
    out, st, _ = ho.simple_hdr_decode(dec, z, "exposure", 1.5)
    assert st["accepted"] == 1
    assert (out - ref).norm() / ref.norm() < 1e-6


def test_banded_oracle_equals_plain_oracle():
    """oracle/big_oracle.py (what the 4096^2 GPU parity test compares against) == FluxDecoder.features + the HDR math
    at a size both run, with band / chunk sizes that do not divide the image."""
    import torch
    from oracle import big_oracle as bo
    from oracle import hdr_oracle as ho
    from oracle.flux_decoder import build_decoder, make_latent
    dec = build_decoder(0)
    z = make_latent(1, 6, 5, seed=3)
    with torch.no_grad():
        a = dec.features(z)
    b = bo.features_banded(dec, z, band=7, q_chunk=11)
    assert float((a - b).norm() / a.norm()) < 1e-5
    o1, s1, _ = ho.simple_hdr_decode(dec, z, "aggressive")
    o2, s2, _ = bo.simple_hdr_decode_banded(dec, z, "aggressive", band=7, q_chunk=11)
    assert float((o1 - o2).norm() / o1.norm()) < 1e-4
    assert s1["norm_function"] == s2["norm_function"] and s1["has_hdr"] == s2["has_hdr"]
