"""SD1.x / SDXL VAEs on the B200: 4-channel latents and post_quant_conv (fused into the latent staging kernels) through
every decode path — features, full decode, node, CUDA-graph staging, batch sharding, row tiling (emulated and on 2 GPUs)
and the three precisions — against the fp32 oracle's SD first stage (seeded weights, fp16 operands unless stated)."""
import os
import sys

import pytest
import torch
import torch.multiprocessing as mp

from oracle import hdr_oracle as ho
from oracle.flux_decoder import FakeComfyVAE, Res, build_decoder, make_latent

from _metrics import rel_l2, rel_l2_outside, saturation_band_mask
from _sd_oracle import FakeComfySDVAE, build_sd_decoder, make_sd_latent

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LOGIT_MODES = ("exposure", "adaptive_recovery", "mathematical_recovery", "aggressive")


def _engine_weights(m):
    from vae_decode_hdr_b200.hdr_vae_decode import _engine_state_dict
    return _engine_state_dict(m.decoder, m.post_quant_conv)


@pytest.fixture(scope="module")
def setup():
    from vae_decode_hdr_b200.engine import HdrVaeEngine
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    m = build_sd_decoder(0).to(DEV)
    eng = HdrVaeEngine(_engine_weights(m), DEV)
    yield m, eng
    eng.close()


def _sd_latent(B, h, w, seed):
    return make_sd_latent(B, h, w, seed=seed).to(DEV)


def _band(m, pre, mode, shape):
    """The logit-recovery modes are compared outside the rule-based saturation band (tests/_metrics.py), as the Flux
    row-tiling tests do; conservative / moderate in full."""
    if mode not in LOGIT_MODES:
        return torch.zeros(shape[:3], dtype=torch.bool, device=DEV)
    band = saturation_band_mask(m, pre)
    assert float(band.float().mean()) < 1e-2
    return band


def test_engine_reports_four_latent_channels(setup):
    _, eng = setup
    assert eng.latent_channels == 4


@pytest.mark.parametrize("B,h,w", [(1, 8, 8), (2, 4, 6), (1, 5, 9), (1, 32, 32)])
def test_sd_features_vs_oracle(setup, B, h, w):
    m, eng = setup
    z = _sd_latent(B, h, w, 200 + h * w)
    with torch.no_grad():
        ref = m.features(z).permute(0, 2, 3, 1)
    got = eng.decode_features(z).float()
    assert got.shape == ref.shape and torch.isfinite(got).all()
    assert rel_l2(got, ref) < 3e-3, rel_l2(got, ref)


@pytest.mark.parametrize("mode", list(ho.HDR_MODES) + ["moderate"])
def test_sd_full_decode_vs_oracle(setup, mode):
    m, eng = setup
    z = _sd_latent(2, 16, 16, 77)
    out, st = eng.decode(z, mode, 1.0)
    ref, rst, pre = ho.simple_hdr_decode(m, z, mode, 1.0)
    assert out.shape == (2, 128, 128, 3) and out.dtype == torch.float32 and out.is_contiguous()
    assert st["accepted"] == rst["accepted"]
    assert st["norm_function"] == rst["norm_function"] and st["has_hdr"] == rst["has_hdr"]
    band = _band(m, pre, mode, out.shape)
    assert rel_l2_outside(out, ref, band) < 1e-2, rel_l2_outside(out, ref, band)
    assert st["pre_max"] == pytest.approx(rst["pre_max"], rel=5e-3)


def test_fused_post_quant_conv_is_exact(setup):
    """With W a permutation x powers of two, a dyadic bias and a latent on a coarse dyadic grid, W z + b is exact in fp32:
    the SD engine on z must then equal, bit for bit, an engine with the same decoder and no post_quant_conv on W z + b."""
    from vae_decode_hdr_b200.engine import HdrVaeEngine
    m, _ = setup
    perm, k = [2, 0, 3, 1], [1, -1, 0, 2]
    Wm = torch.zeros(4, 4)
    for c in range(4):
        Wm[c, perm[c]] = 2.0 ** k[c]
    b = torch.tensor([0.25, -0.5, 0.125, 1.0])
    sd = _engine_weights(m)
    sd["post_quant_conv.weight"] = Wm.view(4, 4, 1, 1).to(DEV)
    sd["post_quant_conv.bias"] = b.to(DEV)
    g = torch.Generator().manual_seed(5)
    z = (torch.randn(2, 4, 6, 10, generator=g) * 8).round().clamp(-32, 32) / 8
    y = torch.einsum("oc,bchw->bohw", Wm, z) + b.view(1, 4, 1, 1)
    assert torch.equal(y, torch.nn.functional.conv2d(z, Wm.view(4, 4, 1, 1), b))     # exact: the order does not matter
    with_pq = HdrVaeEngine(sd, DEV)
    plain = HdrVaeEngine(dict(m.decoder.state_dict()), DEV)
    try:
        assert with_pq.latent_channels == 4 and plain.latent_channels == 4
        a = with_pq.decode_features(z.to(DEV))
        c = plain.decode_features(y.to(DEV))
        assert torch.equal(a, c)
        assert not torch.equal(a, plain.decode_features(z.to(DEV)))
    finally:
        with_pq.close()
        plain.close()


def test_sd_node_end_to_end_and_repack():
    from vae_decode_hdr_b200 import NODE_CLASS_MAPPINGS
    node_cls = NODE_CLASS_MAPPINGS["HDRVAEDecode"]
    m = build_sd_decoder(3).to(DEV)
    vae = FakeComfySDVAE(m)
    z_cpu = make_sd_latent(1, 8, 8, seed=9)                 # ComfyUI hands CPU latents
    node = node_cls()
    (img,) = node.simple_hdr_decode({"samples": z_cpu}, vae, hdr_mode="conservative")
    assert img.dtype == torch.float32 and img.shape == (1, 64, 64, 3) and img.is_contiguous()
    assert img.device == torch.device(vae.output_device)
    ref, _, _ = ho.simple_hdr_decode(m, z_cpu.to(DEV), "conservative", 1.0)
    assert rel_l2(img, ref.to(img.device)) < 1e-2, rel_l2(img, ref.to(img.device))
    engines_before = set(map(id, node_cls._engines.values()))
    with torch.no_grad():
        m.post_quant_conv.weight.mul_(-0.5)                          # in place: the node must repack
    (img2,) = node.simple_hdr_decode({"samples": z_cpu}, vae, hdr_mode="conservative")
    assert set(map(id, node_cls._engines.values())) - engines_before, "no new engine after an in-place weight change"
    ref2, _, _ = ho.simple_hdr_decode(m, z_cpu.to(DEV), "conservative", 1.0)
    assert rel_l2(img2, ref2.to(img2.device)) < 1e-2, rel_l2(img2, ref2.to(img2.device))
    assert rel_l2(img2, img) > 1e-2
    node_cls.release_memory(keep_weights=False)


def test_latent_channel_count_is_checked(setup):
    from vae_decode_hdr_b200 import NODE_CLASS_MAPPINGS
    from vae_decode_hdr_b200.engine import HdrVaeEngine
    from vae_decode_hdr_b200.sharding import decode_batch_sharded
    _, sd_eng = setup
    dec = build_decoder(0).to(DEV)
    flux = HdrVaeEngine(dec.state_dict(), DEV)
    try:
        assert flux.latent_channels == 16
        with pytest.raises(ValueError, match=r"\[B,16,h,w\]"):
            flux.decode(_sd_latent(1, 4, 4, 1))
        with pytest.raises(ValueError, match=r"\[B,4,h,w\]"):
            sd_eng.decode(make_latent(1, 4, 4, seed=1).to(DEV))
        with pytest.raises(ValueError, match=r"\[B,4,h,w\]"):
            sd_eng.decode_features(make_latent(1, 4, 4, seed=1).to(DEV))
        with pytest.raises(ValueError, match=r"\[B,4,h,w\]"):
            decode_batch_sharded(sd_eng, make_latent(2, 4, 4, seed=1).to(DEV), "exposure")
        with pytest.raises(ValueError, match=r"\[B,4,h,w\]"):
            decode_batch_sharded(sd_eng, make_latent(0, 4, 4, seed=1).to(DEV), "exposure")
        with pytest.raises(ValueError, match=r"\[B,16,h,w\]"):
            decode_batch_sharded(flux, _sd_latent(1, 4, 4, 1), "exposure")
    finally:
        flux.close()
    node_cls = NODE_CLASS_MAPPINGS["HDRVAEDecode"]
    with pytest.raises(ValueError, match=r"\[B,16,h,w\]"):
        node_cls().simple_hdr_decode({"samples": make_sd_latent(1, 4, 4, seed=2)}, FakeComfyVAE(dec))
    node_cls.release_memory(keep_weights=False)


def test_cuda_graph_staging_copies_the_four_channel_latent(setup):
    """First decode of a shape runs plain, the second is captured into CUDA graphs, the third replays them: the replay
    of z1 must equal its plain decode exactly (the graph input copy is C_lat channels wide)."""
    _, eng = setup
    z1, z2 = _sd_latent(1, 6, 10, 61), _sd_latent(1, 6, 10, 62)
    a, _ = eng.decode(z1, "exposure")
    a = a.clone()
    b, _ = eng.decode(z2, "exposure")
    b = b.clone()
    c, _ = eng.decode(z1, "exposure")
    assert torch.equal(a, c)
    assert not torch.equal(a, b)


def test_sd_batch_sharded_decode_equals_whole_batch(setup):
    from vae_decode_hdr_b200.sharding import merge_raw_stats, shard_bounds
    _, eng = setup
    z = _sd_latent(4, 8, 8, 31)
    whole, _ = eng.decode(z, "adaptive_recovery")
    blocks, outs = [], []
    bounds = shard_bounds(4, 2)
    for s, e in bounds:
        vmin, vmax, vsum = eng.decode_begin(z[s:e])
        blocks.append((vmin.clone(), vmax.clone(), vsum.clone()))
    mmin, mmax, msum = merge_raw_stats(blocks)
    for s, e in bounds:
        vmin, vmax, vsum = eng.decode_begin(z[s:e])
        vmin.copy_(mmin); vmax.copy_(mmax); vsum.copy_(msum)
        o, _ = eng.decode_finish("adaptive_recovery")
        outs.append(o)
    assert torch.allclose(torch.cat(outs), whole, rtol=1e-6, atol=1e-7)


@pytest.mark.parametrize("world,h,w,mode", [(2, 32, 8, "moderate"), (2, 6, 5, "adaptive_recovery"), (3, 12, 16, "aggressive"),
                                            (4, 8, 12, "exposure"), (4, 16, 16, "conservative")])
def test_sd_row_tiled_decode(setup, world, h, w, mode):
    """Row tiling with `world` virtual ranks: the first latent row of a slab below the top sees post_quant_conv's output
    in its halo row, the outer halo rows of the border ranks stay zero (conv_in's padding)."""
    from vae_decode_hdr_b200.sharding import decode_rows_emulated
    m, eng = setup
    z = _sd_latent(1, h, w, 41 + world)
    tiled, _ = decode_rows_emulated(eng, z, world, mode)
    whole, _ = eng.decode(z, mode)
    assert tiled.shape == whole.shape
    if (world, h, w) == (2, 32, 8):          # the slabs tile like the whole image: identical
        assert rel_l2(tiled, whole) < 1e-6, rel_l2(tiled, whole)
        return
    ref, _, pre = ho.simple_hdr_decode(m, z, mode, 1.0)
    band = _band(m, pre, mode, tiled.shape)
    assert rel_l2_outside(tiled, ref, band) < 1e-2, rel_l2_outside(tiled, ref, band)


def test_sd_high_precision_and_bf16(setup):
    from vae_decode_hdr_b200.engine import HdrVaeEngine
    m, _ = setup
    z = _sd_latent(1, 8, 12, 45)
    with torch.no_grad():
        ref_feat = m.features(z).permute(0, 2, 3, 1)
    high = HdrVaeEngine(_engine_weights(m), DEV, precision="high")
    try:
        assert high.latent_channels == 4
        out, _ = high.decode(z, "conservative", 1.0)
        ref, _, _ = ho.simple_hdr_decode(m, z, "conservative", 1.0)
        assert rel_l2(out, ref) < 1e-3, rel_l2(out, ref)
        assert rel_l2(high.decode_features(z), ref_feat) < 2e-4
    finally:
        high.close()
    bf = HdrVaeEngine(_engine_weights(m), DEV, precision="bf16")
    try:
        got = bf.decode_features(z)
        assert got.dtype == torch.bfloat16
        assert rel_l2(got.float(), ref_feat) < 2e-2, rel_l2(got.float(), ref_feat)
    finally:
        bf.close()


HEADROOM_SCALE = 6.0e4      # tuned on the CPU oracle: residual stream max |x| = 2.6e5 for this seed and latent


def test_sd_headroom_of_the_fp16_residual_stream():
    """The default mode stores the residual stream and h as fp16 x 2^-4 (|x| < 1.05e6).  SDXL's VAE is reported to
    overflow plain fp16 inside its decoder; with the up.2 / up.1 conv2 weights and biases scaled so the oracle's residual
    stream reaches a max |x| in [1e5, 5e5], the features must stay finite and within the usual 3e-3."""
    from vae_decode_hdr_b200.engine import HdrVaeEngine
    m = build_sd_decoder(0)
    with torch.no_grad():
        for lvl in (2, 1):
            for blk in m.decoder.up[lvl].block:
                blk.conv2.weight.mul_(HEADROOM_SCALE)
                blk.conv2.bias.mul_(HEADROOM_SCALE)
    m = m.to(DEV)
    z = _sd_latent(1, 8, 8, 7)
    peaks = []
    hooks = [mod.register_forward_hook(lambda mod, i, o: peaks.append(float(o.abs().max())))
             for mod in m.modules() if isinstance(mod, Res)]
    try:
        with torch.no_grad():
            ref = m.features(z).permute(0, 2, 3, 1)
    finally:
        for h in hooks:
            h.remove()
    assert 1e5 <= max(peaks) <= 5e5, max(peaks)
    eng = HdrVaeEngine(_engine_weights(m), DEV)
    try:
        got = eng.decode_features(z).float()
    finally:
        eng.close()
    assert torch.isfinite(got).all()
    assert rel_l2(got, ref) < 3e-3, rel_l2(got, ref)


# ------------------------------------------------------------------------------------------------------------ 2 GPUs
def _two_gpu_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    sys.path.insert(0, ROOT)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    from vae_decode_hdr_b200.engine import HdrVaeEngine
    from vae_decode_hdr_b200.hdr_vae_decode import _engine_state_dict
    from vae_decode_hdr_b200.sharding import RowsDirect, decode_batch_sharded, decode_rows_sharded, shard_bounds
    m = build_sd_decoder(0)
    eng = HdrVaeEngine(_engine_state_dict(m.decoder, m.post_quant_conv), dev)
    res = {}
    z = make_sd_latent(4, 8, 8, seed=5).to(dev)
    s, e = shard_bounds(4, world)[rank]
    out, _ = decode_batch_sharded(eng, z[s:e], "adaptive_recovery", 1.0)
    whole, _ = eng.decode(z, "adaptive_recovery", 1.0)
    res["batch"] = bool(torch.allclose(out, whole[s:e], rtol=1e-6, atol=1e-7))
    # 32 x 8 latent on 2 ranks: the slabs tile like the whole image, so both transports must equal the single-GPU decode
    zr = make_sd_latent(1, 32, 8, seed=9).to(dev)
    whole, _ = eng.decode(zr, "moderate", 1.0)
    rows = 8 * 32 // world
    mine = whole[:, rank * rows:(rank + 1) * rows]
    out, _ = decode_rows_sharded(eng, zr, "moderate", 1.0)
    res["rows_nccl"] = float((out - mine).double().norm() / mine.double().norm())
    p2p = RowsDirect(eng, 32, 8)
    out2, _ = p2p.decode(zr, "moderate", 1.0)
    p2p.close()
    res["rows_direct"] = float((out2 - mine).double().norm() / mine.double().norm())
    q.put((rank, res))
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_sd_decode_on_two_gpus():
    """Batch sharding over NCCL, and row tiling over NCCL and over the device-driven transport (RowsDirect), each equal
    to the single-GPU SD decode."""
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 31600 + os.getpid() % 1000
    procs = [ctx.Process(target=_two_gpu_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=200) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    for rank, r in res:
        assert r["batch"] and r["rows_nccl"] < 1e-6 and r["rows_direct"] < 1e-6, res
