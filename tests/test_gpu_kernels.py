"""Kernel-level parity on the B200, through the C ABI (vae_decode_hdr_b200.engine -> libhdrvae.so).
Each CUDA kernel against a plain PyTorch fp32 evaluation of the same op on the same (rounded) operands;
the tolerance and where it comes from is written at each check."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
OPS = {"fp16": torch.float16, "bf16": torch.bfloat16, "tf32": torch.float32}
# relative rounding step of one operand element: fp16/tf32 2^-11, bf16 2^-8 (half an ulp)
W_ROUND = {"fp16": 2.0 ** -11, "bf16": 2.0 ** -8, "tf32": 2.0 ** -11}


@pytest.fixture(scope="module")
def engine():
    from oracle.flux_decoder import build_decoder
    from vae_decode_hdr_b200.engine import HdrVaeEngine
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    eng = HdrVaeEngine(build_decoder(0).state_dict(), DEV)
    yield eng
    eng.close()


def _rel(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def _round_tf32(x):
    i = x.contiguous().view(torch.int32)
    return ((i + 0x1000) & ~0x1FFF).view(torch.float32)


def _as_operand(x, op):
    """Values exactly representable in the operand type, as float32."""
    if op == "tf32":
        return _round_tf32(x)
    return x.to(OPS[op]).float()


def _conv_ref(x_nhwc, w, b, ksize, upsample, residual):
    x = x_nhwc.float().permute(0, 3, 1, 2)
    if upsample:
        x = F.interpolate(x, scale_factor=2.0, mode="nearest")
    y = F.conv2d(x, w, b, padding=ksize // 2).permute(0, 2, 3, 1)
    if residual is not None:
        y = y + residual.float()
    return y


CONV_CASES = [
    # B, H, W, Cin, Cout, ksize, upsample, residual
    (1, 8, 16, 64, 128, 3, False, False),     # exactly one 128-pixel tile, one k-block per tap
    (1, 16, 16, 128, 128, 3, False, True),
    (2, 12, 20, 128, 256, 3, False, True),    # ragged tiles (masked rows), BLOCK_N = 256
    (1, 32, 32, 512, 512, 3, False, True),    # two n-tiles, K = 4608
    (1, 16, 16, 256, 128, 1, False, False),   # nin_shortcut shape
    (1, 8, 8, 256, 256, 3, True, False),      # upsample folded into the load
    (2, 5, 7, 128, 128, 3, True, False),      # odd sizes + upsample
    (1, 3, 5, 64, 32, 3, False, False),       # smaller than one tile, narrow N
    (3, 64, 64, 128, 128, 3, False, False),   # many tiles -> several per CTA (pipeline phase wrap)
]


@pytest.mark.parametrize("cta_group", [2, 1], ids=["pair", "single"])
@pytest.mark.parametrize("op", list(OPS))
@pytest.mark.parametrize("case", CONV_CASES, ids=[str(c) for c in CONV_CASES])
def test_conv_tcgen05_matches_torch_and_direct(engine, case, op, cta_group):
    from vae_decode_hdr_b200 import _native as N
    B, H, W, cin, cout, ks, up, res = case
    engine.set_cta_group(cta_group)        # tcgen05 cta_group::2 (CTA pairs, the default) and ::1
    g = torch.Generator(device="cpu").manual_seed(abs(hash(case)) % (2 ** 31))
    x = _as_operand(torch.randn(B, H, W, cin, generator=g), op).to(DEV)
    w = (torch.randn(cout, cin, ks, ks, generator=g) / math.sqrt(cin * ks * ks)).to(DEV)
    b = torch.randn(cout, generator=g).to(DEV)
    OH, OW = (2 * H, 2 * W) if up else (H, W)
    r = torch.randn(B, OH, OW, cout, generator=g).to(DEV) if res else None     # fp32 residual stream
    xo = x.to(OPS[op])
    stats_ok = cout in (128, 256, 512)
    got = engine.conv2d(xo, w, b, ks, up, r, out_dtype=torch.float32, want_stats=stats_ok, impl=N.CONV_TCGEN05)
    y_tc, part = got if stats_ok else (got, None)
    y_dr = engine.conv2d(xo, w, b, ks, up, r, out_dtype=torch.float32, impl=N.CONV_DIRECT)
    torch.cuda.synchronize()
    assert torch.isfinite(y_tc).all()
    # same rounded operands, fp32 accumulation in a different order: 1e-5 relative
    assert _rel(y_tc, y_dr) < 1e-5, ("tcgen05 vs direct", _rel(y_tc, y_dr))
    # torch fp32 conv with UNROUNDED weights: only the operand rounding of the weights differs
    # (relative step W_ROUND per weight, averaged over the K terms; upsample phase weights are pre-summed)
    ref = _conv_ref(x, w, b, ks, up, r)
    assert _rel(y_tc, ref) < 1.1 * W_ROUND[op], ("tcgen05 vs torch", _rel(y_tc, ref))
    # 16-bit output paths
    for od in (torch.float16, torch.bfloat16):
        y16 = engine.conv2d(xo, w, b, ks, up, r, out_dtype=od)
        assert _rel(y16.float(), y_tc) < (2.0 ** -10 if od == torch.float16 else 2.0 ** -7)
    if stats_ok:
        # GroupNorm partials emitted by the conv epilogue == (sum, sum of squares) per group of the fp32 output
        cpg = cout // 32
        yg = y_tc.double().reshape(B, OH * OW, 32, cpg)
        want = torch.stack([yg.sum((1, 3)), (yg * yg).sum((1, 3))], dim=-1)       # [B,32,2]
        assert torch.allclose(part.double().sum(1), want, rtol=2e-5, atol=1e-3), float((part.double().sum(1) - want).abs().max())
    engine.set_cta_group(0)


def test_conv_exact_operands_agree_with_torch_to_fp32_noise(engine):
    """With weights exactly representable in the operand type the kernel must agree with torch to fp32 noise."""
    g = torch.Generator().manual_seed(5)
    for op in OPS:
        x = _as_operand(torch.randn(1, 16, 24, 128, generator=g), op).to(DEV)
        w = _as_operand(torch.randn(256, 128, 3, 3, generator=g) / 34.0, op).to(DEV)
        b = torch.randn(256, generator=g).to(DEV)
        y = engine.conv2d(x.to(OPS[op]), w, b, 3)
        assert _rel(y, _conv_ref(x, w, b, 3, False, None)) < 2e-6, op


def test_tf32_conv_on_unrounded_stream_and_round_flag(engine):
    """kind::tf32 reads the top 19 bits of each fp32: feeding an un-rounded stream costs < 2^-10 relative;
    round_tf32 rounds the fp32 output (RN) so the next tf32 conv reads it exactly."""
    g = torch.Generator().manual_seed(6)
    x = torch.randn(1, 16, 16, 256, generator=g).to(DEV)
    w = (torch.randn(128, 256, 1, 1, generator=g) / 16.0).to(DEV)
    y = engine.conv2d(x, w, None, 1)
    ref = _conv_ref(x, w, None, 1, False, None)
    assert _rel(y, ref) < 2.0 ** -10
    yr = engine.conv2d(x, w, None, 1, round_tf32=True)
    assert torch.equal(yr, _round_tf32(yr)) and _rel(yr, y) < 2.0 ** -11


GN_CASES = [((2, 16, 16, 512), True), ((1, 9, 13, 256), True), ((3, 32, 32, 128), True), ((1, 64, 64, 512), False),
            ((1, 1, 1, 128), True)]


@pytest.mark.parametrize("in_dt", [torch.float32, torch.float16, torch.bfloat16])
@pytest.mark.parametrize("out_dt", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("shape,silu", GN_CASES)
def test_groupnorm_silu(engine, shape, silu, in_dt, out_dt):
    g = torch.Generator().manual_seed(11)
    B, H, W, Cc = shape
    x = (torch.randn(shape, generator=g) * 2.0 + 0.7).to(in_dt).to(DEV)
    gamma = (1.0 + 0.1 * torch.randn(Cc, generator=g)).to(DEV)
    beta = (0.1 * torch.randn(Cc, generator=g)).to(DEV)
    y = engine.groupnorm_silu(x, gamma, beta, silu, out_dtype=out_dt).float()
    ref = F.group_norm(x.float().permute(0, 3, 1, 2), 32, gamma, beta, eps=1e-6)
    if silu:
        ref = F.silu(ref)
    ref = ref.permute(0, 2, 3, 1)
    half_ulp = 2.0 ** -11 if out_dt == torch.float16 else 2.0 ** -8     # the output rounding
    assert torch.allclose(y, ref, rtol=2 * half_ulp, atol=2e-3 if out_dt == torch.bfloat16 else 3e-4), float((y - ref).abs().max())
    assert _rel(y, ref) < 1.5 * half_ulp


def test_groupnorm_from_conv_partials_equals_standalone(engine):
    """The decoder path: statistics emitted by the producing conv's epilogue instead of a second read."""
    g = torch.Generator().manual_seed(13)
    x = torch.randn(2, 20, 28, 128, generator=g).to(DEV).half()
    w = (torch.randn(256, 128, 3, 3, generator=g) / 34.0).to(DEV)
    b = torch.randn(256, generator=g).to(DEV)
    y, part = engine.conv2d(x, w, b, 3, want_stats=True)
    gamma = (1.0 + 0.1 * torch.randn(256, generator=g)).to(DEV)
    beta = (0.1 * torch.randn(256, generator=g)).to(DEV)
    a = engine.groupnorm_silu(y, gamma, beta, True, partials=part).float()
    s = engine.groupnorm_silu(y, gamma, beta, True).float()
    ref = F.silu(F.group_norm(y.permute(0, 3, 1, 2), 32, gamma, beta, eps=1e-6)).permute(0, 2, 3, 1)
    assert _rel(a, ref) < 2.0 ** -10 and _rel(a, s) < 2.0 ** -10
    assert float((a - s).abs().max()) < 2e-3


def test_groupnorm_is_run_to_run_deterministic(engine):
    g = torch.Generator().manual_seed(12)
    x = torch.randn(2, 40, 40, 256, generator=g).to(DEV)
    gamma = torch.ones(256, device=DEV)
    beta = torch.zeros(256, device=DEV)
    a = engine.groupnorm_silu(x, gamma, beta, True)
    b = engine.groupnorm_silu(x, gamma, beta, True)
    assert torch.equal(a, b)


@pytest.mark.parametrize("impl", ["tcgen05", "direct"])
@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("B,T", [(1, 64), (2, 256), (1, 24), (1, 1000), (1, 4096)])
def test_attention(engine, B, T, dt, impl):
    """The fused kernel (tensor-core build) and the GEMM-level form (CUDA-core validation build)."""
    from vae_decode_hdr_b200 import _native as N
    g = torch.Generator().manual_seed(T)
    q = torch.randn(B, T, 512, generator=g).to(dt).to(DEV)
    k = torch.randn(B, T, 512, generator=g).to(dt).to(DEV)
    v = torch.randn(B, T, 512, generator=g).to(dt).to(DEV)
    engine.set_conv_impl(N.CONV_DIRECT if impl == "direct" else N.CONV_TCGEN05)
    try:
        o = engine.attention(q, k, v).float()
    finally:
        engine.set_conv_impl(N.CONV_TCGEN05)
    p = torch.softmax(q.float() @ k.float().transpose(1, 2) / math.sqrt(512.0), dim=-1)
    ref = p @ v.float()
    # exp(s - max) is rounded to the operand type before PV, the output once more: ~half an ulp each
    assert _rel(o, ref) < (1.2e-3 if dt == torch.float16 else 6e-3), _rel(o, ref)


@pytest.mark.parametrize("cta_group", [2, 1])
@pytest.mark.parametrize("T,scale", [(1000, 4.0), (2048, 6.0), (384, 1.0)])
def test_attention_fused_lazy_rescale_paths(engine, T, scale, cta_group):
    """The fused attention kernel (attention.cu) on inputs that exercise its online soft-max: peaked score distributions
    (q scaled: scores ~ N(0, scale^2)) and keys ORDERED by growing norm, so that the running row maximum keeps rising
    from key block to key block and crosses the lazy-rescale threshold (2^8) several times; T = 1000 also masks the tail
    of the last key block.  CTA-pair (cta_group::2, the product path) and single-CTA builds against fp64."""
    g = torch.Generator().manual_seed(T + int(scale))
    q = (torch.randn(1, T, 512, generator=g) * scale).half().to(DEV)
    k = torch.randn(1, T, 512, generator=g)
    k = (k * torch.linspace(0.2, 2.0, T)[None, :, None]).half().to(DEV)        # later keys score higher on average
    v = torch.randn(1, T, 512, generator=g).half().to(DEV)
    engine.set_cta_group(cta_group)
    try:
        o = engine.attention(q, k, v).double()
    finally:
        engine.set_cta_group(0)
    p = torch.softmax(q.double() @ k.double().transpose(1, 2) / math.sqrt(512.0), dim=-1)
    ref = p @ v.double()
    assert bool(torch.isfinite(o).all())
    assert _rel(o, ref) < 1.5e-3, _rel(o, ref)
    row = ((o - ref).norm(dim=-1) / ref.norm(dim=-1)).max()
    assert float(row) < 8e-3, float(row)


def test_pack_half_bit_exact_vs_numpy():
    from vae_decode_hdr_b200.engine import pack_half
    g = torch.Generator().manual_seed(3)
    img = torch.randn(2, 7, 9, 3, generator=g) * 100.0
    img[0, 0, 0, 0] = 70000.0       # overflow -> inf (linear_exr_export.py:155 numpy astype semantics)
    img[0, 0, 0, 1] = -1e-8         # underflow -> -0
    img[0, 0, 0, 2] = 6.0e-6        # fp16 subnormal
    img[0, 0, 1, 0] = 1.00048828125  # exact tie -> round to even
    with np.errstate(over="ignore"):
        want = img.numpy().astype(np.float16)
    got = pack_half(img.to(DEV)).cpu().numpy()
    assert np.array_equal(got.view(np.uint16), want.view(np.uint16))
    planes = pack_half(img.to(DEV), exr_scanline_order=True).cpu().numpy()     # [B,H,3(B,G,R),W]
    assert np.array_equal(planes.view(np.uint16), np.ascontiguousarray(want[..., ::-1].transpose(0, 1, 3, 2)).view(np.uint16))
    assert pack_half(torch.empty(0, 4, 4, 3, device=DEV)).shape == (0, 4, 4, 3)


@pytest.mark.parametrize("n", [1, 7, 1000, 3 * 512 * 512 + 5])
def test_quantiles_radix_select_bit_exact(n):
    """Radix-select quantile indices must be bit-exact (BASELINE.json north_star): == torch.kthvalue."""
    from vae_decode_hdr_b200.engine import quantiles
    g = torch.Generator().manual_seed(n)
    x = (torch.randn(n, generator=g) * 3.0).to(DEV)
    if n > 10:
        x[3] = float("inf"); x[5] = -0.0; x[6] = 0.0; x[7] = -1e-30; x[8:60] = 1.25      # ties, signed zeros, inf
    qs = [0.0, 0.01, 0.5, 0.99, 0.999, 1.0]
    got = quantiles(x, qs)
    for q, v in zip(qs, got):
        k = int(math.floor(q * (n - 1))) + 1
        want = float(torch.kthvalue(x.float().cpu(), k).values)
        assert np.float32(v).tobytes() == np.float32(want).tobytes() or (v == want == 0.0), (q, v, want)
