"""Every tensor-core conv build the upscalers launch, one launch at a time against a plain fp64 evaluation of that launch.

The rows below restate the call sites of csrc/upscaler.cu (up_forward_rrdb, up_forward_compact, up_forward_span) through
hdrvae_conv2d with the same ConvIO fields: channel slices of wider buffers on input and output, the second 16-bit output,
the residual pair with res_scale, and LeakyReLU / PReLU / SiLU / SPAN's gate.  Each row runs
  - on four shapes: whole 8 x 16 slab tiles (every tile takes the epilogue's fast path), a ragged slab shape with an odd
    m-tile count (masked tiles, and a CTA pair with a padding tile), a shape below 128 pixels (the non-slab form) and one
    with several tiles per CTA (the accumulator ring wraps);
  - on the CTA-pair builds, the single-CTA builds and the CUDA-core validation kernel, which is the comparator of every
    tcgen05-vs-CUDA-core network test.
The inputs make small defects visible: operands exactly representable in fp16 (the packing rounds nothing, so the fp64
reference differs from the kernel only by fp32 accumulation order and the output rounding), fp16 NaN in every input channel
the conv must not read, a sentinel bit pattern in every output channel it must not write (and past the end of each
buffer), and biases / residuals that give t both signs.  test_every_launched_build_has_a_row checks that the rows reach
every build the models launch."""
import math
import os
import re
import subprocess
import sys
import zlib

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

F16, F32 = torch.float16, torch.float32
LRELU = float(torch.tensor(0.2, dtype=F32))       # the kernels compute with fp32 0.2
RES_SCALE = LRELU
NAN16 = 0x7E5A                                     # fp16 quiet NaN with a payload: unread input, unwritten fp16 output
SENT32 = 0x7FC0DEAD                                # fp32 NaN with a payload: unwritten fp32 output
GUARD = 64                                         # sentinel elements after the end of every output buffer
# Relative error of the epilogue's sigmoid (common.cuh sigmoid_nr: ex2.approx, a bit-trick reciprocal and two Newton steps):
# the Newton steps leave up to 6.62e-6 = 2^-17.2 of 1 / (1 + e), evaluated over every fp32 mantissa of 1 + e with the
# kernel's fp32 / fma steps; ex2.approx adds ~2^-22.  (The CUDA-core kernel's 1 / (1 + expf(-v)) is far closer.)
SIG_REL = 2.0 ** -17


def row(name, build, cin, cout, *, ks=3, up=False, xc=None, xoff=0, alias=False, yc=None, yoff=0, ydt=F32, y2=None,
        res=False, res_scale=1.0, res2=False, act=None):
    """xc / xoff: x is [B,H,W,xc] and the conv reads channels [xoff, xoff + cin) (xc None: dense, Cin % 64 == 0);
    alias: x is the output buffer (the RRDB dense block); yc / yoff: y is [B,OH,OW,yc] written from yoff on (None: dense);
    y2: (y2c, y2off) of an fp16 second output, y2off None: y2 shares y's layout; act: lrelu / prelu / silu / gate."""
    return dict(name=name, build=build, cin=cin, cout=cout, ks=ks, up=up, xc=xc, xoff=xoff, alias=alias, yc=yc, yoff=yoff,
                ydt=ydt, y2=y2, res=res, res_scale=res_scale, res2=res2, act=act)


# Builds are named as launch_gemm_tc selects them (gemm_tc.cu): slab form (3x3, >= 128 pixels) / non-slab form, CTA pairs.
# With set_cta_group(1) every narrow conv takes launch_tc<32,false,1,EPI_GENERIC,9> / <32,false,1,EPI_GENERIC> (32 columns,
# slab / non-slab) or launch_tc<64,false,1,EPI_GENERIC> (64 columns, both forms).
ROWS = [
    # ---- RRDBNet (up_forward_rrdb): nf 64, gc 32
    *[row(f"rrdb.conv_first.f{f}", "launch_tc<64,false,2,EPI_OUT2,9> / <64,false,2,EPI_OUT2>",
          3 * f * f, 64, xc={1: 8, 2: 16, 4: 48}[f], yc=64, y2=(192, 0)) for f in (1, 2, 4)],
    *[row(f"rrdb.rdb.conv{j + 1}", "launch_tc<32,false,2,EPI_OUT16|EPI_LRELU,9> / <32,false,2,EPI_OUT16|EPI_LRELU>",
          64 + 32 * j, 32, xc=192, alias=True, yc=192, yoff=64 + 32 * j, ydt=F16, act="lrelu") for j in range(4)],
    row("rrdb.rdb.conv5", "launch_tc<64,false,2,EPI_RES|EPI_OUT2,9> / <64,false,2,EPI_RES|EPI_OUT2>",
        192, 64, xc=192, yc=64, y2=(192, 0), res=True),
    row("rrdb.rdb3.conv5", "launch_tc<64,false,2,EPI_RES|EPI_RES2|EPI_OUT2,9> / <64,false,2,EPI_RES|EPI_RES2|EPI_OUT2>",
        192, 64, xc=192, yc=64, y2=(192, 0), res=True, res_scale=RES_SCALE, res2=True),
    row("rrdb.conv_body", "launch_tc<64,false,2,EPI_RES|EPI_OUT2,9> / <64,false,2,EPI_RES|EPI_OUT2>",
        64, 64, xc=192, y2=(64, None), res=True),
    row("rrdb.conv_up1", "launch_tc<64,false,2,EPI_OUT16|EPI_LRELU> (upsample convs never take the slab form here)",
        64, 64, up=True, ydt=F16, act="lrelu"),
    row("rrdb.conv_hr", "launch_tc<64,false,2,EPI_OUT16|EPI_LRELU,9> / <64,false,2,EPI_OUT16|EPI_LRELU>",
        64, 64, ydt=F16, act="lrelu"),
    row("rrdb.conv_last", "launch_tc<32,false,2,0,9> / <32,false,2,0>: n_store 4 of 32 columns", 64, 3, yc=4),
    # ---- Real-ESRGAN Compact (up_forward_compact): activations at a pixel stride of cout_pad
    row("compact.body0.nf64", "launch_tc<64,false,2,EPI_OUT16|EPI_PRELU,9> / <64,false,2,EPI_GENERIC>",
        3, 64, xc=8, yc=64, ydt=F16, act="prelu"),
    row("compact.body.nf64", "launch_tc<64,false,2,EPI_OUT16|EPI_PRELU,9> / <64,false,2,EPI_GENERIC>",
        64, 64, xc=64, yc=64, ydt=F16, act="prelu"),
    row("compact.body0.nf16", "launch_tc<32,false,2,EPI_GENERIC,9> / <32,false,2,EPI_GENERIC>",
        3, 16, xc=8, yc=32, ydt=F16, act="prelu"),
    row("compact.body.nf16", "launch_tc<32,false,2,EPI_GENERIC,9> / <32,false,2,EPI_GENERIC>",
        16, 16, xc=32, yc=32, ydt=F16, act="prelu"),
    row("compact.last.s1", "launch_tc<32,false,2,0,9> / <32,false,2,0>", 64, 3, xc=64, yc=4),
    row("compact.last.s2", "launch_tc<32,false,2,0,9> / <32,false,2,0>", 64, 12, xc=64, yc=12),
    row("compact.last.s4.nf16", "launch_tc<64,false,2,EPI_GENERIC,9> / <64,false,2,EPI_GENERIC>", 16, 48, xc=32, yc=48),
]
for nf in (48, 16):
    # ---- SPAN (up_forward_span): cat = [f | b6 | b1 | b5_2] of 4 nf channels; nf 48 -> 64-column builds, nf 16 -> 32
    wide = nf > 32
    n = 64 if wide else 32
    gen = f"launch_tc<{n},false,2,EPI_GENERIC,9> / <{n},false,2,EPI_GENERIC>"
    ROWS += [
        row(f"span{nf}.conv_1", "launch_tc<64,false,2,EPI_OUT2,9> / <64,false,2,EPI_OUT2>" if wide else gen,
            3, nf, xc=8, yc=nf, y2=(4 * nf, 0)),
        row(f"span{nf}.block_1.c1_r", "launch_tc<64,false,2,EPI_OUT16|EPI_SILU,9> / <64,false,2,EPI_GENERIC>" if wide else gen,
            nf, nf, xc=4 * nf, yc=nf, ydt=F16, act="silu"),
        row(f"span{nf}.block_6.c1_r", "launch_tc<64,false,2,EPI_OUT16|EPI_SILU,9> / <64,false,2,EPI_GENERIC>" if wide else gen,
            nf, nf, xc=nf, yc=4 * nf, yoff=3 * nf, ydt=F16, act="silu"),
        row(f"span{nf}.block_6.c2_r", "launch_tc<64,false,2,EPI_OUT16|EPI_SILU,9> / <64,false,2,EPI_GENERIC>" if wide else gen,
            nf, nf, xc=4 * nf, xoff=3 * nf, yc=nf, ydt=F16, act="silu"),
        row(f"span{nf}.block_1.c3_r",
            "launch_tc<64,false,2,EPI_RES|EPI_GATE|EPI_OUT2,9> / <64,false,2,EPI_GENERIC>" if wide else gen,
            nf, nf, xc=nf, yc=nf, y2=(4 * nf, 2 * nf), res=True, act="gate"),
        row(f"span{nf}.block_2.c3_r",
            "launch_tc<64,false,2,EPI_RES|EPI_GATE|EPI_OUT2,9> / <64,false,2,EPI_GENERIC>" if wide else gen,
            nf, nf, xc=nf, yc=nf, y2=(nf, 0), res=True, act="gate"),
        row(f"span{nf}.conv_2", gen, nf, nf, xc=nf, yc=4 * nf, yoff=nf, ydt=F16),
        row(f"span{nf}.conv_cat", f"launch_tc<{n},false,2,EPI_GENERIC> (1x1: non-slab only)",
            4 * nf, nf, ks=1, xc=4 * nf, yc=nf, ydt=F16),
        row(f"span{nf}.upsampler.0.s4", "launch_tc<64,false,2,EPI_GENERIC,9> / <64,false,2,EPI_GENERIC>", nf, 48, xc=nf, yc=48),
    ]
ROWS.append(row("span16.upsampler.0.s1", "launch_tc<32,false,2,0,9> / <32,false,2,0>", 16, 3, xc=16, yc=4))

# (B, H, W): whole 8 x 16 slab tiles; ragged slab tiles, 3 x 3 = 9 m-tiles (odd: the last CTA pair has a padding tile);
# below 128 pixels (non-slab form, one masked tile); 384 slab tiles, at least 2 per CTA (the accumulator ring wraps)
SHAPES = {"whole": (2, 32, 16), "ragged": (3, 13, 19), "small": (1, 5, 7), "many": (3, 128, 128)}
KERNELS = ["pair", "single", "direct"]


def _seed(*key):
    return zlib.crc32(repr(key).encode())


def _sentinel(shape, dtype):
    """Device tensor [*shape] filled with the sentinel, followed by GUARD sentinel elements: -> (view, whole buffer)."""
    n = math.prod(shape)
    buf = torch.empty(n + GUARD, dtype=dtype, device=DEV)
    if dtype == F32:
        buf.view(torch.int32).fill_(SENT32)
    else:
        buf.view(torch.int16).fill_(NAN16)
    return buf[:n].view(shape), buf


def _n_store(cout):
    """Columns a conv stores: all of them when Cout % 32 == 0, else round_up(Cout, 4) (run_conv)."""
    return cout if cout % 32 == 0 else (cout + 3) // 4 * 4


def make_inputs(r, shape):
    """Operands of one launch (host generator, exact in fp16 where the kernel reads them as fp16)."""
    B, H, W = shape
    OH, OW = (2 * H, 2 * W) if r["up"] else (H, W)
    g = torch.Generator().manual_seed(_seed(r["name"], shape))
    cin, cout, ks = r["cin"], r["cout"], r["ks"]
    d = {}
    d["xs"] = torch.randn(B, H, W, cin, generator=g).to(F16)
    # weights on a 2^-8 grid, |w| < 2: exact in fp16, and so are the sums of up to 4 taps that the folded upsample packs
    # as its phase weights (pack_conv)
    d["w"] = torch.round(torch.randn(cout, cin, ks, ks, generator=g) / math.sqrt(cin * ks * ks) * 256) / 256
    d["b"] = torch.randn(cout, generator=g) * 0.5
    yc = r["yc"] or cout
    d["r"] = torch.randn(B, OH, OW, yc, generator=g) if r["res"] else None
    d["r2"] = torch.randn(B, OH, OW, yc, generator=g) if r["res2"] else None
    d["slope"] = (torch.rand(cout, generator=g) - 0.5).to(F16).float() if r["act"] == "prelu" else None
    return d


def launch(eng, r, shape, kernel, d):
    """One hdrvae_conv2d call as the upscaler makes it.  -> dict of the output buffers (views and whole buffers with the
    guard) and their contents before the call."""
    from vae_decode_hdr_b200 import _native as N
    B, H, W = shape
    OH, OW = (2 * H, 2 * W) if r["up"] else (H, W)
    cin, cout = r["cin"], r["cout"]
    yc = r["yc"] or cout
    y, ybuf = _sentinel((B, OH, OW, yc), r["ydt"])
    if r["alias"]:
        x = y
    else:
        x, _ = _sentinel((B, H, W, r["xc"] or cin), F16)
    x[..., r["xoff"]:r["xoff"] + cin] = d["xs"].to(DEV)
    y2 = y2buf = None
    if r["y2"] is not None:
        y2, y2buf = _sentinel((B, OH, OW, r["y2"][0]), F16)
    before = {"y": ybuf.clone(), "y2": y2buf.clone() if y2buf is not None else None}
    eng.set_cta_group(1 if kernel == "single" else 0)
    eng.conv2d(x, d["w"].to(DEV), d["b"].to(DEV), r["ks"], r["up"], d["r"].to(DEV) if r["res"] else None,
               impl=N.CONV_DIRECT if kernel == "direct" else N.CONV_TCGEN05,
               cin=cin if r["xc"] else None, x_chan_off=r["xoff"], out=y, out_chan_off=r["yoff"],
               out2=y2, out2_chan_off=r["y2"][1] if r["y2"] else None,
               residual2=d["r2"].to(DEV) if r["res2"] else None, res_scale=r["res_scale"],
               lrelu=LRELU if r["act"] == "lrelu" else 0.0, prelu=d["slope"].to(DEV) if r["act"] == "prelu" else None,
               act={"silu": N.ACT_SILU, "gate": N.ACT_GATE}.get(r["act"], N.ACT_NONE))
    eng.set_cta_group(0)
    return dict(y=y, ybuf=ybuf, y2=y2, y2buf=y2buf, before=before)


def reference(r, d):
    """fp64 evaluation of the launch over the n_store columns it writes (padding columns: zero weights and bias), and the
    elementwise bound on the kernel's fp32 result before the output rounding."""
    cout, ks = r["cout"], r["ks"]
    ns = _n_store(cout)
    x = d["xs"].to(DEV).double().permute(0, 3, 1, 2)
    if r["up"]:
        x = F.interpolate(x, scale_factor=2.0, mode="nearest")
    w = torch.zeros(ns, r["cin"], ks, ks, dtype=torch.float64, device=DEV)
    w[:cout] = d["w"].to(DEV).double()
    b = torch.zeros(ns, dtype=torch.float64, device=DEV)
    b[:cout] = d["b"].to(DEV).double()
    t = F.conv2d(x, w, b, padding=ks // 2).permute(0, 2, 3, 1)
    M = F.conv2d(x.abs(), w.abs(), b.abs(), padding=ks // 2).permute(0, 2, 3, 1)
    sl = slice(r["yoff"], r["yoff"] + ns)
    u = t.clone()
    if r["res"]:
        rr = r["res_scale"] * d["r"].to(DEV).double()[..., sl]
        u, M = u + rr, M + rr.abs()
    if r["res2"]:
        r2 = d["r2"].to(DEV).double()[..., sl]
        u, M = u + r2, M + r2.abs()
    # every fp16 x fp16 product is exact in fp32; what remains is the fp32 accumulation over K <= 9 * 192 = 1728 terms
    # (and the bias / residual adds): 2^-18 of the sum of magnitudes
    eps = 2.0 ** -18 * M
    act = r["act"]
    if act == "lrelu":
        y, bound = torch.where(u < 0, u * LRELU, u), eps
    elif act == "prelu":
        s = torch.zeros(ns, dtype=torch.float64, device=DEV)
        s[:cout] = d["slope"].to(DEV).double()
        y, bound = torch.where(u < 0, u * s, u), eps * s.abs().clamp_min(1.0)
    elif act == "silu":
        y = u * torch.sigmoid(u)
        bound = 1.1 * eps + SIG_REL * y.abs()               # |silu'| <= 1.1
    elif act == "gate":
        gt = torch.sigmoid(t) - 0.5                          # from t before the residual
        y = u * gt
        bound = (gt.abs() + u.abs() / 4) * eps + SIG_REL * u.abs()       # |sigmoid'| <= 1/4
    else:
        y, bound = u, eps
    return y, bound


def _half_ulp(v, dtype):
    """Half an ulp of the stored 16-bit value, plus the fp16 subnormal step."""
    return v.abs() * (2.0 ** -11 if dtype == F16 else 2.0 ** -8) + 2.0 ** -24


def _ratio(got, want, bound):
    err = (got.double() - want).abs()
    return float((err / bound.clamp_min(1e-300)).max())


def _bits(t):
    return t.view(torch.int32) if t.dtype == F32 else t.view(torch.int16)


def _untouched(out, before, chans, lo, hi):
    """Every element of the whole buffer (guard included) outside channels [lo, hi) of its [..., chans] view keeps its
    bits."""
    keep = torch.ones(out.numel(), dtype=torch.bool, device=DEV)
    n = out.numel() - GUARD
    keep[:n].view(-1, chans)[:, lo:hi] = False
    return bool(torch.equal(_bits(out)[keep], _bits(before)[keep]))


@pytest.fixture(scope="module")
def engine():
    from vae_decode_hdr_b200.engine import HdrVaeEngine
    from vae_decode_hdr_b200.synthetic import random_decoder_state_dict
    eng = HdrVaeEngine(random_decoder_state_dict(0), DEV)
    yield eng
    eng.close()


@pytest.mark.parametrize("shape", list(SHAPES), ids=list(SHAPES))
@pytest.mark.parametrize("r", ROWS, ids=[r["name"] for r in ROWS])
def test_upscaler_conv_build_against_fp64(engine, r, shape):
    d = make_inputs(r, SHAPES[shape])
    want, bound = reference(r, d)
    ns = _n_store(r["cout"])
    yc = r["yc"] or r["cout"]
    for kernel in KERNELS:
        o = launch(engine, r, SHAPES[shape], kernel, d)
        torch.cuda.synchronize()
        got = o["y"][..., r["yoff"]:r["yoff"] + ns]
        assert torch.isfinite(got).all(), (kernel, "non-finite output: an unread NaN channel reached the result")
        b = bound + (_half_ulp(want.abs() + bound, r["ydt"]) if r["ydt"] != F32 else 0.0)
        ratio = _ratio(got, want, b)
        line = f"{r['name']} {shape} {kernel}: max err/bound y {ratio:.3f}"
        assert ratio <= 1.0, line
        if r["ydt"] == F32:
            rel = float((got.double() - want).norm() / want.norm())
            assert rel <= 1e-5, (line, rel)
        assert _untouched(o["ybuf"], o["before"]["y"], yc, r["yoff"], r["yoff"] + ns), \
            (line, "y changed outside the output slice (or past the buffer end)")
        if r["y2"] is not None:
            y2c, y2off = r["y2"]
            y2off = r["yoff"] if y2off is None else y2off
            got2 = o["y2"][..., y2off:y2off + ns]
            assert torch.isfinite(got2).all(), (line, "non-finite y2")
            ratio2 = _ratio(got2, want, bound + _half_ulp(want.abs() + bound, F16))
            line += f", y2 {ratio2:.3f}"
            assert ratio2 <= 1.0, line
            assert _untouched(o["y2buf"], o["before"]["y2"], y2c, y2off, y2off + ns), \
                (line, "y2 changed outside its slice (or past the buffer end)")
        print(line)


def test_hdrvae_conv2d_rejects_bad_slices(engine):
    """The strides relax the shape checks only as far as the kernels can follow; everything else is refused by name."""
    x = torch.zeros(1, 8, 16, 48, dtype=F16, device=DEV)
    w = torch.zeros(32, 40, 3, 3, device=DEV)
    with pytest.raises(RuntimeError, match="multiple of 64"):
        engine.conv2d(x[..., :40].contiguous(), w, None, 3)                   # Cin 40 without x_channels
    with pytest.raises(RuntimeError, match="x_channels"):
        engine.conv2d(torch.zeros(1, 8, 16, 44, dtype=F16, device=DEV), w, None, 3, cin=40)   # stride 44: not 16 bytes
    with pytest.raises(RuntimeError, match="multiple of 32"):
        engine.conv2d(x, torch.zeros(12, 48, 3, 3, device=DEV), None, 3, cin=48)   # Cout 12 without y_channels
    y = torch.zeros(1, 8, 16, 16, device=DEV)
    with pytest.raises(RuntimeError, match="must lie in y_channels"):
        engine.conv2d(x, torch.zeros(12, 48, 3, 3, device=DEV), None, 3, cin=48, out=y, out_chan_off=8)   # 8 + 12 > 16
    with pytest.raises(RuntimeError, match="must lie in y_channels"):
        engine.conv2d(x, torch.zeros(12, 48, 3, 3, device=DEV), None, 3, cin=48, out=y, out_chan_off=2)   # not 4-aligned


# ---- coverage: the builds the models launch must be builds the rows reach ------------------------------------------
_TAG = re.compile(r"gemm_tc<(\d+),cg(\d),epi(-?\d+),slab(\d+)>")

_MODELS_CHILD = r"""
import torch
from vae_decode_hdr_b200.synthetic import random_compact_state_dict, random_span_state_dict, random_upscaler_state_dict
from vae_decode_hdr_b200.upscaler import HdrUpscalerEngine
forms = [random_upscaler_state_dict(0, nb=1, n_up=u, shuffle=f) for u, f in ((2, 1), (2, 2), (2, 4), (1, 1), (1, 2), (0, 1))]
forms += [random_compact_state_dict(0, nf=nf, nc=2, s=s) for nf in (64, 16) for s in (1, 2, 4)]
forms += [random_span_state_dict(0, nf=nf, s=s) for nf in (48, 16) for s in (1, 2, 4)]
for sd in forms:
    eng = HdrUpscalerEngine(sd, "cuda:0")
    for h, w in ((64, 48), (8, 12)):          # >= 128 network pixels at every unshuffle factor, and < 128
        eng.forward(torch.rand(1, h, w, 3, device="cuda:0"), "none")
    torch.cuda.synchronize()
    eng.close()
"""

_ROWS_CHILD = r"""
import sys
import torch
sys.path.insert(0, "tests")
import test_gpu_conv_upscaler_builds as T
from vae_decode_hdr_b200.engine import HdrVaeEngine
from vae_decode_hdr_b200.synthetic import random_decoder_state_dict
eng = HdrVaeEngine(random_decoder_state_dict(0), T.DEV)
for r in T.ROWS:
    for shape in T.SHAPES.values():
        d = T.make_inputs(r, shape)
        for kernel in ("pair", "single"):
            T.launch(eng, r, shape, kernel, d)
torch.cuda.synchronize()
eng.close()
"""


def _tags_of_child(script):
    """HDRVAE_GEMM_DBG=32 makes every tensor-core conv launch print its build tag; the switch is read once per process."""
    env = dict(os.environ, HDRVAE_GEMM_DBG="32")
    p = subprocess.run([sys.executable, "-c", script], env=env, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-3000:]
    return {m.group(0) for m in _TAG.finditer(p.stdout)}


def test_every_launched_build_has_a_row():
    """One forward of every upscaler form (ESRGAN at every (upsampling convs, unshuffle factor) the library accepts,
    Compact and SPAN at s = 1, 2, 4 and two widths) must launch only builds that the rows above reach: a model form that
    starts launching another build fails here until a row covers it."""
    models = _tags_of_child(_MODELS_CHILD)
    rows = _tags_of_child(_ROWS_CHILD)
    print("builds the models launch:", " ".join(sorted(models)))
    print("builds the rows reach:", " ".join(sorted(rows)))
    assert models, "no build tags: HDRVAE_GEMM_DBG=32 printed nothing"
    assert models <= rows, f"builds launched by a model that no row reaches: {sorted(models - rows)}"
