"""The tensor-core conv builds the SwinIR upscaler launches, one launch at a time against fp64, in the style of
tests/test_gpu_conv_upscaler_builds.py (whose inputs, sentinels, bounds and shapes this file reuses): the GELU epilogue,
the 192-column tiles (qkv, proj, fc1, fc2, the RSTB conv at embed_dim 180), the 3conv triple, and the LeakyReLU slope 0.01
of conv_before_upsample.  test_every_swinir_build_has_a_row checks that every build the SwinIR forms launch is reached by
these rows or by the conv-only upscalers' rows."""
import math
import os
import subprocess
import sys

import pytest
import torch
import torch.nn.functional as F

import test_gpu_conv_upscaler_builds as T

pytestmark = pytest.mark.gpu
DEV = T.DEV
F16, F32 = T.F16, T.F32
LRELU_001 = float(torch.tensor(0.01, dtype=F32))    # nn.LeakyReLU()'s default slope, as the kernels hold it in fp32
GELU_REL = 2.0 ** -21                               # erff's error (2 ulp) and the fp32 products of 0.5 t (1 + erf(t / sqrt 2))


def row(name, build, cin, cout, act=None, slope=None, **k):
    r = T.row(name, build, cin, cout, act=act, **k)
    r["slope"] = slope
    return r


def _rows(C, heads, hidden):
    """The call sites of up_forward_swinir at embed_dim C (fp16 pixel stride CP = round_up(C, 8))."""
    CP, QK, HP = (C + 7) // 8 * 8, heads * 32, (hidden + 7) // 8 * 8
    c4 = C // 4
    c4p = (c4 + 7) // 8 * 8
    n = f"swin{C}"
    return [
        row(f"{n}.conv_first", "generic", 3, C, xc=8, yc=C),
        row(f"{n}.qkv", "192 / generic", C, 3 * QK, ks=1, xc=CP, yc=3 * QK, ydt=F16),
        row(f"{n}.proj", "192 EPI_RES / 64 generic", QK, C, ks=1, xc=QK, yc=C, res=True),
        row(f"{n}.fc1.gelu", "192 / 128 generic (GELU)", C, hidden, ks=1, xc=CP, yc=HP, ydt=F16, act="gelu"),
        row(f"{n}.fc2", "192 EPI_RES / 64 generic", hidden, C, ks=1, xc=HP, yc=C, res=True),
        row(f"{n}.fc2.last", "generic", hidden, C, ks=1, xc=HP, yc=C, res=True, y2=(CP, 0)),
        row(f"{n}.rstb_conv", "192 EPI_RES / 64 slab generic", C, C, xc=CP, yc=C, res=True),
        row(f"{n}.conv_after_body", "generic", C, C, xc=CP, yc=C, res=True, y2=(CP, 0)),
        row(f"{n}.conv3.0", "OUT16|LRELU", C, c4, xc=CP, yc=c4p, ydt=F16, act="lrelu", slope=T.LRELU),
        row(f"{n}.conv3.2", "OUT16|LRELU (1x1)", c4, c4, ks=1, xc=c4p, yc=c4p, ydt=F16, act="lrelu", slope=T.LRELU),
        row(f"{n}.conv3.4", "192 EPI_RES / 64 generic", c4, C, xc=c4p, yc=C, res=True),
        row(f"{n}.conv_before_upsample", "64 OUT16|LRELU at slope 0.01", C, 64, xc=CP, yc=64, ydt=F16, act="lrelu",
            slope=LRELU_001),
        row(f"{n}.direct.s2", "32 / 64", C, 12, xc=CP, yc=12),
        row(f"{n}.direct.s4", "64 generic", C, 48, xc=CP, yc=48),
        row(f"{n}.conv_last.s1", "32", C, 3, xc=CP, yc=4),
    ]


ROWS = _rows(180, 6, 360) + _rows(60, 6, 120) + [
    row("swin.upsample.pixelshuffle", "256 OUT16", 64, 256, xc=64, yc=256, ydt=F16),
    row("swin.conv_hr", "64 OUT16|LRELU", 64, 64, ydt=F16, act="lrelu", slope=T.LRELU),
]


def launch(eng, r, shape, kernel, d):
    """T.launch with this file's GELU and LeakyReLU slope."""
    from vae_decode_hdr_b200 import _native as N
    B, H, W = shape
    cin, cout = r["cin"], r["cout"]
    yc = r["yc"] or cout
    y, ybuf = T._sentinel((B, H, W, yc), r["ydt"])
    x, _ = T._sentinel((B, H, W, r["xc"] or cin), F16)
    x[..., :cin] = d["xs"].to(DEV)
    y2 = y2buf = None
    if r["y2"] is not None:
        y2, y2buf = T._sentinel((B, H, W, r["y2"][0]), F16)
    before = {"y": ybuf.clone(), "y2": y2buf.clone() if y2buf is not None else None}
    eng.set_cta_group(1 if kernel == "single" else 0)
    eng.conv2d(x, d["w"].to(DEV), d["b"].to(DEV), r["ks"], False, d["r"].to(DEV) if r["res"] else None,
               impl=N.CONV_DIRECT if kernel == "direct" else N.CONV_TCGEN05, cin=cin if r["xc"] else None, out=y,
               out2=y2, out2_chan_off=r["y2"][1] if r["y2"] else None,
               lrelu=r["slope"] if r["act"] == "lrelu" else 0.0, act=N.ACT_GELU if r["act"] == "gelu" else N.ACT_NONE)
    eng.set_cta_group(0)
    return dict(y=y, ybuf=ybuf, y2=y2, y2buf=y2buf, before=before)


def reference(r, d):
    cout, ks = r["cout"], r["ks"]
    ns = T._n_store(cout)
    x = d["xs"].to(DEV).double().permute(0, 3, 1, 2)
    w = torch.zeros(ns, r["cin"], ks, ks, dtype=torch.float64, device=DEV)
    w[:cout] = d["w"].to(DEV).double()
    b = torch.zeros(ns, dtype=torch.float64, device=DEV)
    b[:cout] = d["b"].to(DEV).double()
    u = F.conv2d(x, w, b, padding=ks // 2).permute(0, 2, 3, 1)
    M = F.conv2d(x.abs(), w.abs(), b.abs(), padding=ks // 2).permute(0, 2, 3, 1)
    if r["res"]:
        rr = d["r"].to(DEV).double()[..., :ns]
        u, M = u + rr, M + rr.abs()
    eps = 2.0 ** -18 * M
    if r["act"] == "lrelu":
        return torch.where(u < 0, u * r["slope"], u), eps
    if r["act"] == "gelu":
        y = 0.5 * u * (1 + torch.erf(u / math.sqrt(2)))
        return y, 1.13 * eps + GELU_REL * y.abs() + 2.0 ** -30                  # |gelu'| <= 1.13
    return u, eps


@pytest.fixture(scope="module")
def engine():
    from vae_decode_hdr_b200.engine import HdrVaeEngine
    from vae_decode_hdr_b200.synthetic import random_decoder_state_dict
    eng = HdrVaeEngine(random_decoder_state_dict(0), DEV)
    yield eng
    eng.close()


@pytest.mark.parametrize("shape", list(T.SHAPES), ids=list(T.SHAPES))
@pytest.mark.parametrize("r", ROWS, ids=[r["name"] for r in ROWS])
def test_swinir_conv_build_against_fp64(engine, r, shape):
    d = T.make_inputs(r, T.SHAPES[shape])
    want, bound = reference(r, d)
    ns = T._n_store(r["cout"])
    yc = r["yc"] or r["cout"]
    for kernel in T.KERNELS:
        o = launch(engine, r, T.SHAPES[shape], kernel, d)
        torch.cuda.synchronize()
        got = o["y"][..., :ns]
        assert torch.isfinite(got).all(), (kernel, "non-finite output: an unread NaN channel reached the result")
        b = bound + (T._half_ulp(want.abs() + bound, r["ydt"]) if r["ydt"] != F32 else 0.0)
        ratio = T._ratio(got, want, b)
        line = f"{r['name']} {shape} {kernel}: max err/bound y {ratio:.3f}"
        assert ratio <= 1.0, line
        assert T._untouched(o["ybuf"], o["before"]["y"], yc, 0, ns), (line, "y changed outside the output slice")
        if r["y2"] is not None:
            got2 = o["y2"][..., :ns]
            ratio2 = T._ratio(got2, want, bound + T._half_ulp(want.abs() + bound, F16))
            line += f", y2 {ratio2:.3f}"
            assert ratio2 <= 1.0, line
            assert T._untouched(o["y2buf"], o["before"]["y2"], r["y2"][0], 0, ns), (line, "y2 changed outside its slice")
        print(line)


_SWIN_CHILD = r"""
import torch
from vae_decode_hdr_b200.synthetic import random_swinir_state_dict
from vae_decode_hdr_b200.upscaler import HdrUpscalerEngine
forms = [("pixelshuffle", 2), ("pixelshuffle", 4), ("pixelshuffledirect", 2), ("pixelshuffledirect", 4),
         ("nearest+conv", 2), ("nearest+conv", 4), ("", 1)]
sds = [random_swinir_state_dict(0, C, (2,), 6, 2.0, u, s, resi, pn) for C in (180, 60) for u, s in forms
       for resi, pn in (("1conv", True), ("3conv", False))]
for sd in sds:
    eng = HdrUpscalerEngine(sd, "cuda:0")
    for h, w in ((64, 48), (8, 12)):
        eng.forward(torch.rand(1, h, w, 3, device="cuda:0"), "none")
    torch.cuda.synchronize()
    eng.close()
"""

_ROWS_CHILD = r"""
import sys
import torch
sys.path.insert(0, "tests")
import test_gpu_conv_upscaler_builds as T
import test_gpu_conv_swinir_builds as S
from vae_decode_hdr_b200.engine import HdrVaeEngine
from vae_decode_hdr_b200.synthetic import random_decoder_state_dict
eng = HdrVaeEngine(random_decoder_state_dict(0), T.DEV)
for mod in (T, S):
    for r in mod.ROWS:
        for shape in T.SHAPES.values():
            d = T.make_inputs(r, shape)
            for kernel in ("pair", "single"):
                mod.launch(eng, r, shape, kernel, d)
torch.cuda.synchronize()
eng.close()
"""


def test_every_swinir_build_has_a_row():
    """Every SwinIR form (each upsampler at each scale, embed_dim 180 and 60, 1conv and 3conv) must launch only builds
    that the rows here or the conv-only upscalers' rows reach."""
    models = T._tags_of_child(_SWIN_CHILD)
    rows = T._tags_of_child(_ROWS_CHILD)
    print("builds the SwinIR forms launch:", " ".join(sorted(models)))
    assert models, "no build tags: HDRVAE_GEMM_DBG=32 printed nothing"
    assert models <= rows, f"builds launched by a SwinIR form that no row reaches: {sorted(models - rows)}"
