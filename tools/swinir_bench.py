"""SwinIR upscale timings on one GPU, with a same-GPU PyTorch comparator.

python tools/swinir_bench.py [--iters N] [--profile-dir DIR] [--only NAME]

Workloads (random-init weights in spandrel's layout, input in [0, 2.5) so that the first pass is unclamped):
  m-classical-x4    SwinIR-M classical SR: C 180, 6 x 6 blocks, heads 6, "pixelshuffle", 1conv: 1024^2 -> 4096^2
  m-realworld-x4    SwinIR-M real-world SR: as above with "nearest+conv": 1024^2 -> 4096^2
  lightweight-x4    C 60, 4 x 6 blocks, "pixelshuffledirect": 1024^2 -> 4096^2
  m-classical-x2    SwinIR-M classical SR 2x: 2048^2 -> 4096^2
For each: ms per HDRUpscaleWithModel call (both passes, blend, recombination; device events over --iters calls after a
warm-up), the algorithmic network FLOPs over the tiles of both passes (2 x MACs from the shapes, attention with the true
head dimension) and the bytes of the unfused plan's transformer layers and RSTB convs (fp32 stream, fp16 operands, no
weights, no tail), each over the call and against the floors at the HGX B200 data sheet's 2250 TFLOP/s (dense fp16) and
7.7 TB/s; the library's per-op profile of one call grouped into linears, attention, LayerNorm, convs and the rest
(DIR/swinir_<name>.tsv); and PyTorch eager fp16 running the oracle network (tests/_swinir_oracle.py) over the same tiles."""
import argparse
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")]
from _swinir_oracle import build_swinir  # noqa: E402  (test infrastructure: the comparator's fp32 network)
from span_bench import card, read_profile, tiles, timed  # noqa: E402
from vae_decode_hdr_b200 import _native  # noqa: E402
from vae_decode_hdr_b200.upscaler import HdrUpscalerEngine  # noqa: E402

# (name, C, depths, heads, upsampler, scale, resi_connection, input side)
WORKLOADS = [("m-classical-x4", 180, (6,) * 6, 6, "pixelshuffle", 4, "1conv", 1024),
             ("m-realworld-x4", 180, (6,) * 6, 6, "nearest+conv", 4, "1conv", 1024),
             ("lightweight-x4", 60, (6,) * 4, 6, "pixelshuffledirect", 4, "1conv", 1024),
             ("m-classical-x2", 180, (6,) * 6, 6, "pixelshuffle", 2, "1conv", 2048)]
PEAK_TFLOPS, PEAK_TBS = 2250.0, 7.7


def costs(C, depths, heads, upsampler, s, hidden):
    """(FLOPs, bytes) per input pixel of one pass: the network's algorithmic FLOPs; bytes of the STLs and RSTB convs."""
    nstl, nrstb = sum(depths), len(depths)
    stl = 8 * C * C + 4 * hidden * C + 4 * 64 * C                       # qkv, proj, fc1, fc2, q k^T and P V
    body = 2 * 9 * C * C                                                # one 1conv
    f = 2 * 27 * C + nstl * stl + (nrstb + 1) * body
    if upsampler == "pixelshuffle":
        k = {2: 1, 4: 2}[s]
        f += 2 * 9 * C * 64 + sum(2 * 9 * 64 * 256 * 4 ** i for i in range(k)) + 2 * 9 * 64 * 3 * s * s
    elif upsampler == "nearest+conv":
        k = {2: 1, 4: 2}[s]
        f += 2 * 9 * C * 64 + sum(2 * 9 * 64 * 64 * 4 ** i for i in range(1, k + 1)) + 2 * 9 * 64 * (64 + 3) * s * s
    elif upsampler == "pixelshuffledirect":
        f += 2 * 9 * C * 3 * s * s
    else:
        f += 2 * 9 * C * 3
    CP, QK, HP = (C + 7) // 8 * 8, heads * 32, (hidden + 7) // 8 * 8
    b_stl = ((4 * C + 2 * CP) * 2                                       # two LayerNorms
             + 2 * CP + 6 * QK                                          # qkv
             + 6 * QK + 2 * QK                                          # attention
             + 2 * QK + 8 * C                                           # proj + residual
             + 2 * CP + 2 * HP                                          # fc1
             + 2 * HP + 8 * C)                                          # fc2 + residual
    b_rstb = 2 * CP + 8 * C + 2 * CP
    return f, nstl * b_stl + nrstb * b_rstb


GROUPS = (("linears (qkv, proj, fc1, fc2)", lambda k: k.startswith("conv1x1")),
          ("window attention", lambda k: k == "swinir window attention"),
          ("LayerNorm", lambda k: k == "swinir layernorm"),
          ("3x3 convs", lambda k: k.startswith("conv3x3")),
          ("tail shuffles / crop / extract", lambda k: True))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--profile-dir", default=None)
    ap.add_argument("--only", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    lib = _native.load_library()
    print("card:", card())
    torch.backends.cudnn.benchmark = True
    for name, C, depths, heads, ups, s, resi, size in WORKLOADS:
        if a.only and name != a.only:
            continue
        net = build_swinir(0, C, depths, heads, 2.0, ups, s, resi, True)
        eng = HdrUpscalerEngine(net.state_dict(), dev)
        g = torch.Generator().manual_seed(1)
        img = (torch.rand(1, size, size, 3, generator=g) * 2.5).to(dev)
        out = eng.upscale(img, "atanh")
        torch.cuda.synchronize()
        assert out.shape == (1, s * size, s * size, 3) and bool(torch.isfinite(out).all())
        ms = timed(lambda: eng.upscale(img, "atanh", out=out), a.iters)
        ty, tx = tiles(size), tiles(size)
        tile_px = sum(h * w for _, h in ty for _, w in tx)
        fpx, bpx = costs(C, depths, heads, ups, s, 2 * C)
        flops, byts = 2 * tile_px * fpx, 2 * tile_px * bpx                # both passes
        fl_ms, by_ms = flops / PEAK_TFLOPS / 1e9, byts / PEAK_TBS / 1e9
        print(f"{name} (C {C}, {len(depths)} x {depths[0]} blocks, {ups}, {s}x) {size}^2 -> {s * size}^2: {ms:.1f} ms per "
              f"call; {flops / 1e12:.1f} TFLOP = {flops / ms / 1e9:.0f} TFLOP/s (floor {fl_ms:.1f} ms); STL + RSTB bytes "
              f"{byts / 1e12:.3f} TB = {byts / ms / 1e9:.2f} TB/s (floor {by_ms:.1f} ms); "
              f"{'HBM' if by_ms > fl_ms else 'FLOP'}-bound plan, {max(fl_ms, by_ms) / ms * 100:.0f} % of that floor")
        if a.profile_dir:
            os.makedirs(a.profile_dir, exist_ok=True)
            prof = os.path.join(a.profile_dir, f"swinir_{name}.tsv")
            lib.hdrvae_profile_begin()
            eng.upscale(img, "atanh", out=out)
            lib.hdrvae_profile_end(prof.encode())
            rows, _, _ = read_profile(prof)
            total = sum(v for _, v in rows)
            agg = {}
            for k, v in rows:
                grp = next(gname for gname, f in GROUPS if f(k))
                agg[grp] = agg.get(grp, 0.0) + v
            print(f"  per-op (profiled call, {total:.1f} ms):")
            for k, v in sorted(agg.items(), key=lambda kv: -kv[1]):
                print(f"    {k:<36s} {v:8.2f} ms  {v / total * 100:5.1f} %")
        eng.close()
        # comparator: the oracle network in eager fp16 over the same tiles (both passes, per tile shape)
        net16 = net.to(dev).half()
        x = img.movedim(-1, 1)
        groups = {}
        for y0, h in ty:
            for x0, w in tx:
                groups.setdefault((h, w), []).append(x[:, :, y0:y0 + h, x0:x0 + w])
        batches = []
        for tl in groups.values():
            b = torch.cat(tl)
            batches.extend([b.half(), b.clamp(-1, 1).half()])

        def eager():
            with torch.no_grad():
                for b in batches:
                    net16(b)
        eager()
        torch.cuda.synchronize()
        ems = timed(eager, a.iters)
        print(f"  PyTorch eager fp16, network only over the same tiles: {ems:.1f} ms (library call {ms:.1f} ms: "
              f"{ems / ms:.2f}x)")
        del net16, batches
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
