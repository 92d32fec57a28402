"""SPAN upscale timings on one GPU, with Real-ESRGAN Compact general-x4v3 in the same run for reference and a same-GPU
PyTorch comparator.

python tools/span_bench.py [--iters N] [--profile-dir DIR]

Workloads (random-init weights, input in [0, 2.5) so that the first pass is unclamped):
  span-x4        nf 48, 4x: 1024^2 -> 4096^2 (the published default)
  span-x2        nf 48, 2x: 2048^2 -> 4096^2
  span-x1        nf 48, 1x: 1024^2
  general-x4v3   Compact nf 64, nc 32, 4x: 1024^2 -> 4096^2
For each: ms per HDRUpscaleWithModel call (both passes, blend, recombination), output MP/s, the algorithmic network
FLOPs (2 * MACs of the fused convs counted from shapes over the tiles of both passes; SPAN per input pixel per pass:
18 nf (3 + 19 nf + 3 s^2) + 8 nf^2) and their rate over the call, the library's per-op profile (DIR/span_<name>.tsv)
split into network and post-network stages, and PyTorch eager fp16 (cuDNN, channels_last) running the oracle network
over the same tiles as the comparator of the network part (SPAN's eager eval forward re-fuses every Conv3XC on each
call, as spandrel's does)."""
import argparse
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
from _compact_oracle import build_compact  # noqa: E402  (test infrastructure: the comparators' fp32 networks)
from _span_oracle import build_span  # noqa: E402
from vae_decode_hdr_b200 import _native  # noqa: E402
from vae_decode_hdr_b200.upscaler import HdrUpscalerEngine  # noqa: E402

# (name, architecture, nf, Compact body convs, scale, input side)
WORKLOADS = [("span-x4", "span", 48, 0, 4, 1024), ("span-x2", "span", 48, 0, 2, 2048), ("span-x1", "span", 48, 0, 1, 1024),
             ("general-x4v3", "compact", 64, 32, 4, 1024)]
TILE, OVERLAP = 512, 64


def tiles(n):
    """(start, length) of the tiles along one axis (comfy.utils.tiled_scale, as the library cuts them)."""
    pos = [0] if n <= TILE else list(range(0, n - OVERLAP, TILE - OVERLAP))
    out = []
    for p in pos:
        p = max(0, min(n - OVERLAP, p))
        out.append((p, min(TILE, n - p)))
    return out


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "power limit unknown"
    return f"{name} ({q})"


def timed(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def read_profile(path):
    net = post = 0.0
    rows = []
    for line in open(path):
        parts = [p.strip() for p in line.split("\t")]
        if len(parts) < 2 or parts[0].startswith("TOTAL"):
            continue
        ms = float(parts[1].split()[0])
        rows.append((parts[0], ms))
        if parts[0].startswith("conv") or parts[0] in ("upscaler extract tiles", "upscaler pixel shuffle + base",
                                                       "upscaler pixel shuffle"):
            net += ms
        else:
            post += ms
    return rows, net, post


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--profile-dir", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    lib = _native.load_library()
    print("card:", card())
    torch.backends.cudnn.benchmark = True
    for name, arch, nf, nc, s, size in WORKLOADS:
        net = build_span(0, nf=nf, s=s) if arch == "span" else build_compact(0, nf=nf, nc=nc, s=s)
        eng = HdrUpscalerEngine(net.state_dict(), dev)
        g = torch.Generator().manual_seed(1)
        img = (torch.rand(1, size, size, 3, generator=g) * 2.5).to(dev)
        out = eng.upscale(img, "logit")
        torch.cuda.synchronize()
        assert out.shape == (1, s * size, s * size, 3) and bool(torch.isfinite(out).all())
        prof = os.path.join(a.profile_dir or ".", f"span_{name}.tsv") if a.profile_dir else None
        if prof:
            os.makedirs(a.profile_dir, exist_ok=True)
        lib.hdrvae_profile_begin()
        eng.upscale(img, "logit", out=out)
        lib.hdrvae_profile_end(prof.encode() if prof else None)
        ms = timed(lambda: eng.upscale(img, "logit", out=out), a.iters)
        ty, tx = tiles(size), tiles(size)
        tile_px = sum(h * w for _, h in ty for _, w in tx)
        if arch == "span":      # 20 fused 3x3 convs (conv_1, 18 block convs, conv_2), upsampler.0, conv_cat (1x1, 4 nf -> nf)
            flops = 2 * tile_px * (18 * nf * (3 + 19 * nf + 3 * s * s) + 8 * nf * nf)   # both passes
            label = f"{name} (SPAN nf {nf}, {s}x)"
        else:
            flops = 2 * tile_px * 18 * nf * (3 + nc * nf + 3 * s * s)                  # both passes
            label = f"{name} (Compact nf {nf}, nc {nc}, {s}x)"
        print(f"{label} {size}^2 -> {s * size}^2: {ms:.2f} ms per call, "
              f"{flops / 1e12:.2f} TFLOP algorithmic = {flops / ms / 1e9:.0f} TFLOP/s over the call, "
              f"{s * s * size * size / 1e6 / (ms / 1e3):.1f} output MP/s")
        if prof:
            rows, net_ms, post_ms = read_profile(prof)
            agg = {}
            for k, v in rows:
                key = "conv (all)" if k.startswith("conv") else k
                agg[key] = agg.get(key, 0.0) + v
            print(f"  per-op (profiled call): network {net_ms:.2f} ms ({flops / net_ms / 1e9:.0f} TFLOP/s), "
                  f"after the network {post_ms:.2f} ms")
            for k, v in sorted(agg.items(), key=lambda kv: -kv[1]):
                print(f"    {k:<40s} {v:8.3f} ms")
        # comparator: the oracle network in eager fp16 / channels_last over the same tiles (both passes, per tile shape)
        net16 = net.to(dev).half().to(memory_format=torch.channels_last)
        x = img.movedim(-1, 1)
        groups = {}
        for y0, h in ty:
            for x0, w in tx:
                groups.setdefault((h, w), []).append(x[:, :, y0:y0 + h, x0:x0 + w])
        batches = []
        for tl in groups.values():
            b = torch.cat(tl)
            batches.append(torch.cat([b, b.clamp(-1, 1)]).half().contiguous(memory_format=torch.channels_last))

        def eager():
            with torch.no_grad():
                for b in batches:
                    net16(b)
        eager()
        torch.cuda.synchronize()
        ems = timed(eager, a.iters)
        line = f"  PyTorch eager fp16 channels_last, network only over the same tiles: {ems:.2f} ms"
        if prof:
            line += f" (library network part {net_ms:.2f} ms: {ems / net_ms:.2f}x)"
        print(line)
        del net16, batches
        eng.close()
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
