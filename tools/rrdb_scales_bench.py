"""RRDBNet (ESRGAN) upscale timings at 1x and 2x on one GPU, with a same-GPU PyTorch comparator.

python tools/rrdb_scales_bench.py [--iters N] [--profile-dir DIR]

Workloads (nb 23, random-init weights, HDR-like input):
  x2plus      pixel unshuffle f 2, 2 upsampling convs (RealESRGAN_x2plus), 2x: 2048^2 -> 4096^2
  plain-x2    1 upsampling conv, 2x: 2048^2 -> 4096^2
  plain-x1    no upsampling conv (the "1x_" restoration models), 1x: 1024^2
  unshuffle-x1  pixel unshuffle f 4, 2 upsampling convs, 1x: 2048^2
  x4          the 4x model at 1024^2 -> 4096^2, measured in the same run for reference
For each: ms per HDRUpscaleWithModel call (both passes, blend, recombination), algorithmic TFLOP/s of the network (2 *
MACs counted from shapes over the tiles of both passes, over the whole call), output MP/s, the library's per-op profile
(DIR/rrdb_<name>.tsv) split into network and post-network stages, and PyTorch eager fp16 (cuDNN, channels_last) running
the oracle network (tests/_rrdb_oracle.py, reflect pad / unshuffle / crop included) over the same tiles as the
comparator of the network part.  The GPU name and power limit are printed in the same run."""
import argparse
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")]
from _rrdb_oracle import build_upscaler  # noqa: E402  (test infrastructure: the comparator's fp32 network)
from compact_bench import card, read_profile, tiles, timed  # noqa: E402
from vae_decode_hdr_b200 import _native  # noqa: E402
from vae_decode_hdr_b200.upscaler import HdrUpscalerEngine  # noqa: E402

NB = 23
# name, upsampling convs u, unshuffle factor f, input side
WORKLOADS = [("x2plus", 2, 2, 2048), ("plain-x2", 1, 1, 2048), ("plain-x1", 0, 1, 1024), ("unshuffle-x1", 2, 4, 2048),
             ("x4", 2, 1, 1024)]
NETWORK_STAGES = ("upscaler extract tiles", "upscaler crop padded tiles")


def macs_per_net_pixel(nb, u, f):
    """Multiply-adds of the network per pixel of its h' x w' input grid (3x3 convs, nf 64, gc 32)."""
    rdb = sum(32 * (64 + 32 * j) for j in range(4)) + 64 * 192
    m = 64 * 3 * f * f + nb * 3 * rdb + 64 * 64                           # conv_first, trunk, conv_body
    m += sum(4 ** k * 64 * 64 for k in range(1, u + 1))                   # conv_up{k} at 4^k output pixels
    m += 4 ** u * (64 * 64 + 64 * 3)                                      # conv_hr, conv_last
    return 9 * m


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--profile-dir", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    lib = _native.load_library()
    print("card:", card())
    torch.backends.cudnn.benchmark = True
    for name, u, f, size in WORKLOADS:
        s = (1 << u) // f
        net = build_upscaler(0, nb=NB, n_up=u, shuffle=f)
        eng = HdrUpscalerEngine(net.state_dict(), dev)
        assert eng.scale == s
        g = torch.Generator().manual_seed(1)
        img = (torch.rand(1, size, size, 3, generator=g) * 2.5).to(dev)
        out = eng.upscale(img, "atanh")
        torch.cuda.synchronize()
        assert out.shape == (1, s * size, s * size, 3) and bool(torch.isfinite(out).all())
        prof = os.path.join(a.profile_dir, f"rrdb_{name}.tsv") if a.profile_dir else None
        if prof:
            os.makedirs(a.profile_dir, exist_ok=True)
        lib.hdrvae_profile_begin()
        eng.upscale(img, "atanh", out=out)
        lib.hdrvae_profile_end(prof.encode() if prof else None)
        ms = timed(lambda: eng.upscale(img, "atanh", out=out), a.iters)
        ty, tx = tiles(size), tiles(size)
        net_px = sum(-(-h // f) * -(-w // f) for _, h in ty for _, w in tx)
        flops = 2 * 2 * net_px * macs_per_net_pixel(NB, u, f)             # both passes
        print(f"{name} (nb {NB}, u {u}, f {f}, {s}x) {size}^2 -> {s * size}^2: {ms:.2f} ms per call, "
              f"{flops / 1e12:.2f} TFLOP algorithmic = {flops / ms / 1e9:.0f} TFLOP/s over the call, "
              f"{s * s * size * size / 1e6 / (ms / 1e3):.1f} output MP/s")
        if prof:
            rows, _, _ = read_profile(prof)
            net_ms = sum(v for k, v in rows if k.startswith("conv") or k in NETWORK_STAGES)
            post_ms = sum(v for k, v in rows if not (k.startswith("conv") or k in NETWORK_STAGES))
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
