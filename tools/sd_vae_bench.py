"""Flux-layout vs SD-layout decode at the C2 size, in one process: [4, C, 128, 128] latents -> 4 x 1024^2, "moderate".

  * Flux engine: random-init decoder with conv_in 16 -> 512, C = 16;
  * SD engine: the same graph with conv_in 4 -> 512 plus post_quant_conv (4 -> 4, fused into the latent staging kernel),
    C = 4.

conv_in runs with its input channels padded to 64 in both (K = 9 * 64), so the two should take the same time.  Both are
warmed up (plain decode, CUDA-graph capture, replays), then timed alternately with CUDA events around `--iters` decodes per
round.  Prints the GPU's name and power limit next to the numbers and one JSON line at the end.

  python tools/sd_vae_bench.py [--rounds 5] [--iters 10]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from vae_decode_hdr_b200.engine import HdrVaeEngine  # noqa: E402
from vae_decode_hdr_b200.synthetic import random_decoder_state_dict  # noqa: E402


def gpu_description(index: int) -> str:
    name = torch.cuda.get_device_name(index)
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        q = ""
    return f"{name}, power limit {q or 'unknown'}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sd_vae_bench needs a CUDA device (sm_100a)")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    B, L, mode = 4, 128, "moderate"

    flux_sd = random_decoder_state_dict(0)
    sd_sd = random_decoder_state_dict(0, z_channels=4)
    g = torch.Generator().manual_seed(1)
    sd_sd["post_quant_conv.weight"] = (torch.rand(4, 4, 1, 1, generator=g) * 2 - 1) * 0.5
    sd_sd["post_quant_conv.bias"] = (torch.rand(4, generator=g) * 2 - 1) * 0.5
    engines = {"flux_c16": HdrVaeEngine(flux_sd, dev), "sd_c4": HdrVaeEngine(sd_sd, dev)}
    latents = {k: torch.randn(B, e.latent_channels, L, L, generator=torch.Generator().manual_seed(2)).to(dev)
               for k, e in engines.items()}
    stream = torch.cuda.Stream(dev)                  # a non-default stream: the library captures CUDA graphs there
    times = {k: [] for k in engines}
    with torch.cuda.stream(stream):
        for k, e in engines.items():
            for _ in range(max(3, args.warmup)):    # plain decode, capture, replays
                e.decode(latents[k], mode, 1.0, want_stats=False)
        stream.synchronize()
        for _ in range(args.rounds):
            for k, e in engines.items():
                t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0.record(stream)
                for _ in range(args.iters):
                    e.decode(latents[k], mode, 1.0, want_stats=False)
                t1.record(stream)
                t1.synchronize()
                times[k].append(t0.elapsed_time(t1) / args.iters)
    gpu = gpu_description(dev.index)
    print(f"GPU: {gpu}")
    print(f"C2 decode {B} x [C, {L}, {L}] -> {B} x {8 * L}^2, mode {mode}; {args.rounds} alternating rounds of {args.iters}")
    res = {}
    for k, v in times.items():
        res[k] = {"median_ms": statistics.median(v), "min_ms": min(v), "max_ms": max(v), "rounds_ms": v}
        print(f"  {k:9s} (C = {engines[k].latent_channels:2d}): median {res[k]['median_ms']:.2f} ms per decode "
              f"(min {res[k]['min_ms']:.2f}, max {res[k]['max_ms']:.2f})")
    ratio = res["sd_c4"]["median_ms"] / res["flux_c16"]["median_ms"]
    print(f"  SD / Flux median: {ratio:.4f}")
    print(json.dumps({"gpu": gpu, "batch": B, "latent": L, "mode": mode, "ratio_sd_over_flux": ratio, **res}))
    for e in engines.values():
        e.close()


if __name__ == "__main__":
    main()
