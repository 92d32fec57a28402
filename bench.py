#!/usr/bin/env python
"""bench.py — Flux-VAE HDR decode throughput on B200 (BASELINE.json metric: megapixels/s).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
         --master-port P bench.py --gpus N --steps K --warmup W

A step = one pass of the hot path (HDRVAEDecode.simple_hdr_decode's happy path, reference
hdr_vae_decode.py:62-195, ONE decoder pass) over one batch of synthetic latents.
Workload per GPU: BASELINE config C2 — 4x16x128x128 latents -> 4 x 1024x1024, "moderate" mode, bf16
tensor-core decoder (fp16 operands, the 16-bit mode that meets the 1e-2 parity tolerance).  N > 1: batch sharding (config C3 style): every rank decodes 4 more images and
the batch-global HDR statistics are all-reduced over NCCL between epilogue phase A and B ("weak").

value : device-timed MP/s, latents resident in HBM, max over ranks.
e2e   : the same metric through the node API with HOST buffers (pinned latent H2D + IMAGE D2H inside
        the timed region).
roofline : the tcgen05 implicit-GEMM conv kernel (dominant): algorithmic conv FLOPs of one step
        (9.4628 MFLOP per output pixel, SURVEY.md §8d) / summed device time of its launches in one
        step (CUDA events on the launching stream), against the measured sustained bf16 peak.
cpu_baseline : the oracle port of the reference node on the host cores, bounded sample (one C1-sized call).
torch_eager_gpu : the same decoder graph in PyTorch eager (cuDNN) on the SAME B200 + the reference's eager HDR math,
        fp32 (TF32 off) and bf16 autocast, CUDA-event timed — the comparator SURVEY.md §2.1 names.
aux_c4_4096 / aux_c4_rows : BASELINE config C4 (1x16x512x512 -> 4096^2, "aggressive") on one GPU, and — for N > 1 —
        row-tiled over the N GPUs of the job (strong scaling), outside the headline's timed region.
--impl reference : the reference node's CPU path (oracle port, TWO decoder passes + conv_out per call as the
        reference does) on the host cores: every step is ONE image of the C2 batch at its full 1024^2 size.
--dump-outputs DIR : after the timed steps, the IMAGE the last timed step returned is written as DIR/image.npy
        (float32 [4, 1024, 1024, 3]; --impl reference: [1, 1024, 1024, 3]; N > 1: DIR/image_rank<r>.npy per rank, a fixed
        sample of its pixels where the files together would pass 64 MB).  Weights and latents are seeded, so two builds
        run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "flux_vae_hdr_decode_megapixels_per_s"
UNIT = "MP/s"
CONV_MFLOP_PER_PX = 9.4628          # SURVEY.md §8d: 3x3/1x1 convs of the decoder, resolution independent
PER_GPU_BATCH, LATENT = 4, 128      # config C2
MODE = "moderate"
C4_ROOFLINE_MP_S = 76.8             # SURVEY.md §8d: 17.851 MFLOP/px at 4096^2 against the sustained bf16 peak, per GPU
DUMP_BYTES = 64 * 10 ** 6           # --dump-outputs: at most this many bytes over all files of all ranks


def workload_config(world: int) -> dict:
    """The `config` object of the JSON line: ONE function for both arms, so the reference arm reports exactly the
    configuration the B200 arm measures (arm-specific detail lives outside `config`)."""
    B, L = PER_GPU_BATCH, LATENT
    return {"workload": f"C2 per GPU: {B}x16x{L}x{L} random latents -> {B} x {8 * L}x{8 * L}, mode {MODE} "
                        "(smart expansion x3), Flux.1 AE decoder random-init",
            "global_batch": B * world,
            "parallelism": "single GPU" if world == 1 else f"batch-sharded dp{world} + all-reduce of HDR statistics",
            "l2": "inputs larger than L2: ~6 GB of activations stream through HBM every step (L2 126 MB)"}


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["bf16_tflops_sustained"]), float(p["hbm_gbs"]), "measured"
    except Exception:
        return 1400.0, 6650.0, "fallback"      # B200_PROFILING.md fallback (sustained bf16, HBM copy)


def _burst_peak():
    """cuBLAS bf16 rate of a GEMM timed alone (best of 10), the other figure MEASURED_PEAKS.json holds."""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["bf16_tflops"])
    except Exception:
        return 1650.0


class ClockSampler:
    """SM clock and throttle reasons of one GPU sampled DURING the timed region (B200_PROFILING.md recipe).
    NVML in-process (microseconds per query, so even a 0.2 s region yields dozens of samples on an 8-GPU box where
    spawning nvidia-smi takes longer than the region); `nvidia-smi -lms` as the fallback."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index: int):
        self.rows, self.proc, self.index, self.stop, self.t, self.src = [], None, index, False, None, None

    def _nvml_loop(self, nv, h):
        bits = [(getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8), "hw_slowdown"),
                (getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40), "hw_thermal_slowdown"),
                (getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20), "sw_thermal_slowdown"),
                (getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4), "sw_power_cap")]
        try:
            mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        except Exception:
            mx = 0
        while not self.stop:
            try:
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.rows.append([str(sm), str(mx)] + ["Active" if r & b else "Not Active" for b, _ in bits])
            except Exception:
                pass
            time.sleep(0.005)

    def __enter__(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            # NVML enumerates physical devices: honour CUDA_VISIBLE_DEVICES when it is a plain index list
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            phys = self.index
            if vis and all(v.strip().isdigit() for v in vis.split(",")):
                phys = int(vis.split(",")[self.index])
            h = nv.nvmlDeviceGetHandleByIndex(phys)
            self.src = "nvml"
            self.t = threading.Thread(target=self._nvml_loop, args=(nv, h), daemon=True)
            self.t.start()
            return self
        except Exception:
            pass
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.src = "nvidia-smi"
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        self.stop = True
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        elif self.t is not None:
            self.t.join(timeout=1)

    def summary(self):
        sm, mx, reasons = [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
                for n, v in zip(self.NAMES, r[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm), "source": self.src}


def cpu_reference_run(steps: int, warmup: int, sample_latent: int = 64, dec=None):
    """The reference node's CPU path (oracle port: fp32 PyTorch eager decoder + the restated HDR math, with the
    reference's real call structure: TWO decoder passes + a third conv_out per call, hdr_vae_decode.py:859,876,1022)
    on all host cores.  One 1x16xSxS latent per step, `steps` timed steps.
    -> (summary dict, seconds per step, the image the last timed step returned)."""
    import torch
    from oracle import hdr_oracle as ho
    from oracle.flux_decoder import build_decoder, make_latent
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    dec = dec if dec is not None else build_decoder(0)
    z = make_latent(1, sample_latent, sample_latent, seed=1234)
    times = []
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            _ = dec(z)                                            # analyze_conv_out's vae.decode (:859)
            out, st, _pre = ho.simple_hdr_decode(dec, z, MODE, 1.0)   # second decode (:1022) + conv_out + HDR math
            dt = time.perf_counter() - t0
            if i >= warmup:
                times.append(dt)
    mp = (8 * sample_latent) ** 2 / 1e6
    per = sum(times) / len(times)
    return {"value": mp / per, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{len(times)} x (1x16x{sample_latent}x{sample_latent} latent -> {8 * sample_latent}^2, {MODE}; "
                      f"2 decoder passes + conv_out as the reference node does), {per:.2f} s per call, fp32 torch CPU, "
                      f"{cores} threads"}, per, out


def run_reference_arm(args):
    """`--impl reference`: the reference's CPU implementation of the path on the box's host cores, on the B200 arm's
    config.  Every step decodes ONE image of the C2 batch at its full size (1x16x128x128 -> 1024^2, "moderate") with
    the reference node's call structure; MP/s is per pixel, so one image of the batch is a bounded sample of the
    4-image step.  Warm-up is a single C2-sized call, then exactly --steps timed calls (each takes seconds to minutes
    on the host cores).  Three C1-sized calls (1x16x64x64 -> 512^2, BASELINE configs[0], the reference's own
    CPU-runnable case) are timed as well and reported in cpu_baseline.  --dump-outputs: the image of the last timed call,
    DIR/image.npy (float32 [1, 1024, 1024, 3])."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle.flux_decoder import build_decoder
    dec = build_decoder(0)
    c1, c1_per, _ = cpu_reference_run(3, 1, 64, dec=dec)
    base, per, last_out = cpu_reference_run(args.steps, 1, LATENT, dec=dec)
    if args.dump_outputs:
        dump_output(args.dump_outputs, "image", last_out, DUMP_BYTES)
    base["c1_512"] = {"value": c1["value"], "unit": UNIT, "s_per_call": c1_per, "calls": 3,
                      "workload": "C1: 1x16x64x64 latent -> 512x512, reference node call structure"}
    line = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": 1, "ms_per_step": per * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.gpus),
            "reference_step": f"one image of the C2 batch at full size: 1x16x{LATENT}x{LATENT} -> {8 * LATENT}^2, {MODE}, "
                              "two decoder passes + conv_out + eager HDR math per call (hdr_vae_decode.py:859,876,1022)",
            "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


def torch_eager_gpu(dev, B: int, L: int, seed: int) -> dict:
    """Same-box comparator (SURVEY.md §2.1): the decoder graph in PyTorch eager on this B200 (cuDNN convs, eager
    GroupNorm / SiLU / attention) + the reference's eager HDR math, on the headline workload.  (i) fp32 with TF32 off,
    (ii) bf16 autocast.  Timed with CUDA events: `node_call` = the reference node's call structure (two decoder passes +
    conv_out, hdr_vae_decode.py:859,876,1022), `one_pass` = a single decoder pass + HDR math (what this library runs).
    The oracle decoder is used here as a timed baseline only, never by the product path."""
    import torch
    from oracle import hdr_oracle as ho
    from oracle.flux_decoder import build_decoder, make_latent
    res = {}
    tf32 = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    try:
        dec = build_decoder(0).to(dev)
        z = make_latent(B, L, L, seed=seed).to(dev)
        mp = B * (8 * L) ** 2 / 1e6

        def timed(fn, reps):
            fn(); torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                fn()
            e1.record(); torch.cuda.synchronize(dev)
            return e0.elapsed_time(e1) / reps

        for name, ctx, reps in (("fp32_tf32_off", torch.autocast("cuda", enabled=False), 2),
                                ("bf16_autocast", torch.autocast("cuda", dtype=torch.bfloat16), 3)):
            with torch.no_grad(), ctx:
                def one_pass():
                    return ho.simple_hdr_decode(dec, z, MODE, 1.0)[0]

                def node_call():
                    dec(z)
                    return ho.simple_hdr_decode(dec, z, MODE, 1.0)[0]
                ms1 = timed(one_pass, reps)
                ms2 = timed(node_call, reps)
            res[name] = {"node_call_ms": ms2, "node_call_mp_s": mp / (ms2 / 1e3), "one_pass_ms": ms1,
                         "one_pass_mp_s": mp / (ms1 / 1e3)}
        res["workload"] = f"{B}x16x{L}x{L} -> {B} x {8 * L}^2, {MODE}; torch {torch.__version__} eager, cuDNN {torch.backends.cudnn.version()}"
        del dec, z
    except Exception as exc:      # a comparator must never cost the headline line
        res["error"] = repr(exc)[:300]
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = tf32
        torch.cuda.empty_cache()
    return res


_REAL_STDOUT = None


def guard_stdout() -> None:
    """stdout carries exactly ONE JSON line.  Libraries write there too (NCCL prints its version banner with printf when
    NCCL_DEBUG is set on the box, regardless of NCCL_DEBUG_FILE), so file descriptor 1 is pointed at stderr for the whole
    run and the JSON line goes to a private duplicate of the original stdout."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line: dict) -> None:
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def dump_output(dirname: str, name: str, t, budget: int) -> None:
    """Write tensor `t` as dirname/name.npy in float32.  When it would exceed `budget` bytes, a fixed sample of its pixels
    (rows of the last dimension, drawn with seed 0 and kept in order) is written instead, [n_sampled, last dim]: the same
    pixels on every run for the same shape."""
    import numpy as np
    import torch
    t = t.detach().float()
    if t.numel() * 4 + 128 > budget:                          # 128: the .npy header
        rows = t.reshape(-1, t.shape[-1])
        keep = (budget - 128) // (4 * rows.shape[1])
        idx = torch.randperm(rows.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values
        t = rows[idx.to(rows.device)]
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, name + ".npy"), t.cpu().numpy())


def main():
    guard_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-aux", action="store_true", help="skip the auxiliary 4096^2 single-GPU measurement")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager", action="store_true", help="skip the PyTorch-eager-on-the-same-GPU comparator")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the image of the last timed step to DIR/image.npy (float32) for output comparisons")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference_arm(args)
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    from vae_decode_hdr_b200 import NODE_CLASS_MAPPINGS, _native
    from vae_decode_hdr_b200.engine import HdrVaeEngine
    from vae_decode_hdr_b200.sharding import decode_batch_sharded
    from vae_decode_hdr_b200.synthetic import SyntheticVAE, random_decoder_state_dict, synthetic_latent

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N > 1")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # NCCL writes its debug output (the "NCCL version ..." banner on boxes that set NCCL_DEBUG) to stdout by
        # default: send it to stderr so that stdout stays the one JSON line
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    lib = _native.load_library()

    B, L = PER_GPU_BATCH, LATENT
    sd = random_decoder_state_dict(0)
    engine = HdrVaeEngine(sd, dev)
    z_dev = synthetic_latent(B, L, L, seed=1234 + rank).to(dev)
    mp_per_rank = B * (8 * L) ** 2 / 1e6

    def step_device():
        if world > 1:
            return decode_batch_sharded(engine, z_dev, MODE, 1.0, want_stats=False)
        return engine.decode(z_dev, MODE, 1.0, want_stats=False)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(args.warmup):
        step_device()
    barrier()
    n0 = lib.hdrvae_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clocks:
        barrier()
        e0.record()
        for _ in range(args.steps - 1):
            step_device()
        last_out, _ = step_device()
        e1.record()
        barrier()
    launches = lib.hdrvae_launch_count() - n0
    if args.dump_outputs:
        dump_output(args.dump_outputs, "image" if world == 1 else f"image_rank{rank}", last_out, DUMP_BYTES // world)
    del last_out
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    ms_step = ms_total / args.steps
    value = mp_per_rank * world / (ms_step / 1e3)

    # ---- roofline of the dominant kernel (tcgen05 conv): per-op CUDA events over one extra step
    peak_tf, peak_gbs, peak_src = _peaks()
    prof_path = os.path.join(tempfile.gettempdir(), f"hdrvae_prof_{os.getpid()}.tsv")
    lib.hdrvae_profile_begin()
    engine.decode(z_dev, MODE, 1.0, want_stats=False)
    lib.hdrvae_profile_end(prof_path.encode())
    conv_ms = gn_ms = attn_ms = epi_ms = gn_bytes = 0.0
    attn_kernel_ms = None
    n_conv = 0
    with open(prof_path) as f:
        for ln in f:
            cols = ln.split("\t")
            name, t = cols[0].strip(), float(cols[1].split()[0])
            if name.startswith("conv3x3 128->8 "):
                continue      # conv_out on the tensor cores: nested inside (and counted with) "epilogue phase A"
            if name.startswith("attention fused kernel"):
                attn_kernel_ms = t
                continue      # nested inside (and counted with) "attention core"
            if name.startswith("conv"):
                conv_ms += t; n_conv += 1
            elif name.startswith("groupnorm"):
                gn_ms += t
                gn_bytes += float(cols[3].split()[0]) * 1e9 * t / 1e3      # the scope's own byte count (actual dtypes)
            elif name.startswith("attention"):
                attn_ms += t
            elif name.startswith("epilogue"):
                epi_ms += t
    os.unlink(prof_path)
    conv_flops = CONV_MFLOP_PER_PX * 1e6 * B * (8 * L) ** 2 - 2.0 * 1152 * 3 * B * (8 * L) ** 2  # conv_out runs in the epilogue
    achieved_tf = conv_flops / (conv_ms / 1e3) / 1e12
    # the three upsample convs run as four 2x2-tap phase convs (nearest-2x folded into the load): 4/9 of their
    # algorithmic FLOPs are executed.  Per output pixel of the decoder: up convs = 2*9*(512*512/16 + 512*512/4 + 256*256)
    up_flops = 2.0 * 9 * (512 * 512 / 16.0 + 512 * 512 / 4.0 + 256 * 256) * B * (8 * L) ** 2
    executed_tf = (conv_flops - up_flops * 5.0 / 9.0) / (conv_ms / 1e3) / 1e12
    roofline = {"bound": "tensor", "kernel": "gemm_tc_kernel (tcgen05 implicit-GEMM conv, all conv layers of one step)",
                "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved_tf / peak_tf,
                "peak_source": f"{peak_src} bf16_tflops_sustained",
                # ncu dram__bytes_read.sum + dram__bytes_write.sum summed over the 51 gemm_tc launches of one C2 step
                # (profiles/r02_step8_ncu_dram_traffic_c2_summary.json, captured on this workload with the final round-2
                # build: 26.1 GB read + 14.3 GB written; 58.3 GB before the 16-bit residual stream, round 1: 79.3 GB over 61
                # launches).  The kernel is tensor bound; the figure shows there is no re-read waste (the remaining
                # GroupNorm launches: 18.0 GB measured vs 18.4 GB by the kernels' own byte count; whole step 60.4 GB)
                "traffic": (40.36e9 if (B, L) == (4, 128) else None), "traffic_unit": "bytes per step, all conv launches (ncu)",
                "achieved_executed": executed_tf, "frac_executed": executed_tf / peak_tf,
                # The sustained figure is cuBLAS running back to back at the power cap; in this step the convs alternate with
                # HBM-bound kernels that draw less, so the cap lets them clock higher and the fractions above can pass 1.
                # Against the burst figure (a GEMM timed alone) the executed-FLOP rate is:
                "peak_burst": _burst_peak(), "frac_executed_vs_burst": executed_tf / _burst_peak(),
                "note": "achieved = algorithmic conv FLOPs (SURVEY 8d) / summed conv launch time of one step; "
                        "achieved_executed discounts the 5/9 of the upsample convs' FLOPs that phase decomposition removes",
                "step_breakdown_ms": {"conv": conv_ms, "groupnorm_silu": gn_ms, "attention": attn_ms, "epilogue": epi_ms},
                # GroupNorm + SiLU (HBM bound).  bytes_moved = what the kernels actually read + write (conv1 outputs and, since
                # the 16-bit residual stream, x too are 16-bit: 4 B per element; HDRVAE_X16=0: half of the layers 6 B); gbs_vs_6B = the same time charged with
                # the 6 B / element of an fp32-in / 16-bit-out pass over every layer (round-1 definition); SURVEY 8d's
                # algorithmic minimum is 4 B / element
                "groupnorm": {"ms": gn_ms, "elements": 1837.1e6 * B, "bytes_moved": gn_bytes,
                              "gbs_moved": (gn_bytes / (gn_ms / 1e3) / 1e9) if gn_ms > 0 else None,
                              "frac_of_hbm_peak": (gn_bytes / (gn_ms / 1e3) / 1e9 / peak_gbs) if gn_ms > 0 else None,
                              "gbs_vs_6B": (1837.1e6 * B * 6.0 / (gn_ms / 1e3) / 1e9) if gn_ms > 0 else None,
                              "gbs_vs_4B_minimum": (1837.1e6 * B * 4.0 / (gn_ms / 1e3) / 1e9) if gn_ms > 0 else None},
                "attention_fused_kernel": ({"ms": attn_kernel_ms,
                                            "tflops_effective": 4.0 * B * (L * L) ** 2 * 512 / (attn_kernel_ms / 1e3) / 1e12,
                                            "note": "one launch, O = softmax(QK^T)V for all images; effective = 4*T^2*512 per image "
                                                    "(the kernel executes 1.5x that: S is recomputed for each d_v half)"}
                                           if attn_kernel_ms else None),
                "hbm_peak_gbs": peak_gbs}

    # ---- e2e through the node API with host buffers: same number of steps as the device-timed value
    vae = SyntheticVAE(sd, device=dev, output_device="cpu")
    node = NODE_CLASS_MAPPINGS["HDRVAEDecode"]()
    node.adopt_engine(vae, dev, engine)          # reuse the packed weights (same state dict)
    z_host = synthetic_latent(B, L, L, seed=1234 + rank).pin_memory()
    e2e_steps = args.steps
    for _ in range(2):
        (img,) = node.simple_hdr_decode({"samples": z_host}, vae, hdr_mode=MODE)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        (img,) = node.simple_hdr_decode({"samples": z_host}, vae, hdr_mode=MODE)
        assert img.device.type == "cpu"
    torch.cuda.synchronize(dev)
    dt = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    e2e = {"value": mp_per_rank * world / (float(dt.item()) / e2e_steps), "unit": UNIT,
           "h2d_bytes_per_step": z_host.numel() * 4, "d2h_bytes_per_step": img.numel() * 4, "steps": e2e_steps,
           "note": "node API, pinned host latent in, host IMAGE out (wall clock incl. both copies); N>1: independent per-rank node calls"}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "fp16", "data": "synthetic",
            "config": workload_config(world),
            "precision": "fp16 tensor-core operands (16-bit, same width and rate as the bf16 BASELINE names; bf16 "
                         "misses its 1e-2 parity bar, DESIGN.md), fp32 accumulate, fp32 residual stream",
            "roofline": roofline, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks.summary()}
    del img
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # bounded sample: C1-sized calls (BASELINE configs[0], 1x16x64x64 -> 512^2) with the reference's call structure
        line["cpu_baseline"], _, _ = cpu_reference_run(2, 1, 64)
    if rank == 0 and not args.no_eager:
        engine._workspace = None
        torch.cuda.empty_cache()
        line["torch_eager_gpu"] = torch_eager_gpu(dev, B, L, 1234)
        te = line["torch_eager_gpu"]
        if "bf16_autocast" in te:
            line["speedup_vs_torch_eager_same_gpu"] = {
                "per_gpu_value_mp_s": value / world,
                "vs_bf16_autocast_node_call": (value / world) / te["bf16_autocast"]["node_call_mp_s"],
                "vs_bf16_autocast_one_pass": (value / world) / te["bf16_autocast"]["one_pass_mp_s"],
                "vs_fp32_node_call": (value / world) / te["fp32_tf32_off"]["node_call_mp_s"]}
    if rank == 0 and world == 1 and not args.no_aux:
        # cost of the <= 1e-3 precision mode on the same workload (fp16 hi + lo split operands: 3 MMAs per product)
        try:
            engine._workspace = None
            torch.cuda.empty_cache()
            eng_hi = HdrVaeEngine(sd, dev, precision="high")
            for _ in range(2):
                eng_hi.decode(z_dev, MODE, 1.0, want_stats=False)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(3):
                eng_hi.decode(z_dev, MODE, 1.0, want_stats=False)
            e1.record()
            torch.cuda.synchronize(dev)
            ms_hi = e0.elapsed_time(e1) / 3
            line["precision_high"] = {"ms_per_step": ms_hi, "value": mp_per_rank / (ms_hi / 1e3), "unit": UNIT,
                                      "note": "same C2 workload with precision='high' (image rel-L2 <= 1e-3 vs the fp32 oracle, "
                                              "tests/test_gpu_parity_big.py::test_high_precision_mode_meets_1e3)"}
            eng_hi.close()
            del eng_hi
            torch.cuda.empty_cache()
        except Exception as exc:
            line["precision_high"] = {"error": repr(exc)[:200]}
    if world == 1 and not args.no_aux:
        # BASELINE.json quotes the metric at 1024^2 AND 4096^2: config C4 (1x16x512x512 -> 4096^2, "aggressive") on this
        # one GPU, outside the timed region of the headline value
        try:
            engine._workspace = None
            torch.cuda.empty_cache()
            z4 = synthetic_latent(1, 512, 512, seed=1234).to(dev)
            engine.decode(z4, "aggressive", want_stats=False)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(2):
                out4, _ = engine.decode(z4, "aggressive", want_stats=False)
            e1.record()
            torch.cuda.synchronize(dev)
            ms4 = e0.elapsed_time(e1) / 2
            line["aux_c4_4096"] = {"workload": "C4 on one GPU: 1x16x512x512 latent -> 4096x4096, aggressive (not row-tiled)",
                                   "ms_per_image": ms4, "value": 16.777216 / (ms4 / 1e3), "unit": UNIT,
                                   "roofline_frac": 16.777216 / (ms4 / 1e3) / C4_ROOFLINE_MP_S,
                                   "finite": bool(torch.isfinite(out4).all())}
            del out4, z4
        except Exception as exc:      # never lose the headline line to the auxiliary measurement
            line["aux_c4_4096"] = {"error": repr(exc)[:200]}
    if world > 1:
        line["multi_gpu_selftest"] = multi_gpu_selftest(engine, dev, rank, world)
    if world > 1 and not args.no_aux:
        line["aux_c4_rows"] = aux_c4_rows(engine, dev, rank, world, args)
    if rank == 0:
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def multi_gpu_selftest(engine, dev, rank: int, world: int) -> dict:
    """Real-NCCL parity checks run inside the driver's multi-GPU step (the pytest box has one GPU): every rank compares
    what the sharded paths gave it with its OWN single-GPU decode of the same input; the worst difference over ranks is
    reported.  (a) ragged batch sharding (world + 1 images: the first rank gets two), (b) a batch of ONE image over all
    ranks (every rank but the first holds an empty shard), (c) row tiling of one image with 16 latent rows per rank
    (conv tiles coincide with the single-GPU tiling, so the result must be identical), over NCCL and over the device-driven
    transport (sharding.RowsDirect)."""
    import torch
    import torch.distributed as dist
    from vae_decode_hdr_b200.sharding import RowsDirect, decode_batch_sharded, decode_rows_sharded, shard_bounds
    from vae_decode_hdr_b200.synthetic import synthetic_latent
    res = {}
    try:
        def worst(x: float) -> float:
            t = torch.tensor([x], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())

        def rel(a, b):
            return float((a.double() - b.double()).norm() / b.double().norm()) if b.numel() else 0.0
        zb = synthetic_latent(world + 1, 8, 8, seed=5).to(dev)
        s, e = shard_bounds(world + 1, world)[rank]
        out, st = decode_batch_sharded(engine, zb[s:e], "adaptive_recovery", 1.0)
        whole, st1 = engine.decode(zb, "adaptive_recovery", 1.0)
        res["batch_ragged_rel"] = worst(rel(out, whole[s:e]))
        res["batch_stats_rel"] = worst(max(abs(st[k] - st1[k]) / max(1.0, abs(st1[k])) for k in ("pre_min", "pre_max", "pre_mean", "rec_max", "aligned_max")))
        z1 = synthetic_latent(1, 8, 8, seed=6).to(dev)
        s, e = shard_bounds(1, world)[rank]
        out, _ = decode_batch_sharded(engine, z1[s:e], "exposure", 1.0)
        whole, _ = engine.decode(z1, "exposure", 1.0)
        res["batch_empty_shards_rel"] = worst(rel(out, whole[s:e]) if tuple(out.shape) == (e - s, 64, 64, 3) else 1.0)
        zr = synthetic_latent(1, 16 * world, 8, seed=9).to(dev)
        out, _ = decode_rows_sharded(engine, zr, "moderate", 1.0)
        whole, _ = engine.decode(zr, "moderate", 1.0)
        rows = 8 * 16
        res["rows_tiled_rel"] = worst(rel(out, whole[:, rank * rows:(rank + 1) * rows]))
        direct = RowsDirect(engine, 16 * world, 8)                       # device-driven transport, three decodes back to back
        d = 0.0
        for _ in range(3):
            out, _ = direct.decode(zr, "moderate", 1.0)
            d = max(d, rel(out, whole[:, rank * rows:(rank + 1) * rows]))
        direct.close()
        res["rows_tiled_direct_rel"] = worst(d)
        res["pass"] = bool(res["batch_ragged_rel"] < 1e-6 and res["batch_stats_rel"] < 1e-6 and
                           res["batch_empty_shards_rel"] < 1e-6 and res["rows_tiled_rel"] < 1e-6 and
                           res["rows_tiled_direct_rel"] < 1e-6)
    except Exception as exc:
        res["error"] = repr(exc)[:300]
        res["pass"] = False
    return res


def aux_c4_rows(engine, dev, rank: int, world: int, args) -> dict:
    """BASELINE config C4 under the driver's eyes: ONE 1x16x512x512 latent -> 4096x4096, "aggressive", spatially
    row-tiled over the N GPUs of this job (conv halos over NVLink, GroupNorm sums all-reduced, attention K/V
    all-gathered; sharding.decode_rows_sharded) — strong scaling.  Device-timed, max over ranks; the tiled image is
    compared with the single-GPU decode of the same latent on rank 0."""
    import torch
    import torch.distributed as dist
    from vae_decode_hdr_b200.sharding import RowsDirect, decode_rows_sharded
    from vae_decode_hdr_b200.synthetic import synthetic_latent
    L4 = int(os.environ.get("HDRVAE_BENCH_C4_LATENT", "512"))
    res = {"workload": f"C4: 1x16x{L4}x{L4} latent -> {8 * L4}x{8 * L4}, aggressive, row-tiled over {world} GPUs "
                       f"({L4 // world} latent rows per GPU)", "n_gpus": world,
           "transport": "direct (library-owned IPC workspaces; push / wait kernels over NVLink, no NCCL on the data path)"}
    try:
        engine._workspace = None
        torch.cuda.empty_cache()
        z4 = synthetic_latent(1, L4, L4, seed=1234).to(dev)
        reps = 3

        def timed(run):
            for _ in range(2):
                out, _ = run()
            torch.cuda.synchronize(dev); dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                out, _ = run()
            e1.record()
            torch.cuda.synchronize(dev); dist.barrier()
            t = torch.tensor([e0.elapsed_time(e1) / reps], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item()), out

        # host-driven NCCL transport first (its workspace is a torch tensor, freed afterwards)
        ms_nccl, out_nccl = timed(lambda: decode_rows_sharded(engine, z4, "aggressive", 1.0, want_stats=False))
        torch.cuda.empty_cache()
        direct = RowsDirect(engine, L4, L4)
        ms, out = timed(lambda: direct.decode(z4, "aggressive", 1.0, want_stats=False))
        res["nccl_transport_ms_per_image"] = ms_nccl
        res["rel_l2_direct_vs_nccl_transport"] = float((out.double() - out_nccl.double()).norm() / out_nccl.double().norm())
        del out_nccl
        mp = (8 * L4) ** 2 / 1e6
        res.update({"ms_per_image": ms, "value": mp / (ms / 1e3), "unit": UNIT, "scaling": "strong",
                    "per_gpu_mp_s": mp / (ms / 1e3) / world,
                    "per_gpu_roofline_frac": mp / (ms / 1e3) / world / C4_ROOFLINE_MP_S,
                    "roofline_mp_s_per_gpu": C4_ROOFLINE_MP_S})
        parts = [torch.empty_like(out) for _ in range(world)] if rank == 0 else None
        dist.gather(out.contiguous(), parts, dst=0)
        del out
        if rank == 0:
            tiled = torch.cat(parts, dim=1)
            del parts
            torch.cuda.empty_cache()
            whole, _ = engine.decode(z4, "aggressive", 1.0, want_stats=False)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            whole, _ = engine.decode(z4, "aggressive", 1.0, want_stats=False)
            e1.record()
            torch.cuda.synchronize(dev)
            res["single_gpu_ms"] = e0.elapsed_time(e1)
            res["speedup_vs_single_gpu"] = res["single_gpu_ms"] / ms
            d = n = 0.0
            for r0 in range(0, whole.shape[1], 256):       # chunked: fp64 copies of a 4096^2 image are large
                wch, tch = whole[:, r0:r0 + 256].double(), tiled[:, r0:r0 + 256].double()
                d += float(((wch - tch) ** 2).sum()); n += float((wch ** 2).sum())
            res["rel_l2_vs_single_gpu"] = (d / n) ** 0.5
            del whole, tiled
        direct.close()
        engine._workspace = None
        torch.cuda.empty_cache()
        dist.barrier()
    except Exception as exc:
        res["error"] = repr(exc)[:300]
    return res


if __name__ == "__main__":
    main()
