"""Attention core alone (hdrvae_attention: q, k, v 16-bit [B, T, 512]): device time of the whole test entry (which also
allocates its workspace and transposes / interleaves the operands) and of the fused kernel itself (library profile
scope).  python tools/attn_bench.py [BxT ...]"""
import os
import sys
import tempfile
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from vae_decode_hdr_b200.engine import HdrVaeEngine  # noqa: E402
from vae_decode_hdr_b200.synthetic import random_decoder_state_dict  # noqa: E402

dev = torch.device("cuda:0")
eng = HdrVaeEngine(random_decoder_state_dict(0), dev)
cases = [(4, 4096), (4, 16384), (1, 65536), (1, 262144)]
if len(sys.argv) > 1:
    cases = [(int(a.split("x")[0]), int(a.split("x")[1])) for a in sys.argv[1:]]
for B, T in cases:
    g = torch.Generator(device=dev).manual_seed(T)
    q = (torch.randn(B, T, 512, generator=g, device=dev) * 2).half()
    k = torch.randn(B, T, 512, generator=g, device=dev).half()
    v = torch.randn(B, T, 512, generator=g, device=dev).half()
    o = eng.attention(q, k, v)
    torch.cuda.synchronize()
    reps = 3 if T >= 65536 else 10
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        o = eng.attention(q, k, v)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    tf = 4.0 * B * T * T * 512 / (ms / 1e3) / 1e12
    kern = ""
    path = os.path.join(tempfile.gettempdir(), "attn_prof.tsv")
    eng.lib.hdrvae_profile_begin()
    eng.attention(q, k, v)
    eng.lib.hdrvae_profile_end(path.encode())
    for ln in open(path):
        if ln.startswith("attention fused kernel"):
            kms = float(ln.split("\t")[1].split()[0])
            kern = f"  kernel alone {kms:.3f} ms = {4.0 * B * T * T * 512 / (kms / 1e3) / 1e12:.1f} TFLOP/s"
    print(f"B={B} T={T}: entry {ms:.3f} ms  {tf:.1f} TFLOP/s effective{kern}", flush=True)
