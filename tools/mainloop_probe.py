"""Times decoder-shaped convs with the TMA loads and/or the MMAs switched off: which of the two paces the main loop?
The library reads HDRVAE_GEMM_DBG once per process, so one run measures one setting (tools/gpu_mainloop.sh runs 0..3):
HDRVAE_GEMM_DBG=1 python tools/mainloop_probe.py"""
import os
import sys

import torch

sys.path.insert(0, ".")
from vae_decode_hdr_b200.engine import HdrVaeEngine  # noqa: E402
from vae_decode_hdr_b200.synthetic import random_decoder_state_dict  # noqa: E402

dev = "cuda:0"
dbg = int(os.environ.get("HDRVAE_GEMM_DBG", "0"))
eng = HdrVaeEngine(random_decoder_state_dict(0), dev)
for name, B, H, cin, cout in [("512->512@256", 4, 256, 512, 512), ("128->128@1024", 4, 1024, 128, 128), ("256->256@512", 4, 512, 256, 256)]:
    x = torch.randn(B, H, H, cin, device=dev).half()
    w = torch.randn(cout, cin, 3, 3, device=dev) * 0.02
    b = torch.zeros(cout, device=dev)
    eng.lib.hdrvae_profile_begin()
    for _ in range(3):
        eng.conv2d(x, w, b, 3, out_dtype=torch.float32)
    path = f"/tmp/probe_{dbg}.tsv"
    eng.lib.hdrvae_profile_end(path.encode())
    ms = [float(l.split("\t")[1].split()[0]) for l in open(path) if l.startswith("conv")]
    fl = 2.0 * B * H * H * cin * cout * 9
    print(f"{name:16s} dbg={dbg} ({'no TMA ' if dbg & 1 else 'TMA    '}{'no MMA' if dbg & 2 else 'MMA   '}): {min(ms):8.3f} ms  {fl / min(ms) / 1e9:8.1f} TFLOP/s-equivalent")
    del x
