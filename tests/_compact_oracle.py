"""fp32 restatement of Real-ESRGAN's SRVGGNetCompact as spandrel builds it (act_type "prelu"), next to the RRDBNet of
oracle/upscaler_oracle.py — TEST INFRASTRUCTURE ONLY (tests and tools/compact_bench.py).  Parity unpinned: spandrel and
Real-ESRGAN are not installed; restated from their published architecture.  The tiling, hook and recombination around the
model are oracle/upscaler_oracle.py's `upscale()`, which already takes `descriptor.scale`."""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F


class SRVGGNetCompact(nn.Module):
    """Real-ESRGAN's SRVGGNetCompact with act_type "prelu" (realesr-general-x4v3: nf 64, nc 32, s 4; realesr-animevideov3:
    nf 64, nc 16, s 4).  `body` holds, in order: conv 3 -> nf, PReLU, nc x (conv nf -> nf, PReLU), conv nf -> 3 s^2 —
    the state-dict keys body.0 / body.{2k+1} (slopes, [nf]) / body.{2+2m} / body.{2nc+2}.  The network output is the
    pixel shuffle of the last conv plus the nearest-upsampled input."""

    def __init__(self, nf=64, nc=32, scale=4, in_ch=3, out_ch=3):
        super().__init__()
        self.nf, self.nc, self.scale = nf, nc, scale
        layers = [nn.Conv2d(in_ch, nf, 3, 1, 1), nn.PReLU(num_parameters=nf)]
        for _ in range(nc):
            layers += [nn.Conv2d(nf, nf, 3, 1, 1), nn.PReLU(num_parameters=nf)]
        layers.append(nn.Conv2d(nf, out_ch * scale * scale, 3, 1, 1))
        self.body = nn.ModuleList(layers)
        self.upsampler = nn.PixelShuffle(scale)

    def forward(self, x):
        out = x
        for layer in self.body:
            out = layer(out)
        return self.upsampler(out) + F.interpolate(x, scale_factor=self.scale, mode="nearest")


def build_compact(seed: int = 0, nf: int = 64, nc: int = 32, s: int = 4, gain: float = 1.0) -> SRVGGNetCompact:
    """Random-init SRVGGNetCompact under `seed`: PyTorch's default conv init, PReLU slopes drawn from U(-0.5, 0.5) per
    channel (the default constant 0.25 would hide a channel-indexing error).  `gain` scales the last conv."""
    torch.manual_seed(seed)
    net = SRVGGNetCompact(nf=nf, nc=nc, scale=s).eval()
    with torch.no_grad():
        for layer in net.body:
            if isinstance(layer, nn.PReLU):
                layer.weight.uniform_(-0.5, 0.5)
        if gain != 1.0:
            net.body[-1].weight.mul_(gain)
            net.body[-1].bias.mul_(gain)
    for p in net.parameters():
        p.requires_grad_(False)
    return net
