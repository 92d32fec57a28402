"""fp32 restatement of every RRDBNet form the upscaler runs -- 0, 1 or 2 upsampling convs, pixel-unshuffle factor 1, 2 or
4 -- as spandrel builds them.  TEST INFRASTRUCTURE ONLY (tests and tools/rrdb_scales_bench.py).  With the defaults
(n_up 2, shuffle 1) it is oracle/upscaler_oracle.py's 4x RRDBNet: same module order, so the same parameters under a seed,
and the same state-dict keys in both layouts (tests/test_upscaler_rrdb_scales_cpu.py checks that).  The tiling, hook and
recombination around the model are oracle/upscaler_oracle.py's `upscale()`, which takes `descriptor.scale`.

Parity unpinned, like the 4x RRDBNet: spandrel is not installed, and this is restated from its published source.  That
includes the pixel-unshuffle form's input rule (spandrel's RRDBNet.forward with a shuffle factor f): reflect-pad the
bottom / right edge of an h x w input by (f - h mod f) mod f rows and (f - w mod f) mod f columns, pixel_unshuffle by f,
run the network, crop the output to its top-left s h x s w.  The rule is exactly as checkable as the RRDBNet itself and
comfy.utils.tiled_scale, which this repository restates the same way: against spandrel's source, not offline.  With the
node's 512-pixel tiles and 64 overlap, tile origins are multiples of 448 and a tile side is 512 or the rest of the image,
so only an image side that is not a multiple of f ever pads a tile."""
from __future__ import annotations

from collections import OrderedDict

import torch
import torch.nn as nn
import torch.nn.functional as F

from oracle.upscaler_oracle import _RRDB


class RRDBNet(nn.Module):
    """ESRGAN generator with `n_up` (nearest 2x, conv, LeakyReLU 0.2) upsampling stages on a pixel-unshuffled input:
    conv_first reads 3 shuffle^2 channels; the scale is 2^n_up / shuffle.  Real-ESRGAN parameter names (conv_up1 ...);
    `old_arch_key` gives the BasicSR / spandrel ones."""

    def __init__(self, nf=64, nb=23, gc=32, in_ch=3, out_ch=3, n_up=2, shuffle=1):
        super().__init__()
        if (1 << n_up) < shuffle:
            raise ValueError(f"scale 2^{n_up} / {shuffle} is below 1")
        self.nf, self.nb, self.gc, self.n_up, self.shuffle = nf, nb, gc, n_up, shuffle
        self.scale = (1 << n_up) // shuffle
        self.conv_first = nn.Conv2d(in_ch * shuffle * shuffle, nf, 3, 1, 1)
        self.body = nn.Sequential(*[_RRDB(nf, gc) for _ in range(nb)])
        self.conv_body = nn.Conv2d(nf, nf, 3, 1, 1)
        for k in range(n_up):
            setattr(self, f"conv_up{k + 1}", nn.Conv2d(nf, nf, 3, 1, 1))
        self.conv_hr = nn.Conv2d(nf, nf, 3, 1, 1)
        self.conv_last = nn.Conv2d(nf, out_ch, 3, 1, 1)

    def forward(self, x):
        h, w = x.shape[-2:]
        f = self.shuffle
        if f > 1:
            x = F.pad(x, (0, (f - w % f) % f, 0, (f - h % f) % f), "reflect")
            x = F.pixel_unshuffle(x, f)
        feat = self.conv_first(x)
        feat = feat + self.conv_body(self.body(feat))
        for k in range(self.n_up):
            feat = F.leaky_relu(getattr(self, f"conv_up{k + 1}")(F.interpolate(feat, scale_factor=2, mode="nearest")), 0.2)
        out = self.conv_last(F.leaky_relu(self.conv_hr(feat), 0.2))
        return out[..., :self.scale * h, :self.scale * w]


def old_arch_key(key: str, nb: int = 23, n_up: int = 2) -> str:
    """Real-ESRGAN name -> the `model.N...` name spandrel's ESRGAN module uses for the same tensor.  BasicSR's
    sequential() flattens each upsampling stage into (Upsample, conv, LeakyReLU) and conv_hr into (conv, LeakyReLU)."""
    head, _, leaf = key.rpartition(".")
    table = {"conv_first": "model.0", "conv_body": f"model.1.sub.{nb}", "conv_hr": f"model.{3 * n_up + 2}",
             "conv_last": f"model.{3 * n_up + 4}"}
    table.update({f"conv_up{k + 1}": f"model.{3 + 3 * k}" for k in range(n_up)})
    if head in table:
        return f"{table[head]}.{leaf}"
    _, i, rdb, conv = head.split(".")                      # body.i.rdbK.convJ
    return f"model.1.sub.{i}.RDB{rdb[-1]}.{conv}.0.{leaf}"


def build_upscaler(seed: int = 0, nb: int = 23, gain: float = 1.0, n_up: int = 2, shuffle: int = 1) -> RRDBNet:
    """Random-init RRDBNet (PyTorch default init under `seed`).  `gain` scales conv_last."""
    torch.manual_seed(seed)
    net = RRDBNet(nb=nb, n_up=n_up, shuffle=shuffle).eval()
    if gain != 1.0:
        with torch.no_grad():
            net.conv_last.weight.mul_(gain)
            net.conv_last.bias.mul_(gain)
    for p in net.parameters():
        p.requires_grad_(False)
    return net


def state_dict_old_arch(net: RRDBNet) -> "OrderedDict[str, torch.Tensor]":
    return OrderedDict((old_arch_key(k, net.nb, net.n_up), v) for k, v in net.state_dict().items())
