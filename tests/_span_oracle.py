"""fp32 restatement of SPAN (Swift Parameter-free Attention Network, hongyuanyu/SPAN) as spandrel builds it (architecture
name "SPAN") — TEST INFRASTRUCTURE ONLY (tests and tools/span_bench.py).  Parity unpinned: spandrel and the SPAN source
are not installed; restated from the published architecture.  The tiling, hook and recombination around the model are
oracle/upscaler_oracle.py's `upscale()`, which takes `descriptor.scale`; "SPAN" gets the logit reversal there.

The points a reviewer with spandrel's source can check line by line:
  * keys / detection: conv_1.sk.weight is [nf, in_ch, 1, 1] (nf and in_ch); the optional buffer `no_norm` switches the
    input normalisation off; block_1 .. block_6 each hold c1_r, c2_r, c3_r; then conv_2, conv_cat.{weight [nf, 4 nf, 1, 1],
    bias} and upsampler.0.{weight [3 s^2, nf, 3, 3], bias}; s = sqrt(rows / 3).
  * Conv3XC (conv_1, every c*_r, conv_2): sk (1x1, cin -> cout), conv.0 (1x1, cin -> g cin), conv.1 (3x3, pad 0,
    g cin -> g cout), conv.2 (1x1, g cout -> cout), eval_conv (3x3, pad 1); g = gain1 = 2.  In eval mode `forward` calls
    `update_params()` on EVERY call, which rebuilds eval_conv from conv.* and sk (W = w3 . w2 . w1 plus sk at the centre
    tap; b = w3 (sum w2 b1 + b2) + b3 + b_sk), then runs eval_conv(x) with zero padding 1.  No activation (relu=False).
    Training form: conv(pad(x, 1)) + sk(x).
  * SPAB: out1 = act1(c1_r(x)) with act1 = SiLU(inplace=True), so the returned out1 is the ACTIVATED tensor;
    out2 = act1(c2_r(out1)); out3 = c3_r(out2); att = sigmoid(out3) - 0.5; out = (out3 + x) att; returns (out, out1, att).
    act2 exists and is never called.
  * SPAN forward: if norm, x = (x - mean) 255 with mean (0.4488, 0.4371, 0.4040); f = conv_1(x); b1 .. b5 through blocks
    1-5; (b6, b5_2, _) = block_6(b5); b6 = conv_2(b6); out = conv_cat(cat[f, b6, b1, b5_2]); y = pixel_shuffle(
    upsampler.0(out), s).  No de-normalisation, no base / skip add at the end."""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F


class Conv3XC(nn.Module):
    def __init__(self, c_in, c_out, gain1=2):
        super().__init__()
        self.sk = nn.Conv2d(c_in, c_out, 1, padding=0, bias=True)
        self.conv = nn.Sequential(
            nn.Conv2d(c_in, c_in * gain1, 1, padding=0, bias=True),
            nn.Conv2d(c_in * gain1, c_out * gain1, 3, padding=0, bias=True),
            nn.Conv2d(c_out * gain1, c_out, 1, padding=0, bias=True),
        )
        self.eval_conv = nn.Conv2d(c_in, c_out, 3, padding=1, bias=True)
        self.eval_conv.weight.requires_grad = False
        self.eval_conv.bias.requires_grad = False
        self.update_params()

    def update_params(self):
        w1, b1 = self.conv[0].weight.data.clone().detach(), self.conv[0].bias.data.clone().detach()
        w2, b2 = self.conv[1].weight.data.clone().detach(), self.conv[1].bias.data.clone().detach()
        w3, b3 = self.conv[2].weight.data.clone().detach(), self.conv[2].bias.data.clone().detach()
        w = F.conv2d(w1.flip(2, 3).permute(1, 0, 2, 3), w2, padding=2, stride=1).flip(2, 3).permute(1, 0, 2, 3)
        b = (w2 * b1.reshape(1, -1, 1, 1)).sum((1, 2, 3)) + b2
        weight = F.conv2d(w.flip(2, 3).permute(1, 0, 2, 3), w3, padding=0, stride=1).flip(2, 3).permute(1, 0, 2, 3)
        bias = (w3 * b.reshape(1, -1, 1, 1)).sum((1, 2, 3)) + b3
        sk_w = F.pad(self.sk.weight.data.clone().detach(), [1, 1, 1, 1])
        self.eval_conv.weight.data = weight + sk_w
        self.eval_conv.bias.data = bias + self.sk.bias.data.clone().detach()

    def forward(self, x):
        if self.training:
            return self.conv(F.pad(x, (1, 1, 1, 1), "constant", 0)) + self.sk(x)
        self.update_params()
        return self.eval_conv(x)


class SPAB(nn.Module):
    def __init__(self, nf):
        super().__init__()
        self.c1_r = Conv3XC(nf, nf)
        self.c2_r = Conv3XC(nf, nf)
        self.c3_r = Conv3XC(nf, nf)
        self.act1 = nn.SiLU(inplace=True)
        self.act2 = nn.LeakyReLU(0.1, inplace=True)       # never called

    def forward(self, x):
        out1 = self.c1_r(x)
        out1_act = self.act1(out1)                          # in place: out1 IS the activated tensor
        out2 = self.c2_r(out1_act)
        out2_act = self.act1(out2)
        out3 = self.c3_r(out2_act)
        sim_att = torch.sigmoid(out3) - 0.5
        out = (out3 + x) * sim_att
        return out, out1, sim_att


class SPAN(nn.Module):
    def __init__(self, nf=48, scale=4, in_ch=3, out_ch=3, norm=True):
        super().__init__()
        self.nf, self.scale = nf, scale
        self.mean = torch.tensor((0.4488, 0.4371, 0.4040)).view(1, 3, 1, 1)
        if not norm:
            self.register_buffer("no_norm", torch.zeros(1))
        else:
            self.no_norm = None
        self.conv_1 = Conv3XC(in_ch, nf)
        for k in range(1, 7):
            setattr(self, f"block_{k}", SPAB(nf))
        self.conv_cat = nn.Conv2d(nf * 4, nf, 1, padding=0, bias=True)
        self.conv_2 = Conv3XC(nf, nf)
        self.upsampler = nn.Sequential(nn.Conv2d(nf, out_ch * scale * scale, 3, padding=1), nn.PixelShuffle(scale))

    @property
    def is_norm(self):
        return self.no_norm is None

    def forward(self, x):
        if self.is_norm:
            x = (x - self.mean.type_as(x)) * 255.0
        out_feature = self.conv_1(x)
        out_b1, _, _ = self.block_1(out_feature)
        out_b2, _, _ = self.block_2(out_b1)
        out_b3, _, _ = self.block_3(out_b2)
        out_b4, _, _ = self.block_4(out_b3)
        out_b5, _, _ = self.block_5(out_b4)
        out_b6, out_b5_2, _ = self.block_6(out_b5)
        out_b6 = self.conv_2(out_b6)
        out = self.conv_cat(torch.cat([out_feature, out_b6, out_b1, out_b5_2], 1))
        return self.upsampler(out)


def build_span(seed: int = 0, nf: int = 48, s: int = 4, norm: bool = True, gain: float = 1.0) -> SPAN:
    """Random-init SPAN under `seed` in eval mode.  PyTorch's default init makes every Conv3XC nearly a zero map (three
    products of ~1/sqrt(fan_in) factors), so that after six gated blocks the output would be the biases; the convs are
    drawn from N(0, 1 / fan_in) instead, the Conv3XC chains rescaled to unit gain and biases kept small
    (tests/test_upscaler_span_cpu.py checks that the output depends on the input).  `gain` scales upsampler.0."""
    torch.manual_seed(seed)
    net = SPAN(nf=nf, scale=s, norm=norm).eval()
    with torch.no_grad():
        for m in net.modules():
            if isinstance(m, nn.Conv2d):
                fan_in = m.weight.shape[1] * m.weight.shape[2] * m.weight.shape[3]
                m.weight.normal_(0.0, (1.0 / fan_in) ** 0.5)
                m.bias.uniform_(-0.05, 0.05)
        if norm:
            net.conv_1.sk.weight.mul_(1.0 / 255)             # keeps conv_1's gain near 1 on the x 255 input
            net.conv_1.conv[0].weight.mul_(1.0 / 255)
        if gain != 1.0:
            net.upsampler[0].weight.mul_(gain)
            net.upsampler[0].bias.mul_(gain)
        for m in net.modules():
            if isinstance(m, Conv3XC):
                m.update_params()
    for p in net.parameters():
        p.requires_grad_(False)
    return net


def stale_eval_conv(net: SPAN, seed: int = 99) -> dict:
    """The state dict of `net` with every Conv3XC's eval_conv.* overwritten by garbage (what a checkpoint saved between
    optimiser steps holds): a loader must fuse conv.* and sk itself."""
    g = torch.Generator().manual_seed(seed)
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    for k in sd:
        if ".eval_conv." in k:
            sd[k] = torch.randn(sd[k].shape, generator=g) * 100.0
    return sd
