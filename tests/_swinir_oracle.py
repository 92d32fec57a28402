"""fp32 SwinIR in spandrel's key names: the oracle of the library's SwinIR forward (tests/test_gpu_upscaler_swinir.py).

A restatement of JingyunLiang/SwinIR models/network_swinir.py as spandrel loads it ("SwinIR"), to be checked line by line
against that source; spandrel is not installed here, so parity with it is unpinned.  The Swin transformer layer is pinned
against torchvision's independent SwinTransformerBlock (tests/test_upscaler_swinir_cpu.py).  Architecture points:
  1. forward: x is reflect-padded at the bottom / right to a multiple of the window (check_image_size), then
     x = (x - mean) * img_range with mean = (0.4488, 0.4371, 0.4040) and img_range 1, and at the end x / img_range + mean,
     cropped to (s H, s W).
  2. conv_first 3x3, 3 -> C.  patch_embed: flatten to tokens (B, HW, C) + LayerNorm when patch_norm; no ape.
  3. RSTB i: the Swin transformer layers blocks.0 .. of layers.i.residual_group, then conv(patch_unembed(x)) + x (the RSTB
     input), re-flattened without a norm.  resi_connection "1conv": one 3x3 conv C -> C; "3conv": conv.0 3x3 C -> C/4,
     LeakyReLU 0.2, conv.2 1x1 C/4 -> C/4, LeakyReLU 0.2, conv.4 3x3 C/4 -> C.
  4. Swin transformer layer j: shift = 0 for even j, ws / 2 = 4 for odd j.  x + attn(norm1(x)) then x + mlp(norm2(x)),
     LayerNorm eps 1e-5, mlp = fc1, GELU (erf), fc2.
  5. attention on the image rolled by (-shift, -shift), 8 x 8 windows: qkv Linear C -> 3C split as (3, heads, hd), q * hd^-0.5,
     q k^T + relative_position_bias_table[index][:, :, h] with index (ri - rj + 7) * 15 + (ci - cj + 7), + calculate_mask of
     the padded size when shifting (regions of slices (0, -ws), (-ws, -shift), (-shift, None) per axis, -100 across
     regions), softmax, @ v, heads concatenated, proj; windows reversed and rolled back by (+shift, +shift).
  6. after the last RSTB: norm (LayerNorm), patch_unembed, conv_after_body (1conv / 3conv as in 3) + conv_first's output.
  7. upsampler "pixelshuffle": conv_before_upsample.0 3x3 C -> 64 + LeakyReLU (default slope 0.01), upsample.{2k} 3x3
     64 -> 256 + PixelShuffle(2) per 2x stage, conv_last 3x3 64 -> 3.  "pixelshuffledirect": upsample.0 3x3 C -> 3 s^2 +
     PixelShuffle(s).  "nearest+conv": conv_before_upsample.0 (+ LeakyReLU 0.01), conv_up1 (and conv_up2 at 4x) on the
     nearest-2x upsampled tensor with LeakyReLU 0.2, conv_hr + LeakyReLU 0.2, conv_last.  "": x + conv_last(res) with x
     the normalised input, conv_last 3x3 C -> 3.
  8. stored buffers relative_position_index and attn_mask are loaded (strict) but the forward recomputes both."""
import math

import torch
import torch.nn as nn
import torch.nn.functional as F

WS = 8
MEAN = (0.4488, 0.4371, 0.4040)


def region_mask(H, W, shift, ws=WS):
    """calculate_mask of network_swinir.py for an H x W (padded) image: [nW, ws^2, ws^2] with 0 / -100."""
    img = torch.zeros(H, W)
    cnt = 0
    for hs in (slice(0, -ws), slice(-ws, -shift), slice(-shift, None)):
        for wsl in (slice(0, -ws), slice(-ws, -shift), slice(-shift, None)):
            img[hs, wsl] = cnt
            cnt += 1
    win = img.view(H // ws, ws, W // ws, ws).permute(0, 2, 1, 3).reshape(-1, ws * ws)
    m = win[:, None, :] - win[:, :, None]
    return m.masked_fill(m != 0, -100.0).masked_fill(m == 0, 0.0)


def rel_index(ws=WS):
    r = torch.arange(ws * ws)
    return ((r[:, None] // ws - r[None, :] // ws) + ws - 1) * (2 * ws - 1) + (r[:, None] % ws - r[None, :] % ws) + ws - 1


class WindowAttention(nn.Module):
    def __init__(self, dim, heads):
        super().__init__()
        self.heads = heads
        self.relative_position_bias_table = nn.Parameter(torch.zeros((2 * WS - 1) ** 2, heads))
        self.register_buffer("relative_position_index", rel_index())
        self.qkv = nn.Linear(dim, 3 * dim)
        self.proj = nn.Linear(dim, dim)

    def forward(self, x, mask=None):
        B_, N, C = x.shape
        hd = C // self.heads
        qkv = self.qkv(x).reshape(B_, N, 3, self.heads, hd).permute(2, 0, 3, 1, 4)
        q, k, v = qkv[0] * hd ** -0.5, qkv[1], qkv[2]
        attn = q @ k.transpose(-2, -1)
        bias = self.relative_position_bias_table[rel_index().view(-1).to(x.device)].view(N, N, -1).permute(2, 0, 1)
        attn = attn + bias.unsqueeze(0)
        if mask is not None:
            nW = mask.shape[0]
            attn = attn.view(B_ // nW, nW, self.heads, N, N) + mask.unsqueeze(1).unsqueeze(0)
            attn = attn.view(-1, self.heads, N, N)
        attn = attn.softmax(-1)
        return self.proj((attn @ v).transpose(1, 2).reshape(B_, N, C))


class SwinLayer(nn.Module):
    """One Swin transformer layer (network_swinir.py SwinTransformerBlock) on tokens [B, H W, C] of an H x W image."""

    def __init__(self, dim, heads, hidden, shift, img_size=64):
        super().__init__()
        self.shift = shift
        self.norm1 = nn.LayerNorm(dim)
        self.attn = WindowAttention(dim, heads)
        self.norm2 = nn.LayerNorm(dim)
        self.mlp = nn.Module()
        self.mlp.fc1 = nn.Linear(dim, hidden)
        self.mlp.act = nn.GELU()
        self.mlp.fc2 = nn.Linear(hidden, dim)
        if shift:
            self.register_buffer("attn_mask", region_mask(img_size, img_size, shift))
        else:
            self.attn_mask = None

    def forward(self, x, H, W):
        B, L, C = x.shape
        s = self.shift
        h = self.norm1(x).view(B, H, W, C)
        if s:
            h = torch.roll(h, shifts=(-s, -s), dims=(1, 2))
        win = h.view(B, H // WS, WS, W // WS, WS, C).permute(0, 1, 3, 2, 4, 5).reshape(-1, WS * WS, C)
        a = self.attn(win, region_mask(H, W, s).to(x) if s else None)
        h = a.view(B, H // WS, W // WS, WS, WS, C).permute(0, 1, 3, 2, 4, 5).reshape(B, H, W, C)
        if s:
            h = torch.roll(h, shifts=(s, s), dims=(1, 2))
        x = x + h.reshape(B, L, C)
        return x + self.mlp.fc2(self.mlp.act(self.mlp.fc1(self.norm2(x))))


def _resi(dim, kind):
    if kind == "1conv":
        return nn.Conv2d(dim, dim, 3, 1, 1)
    return nn.Sequential(nn.Conv2d(dim, dim // 4, 3, 1, 1), nn.LeakyReLU(0.2), nn.Conv2d(dim // 4, dim // 4, 1),
                         nn.LeakyReLU(0.2), nn.Conv2d(dim // 4, dim, 3, 1, 1))


class RSTB(nn.Module):
    def __init__(self, dim, depth, heads, hidden, resi, img_size):
        super().__init__()
        self.residual_group = nn.Module()
        self.residual_group.blocks = nn.ModuleList(
            [SwinLayer(dim, heads, hidden, 0 if j % 2 == 0 else WS // 2, img_size) for j in range(depth)])
        self.conv = _resi(dim, resi)

    def forward(self, x, H, W):
        y = x
        for b in self.residual_group.blocks:
            y = b(y, H, W)
        B, L, C = y.shape
        y = self.conv(y.transpose(1, 2).reshape(B, C, H, W))
        return y.flatten(2).transpose(1, 2) + x


class SwinIR(nn.Module):
    def __init__(self, embed_dim=180, depths=(6, 6, 6, 6, 6, 6), heads=6, mlp_ratio=2.0, upsampler="pixelshuffle", s=4,
                 resi_connection="1conv", patch_norm=True, img_size=64):
        super().__init__()
        C = embed_dim
        self.upsampler, self.s, self.patch_norm = upsampler, s, patch_norm
        self.register_buffer("mean", torch.tensor(MEAN).view(1, 3, 1, 1), persistent=False)
        self.conv_first = nn.Conv2d(3, C, 3, 1, 1)
        self.patch_embed = nn.Module()
        if patch_norm:
            self.patch_embed.norm = nn.LayerNorm(C)
        hidden = int(C * mlp_ratio)
        self.layers = nn.ModuleList([RSTB(C, d, heads, hidden, resi_connection, img_size) for d in depths])
        self.norm = nn.LayerNorm(C)
        self.conv_after_body = _resi(C, resi_connection)
        if upsampler in ("pixelshuffle", "nearest+conv"):
            self.conv_before_upsample = nn.Sequential(nn.Conv2d(C, 64, 3, 1, 1), nn.LeakyReLU())
        if upsampler == "pixelshuffle":
            mods = []
            for _ in range(int(math.log2(s))):
                mods += [nn.Conv2d(64, 256, 3, 1, 1), nn.PixelShuffle(2)]
            self.upsample = nn.Sequential(*mods)
            self.conv_last = nn.Conv2d(64, 3, 3, 1, 1)
        elif upsampler == "pixelshuffledirect":
            self.upsample = nn.Sequential(nn.Conv2d(C, 3 * s * s, 3, 1, 1), nn.PixelShuffle(s))
        elif upsampler == "nearest+conv":
            self.conv_up1 = nn.Conv2d(64, 64, 3, 1, 1)
            if s == 4:
                self.conv_up2 = nn.Conv2d(64, 64, 3, 1, 1)
            self.conv_hr = nn.Conv2d(64, 64, 3, 1, 1)
            self.conv_last = nn.Conv2d(64, 3, 3, 1, 1)
        else:
            self.conv_last = nn.Conv2d(C, 3, 3, 1, 1)

    def features(self, x):
        B, C, H, W = x.shape
        t = x.flatten(2).transpose(1, 2)
        if self.patch_norm:
            t = self.patch_embed.norm(t)
        for layer in self.layers:
            t = layer(t, H, W)
        return self.norm(t).transpose(1, 2).reshape(B, C, H, W)

    def forward(self, x):
        H, W = x.shape[2:]
        ph, pw = (WS - H % WS) % WS, (WS - W % WS) % WS
        x = F.pad(x, (0, pw, 0, ph), "reflect")
        x = x - self.mean
        lrelu = nn.LeakyReLU(0.2)
        if self.upsampler == "pixelshuffle":
            x = self.conv_first(x)
            x = self.conv_after_body(self.features(x)) + x
            x = self.conv_last(self.upsample(self.conv_before_upsample(x)))
        elif self.upsampler == "pixelshuffledirect":
            x = self.conv_first(x)
            x = self.upsample(self.conv_after_body(self.features(x)) + x)
        elif self.upsampler == "nearest+conv":
            x = self.conv_first(x)
            x = self.conv_before_upsample(self.conv_after_body(self.features(x)) + x)
            x = lrelu(self.conv_up1(F.interpolate(x, scale_factor=2, mode="nearest")))
            if self.s == 4:
                x = lrelu(self.conv_up2(F.interpolate(x, scale_factor=2, mode="nearest")))
            x = self.conv_last(lrelu(self.conv_hr(x)))
        else:
            f = self.conv_first(x)
            x = x + self.conv_last(self.conv_after_body(self.features(f)) + f)
        x = x + self.mean
        return x[:, :, :H * self.s, :W * self.s]


def build_swinir(seed, embed_dim=60, depths=(2, 2), heads=6, mlp_ratio=2.0, upsampler="pixelshuffle", s=4,
                 resi_connection="1conv", patch_norm=True):
    """The oracle network loaded (strict) from synthetic.random_swinir_state_dict with the same arguments."""
    from vae_decode_hdr_b200.synthetic import random_swinir_state_dict
    net = SwinIR(embed_dim, depths, heads, mlp_ratio, upsampler, 1 if upsampler == "" else s, resi_connection, patch_norm)
    net.load_state_dict(random_swinir_state_dict(seed, embed_dim, depths, heads, mlp_ratio, upsampler,
                                                 1 if upsampler == "" else s, resi_connection, patch_norm))
    return net.eval()
