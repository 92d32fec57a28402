"""Synthetic stand-ins for what ComfyUI hands the node: a random-init Flux AE decoder state dict and
a minimal VAE object exposing the attributes the node reads (vae.first_stage_model.decoder,
vae.device, vae.output_device).  Used by bench.py and __graft_entry__.smoke(); there is no network
for real checkpoints (BASELINE.json: "random-init Flux AE weights and synthetic latents")."""
from __future__ import annotations

import math
from typing import Dict, Iterator, List, Optional, Tuple

import torch

CH, CH_MULT, Z = 128, (1, 2, 4, 4), 16


def decoder_param_shapes(z_channels: int = Z) -> List[Tuple[str, Tuple[int, ...]]]:
    """State-dict keys/shapes of the Flux.1 AE decoder (BFL / ComfyUI naming; SURVEY.md §8b); z_channels = 4 gives the
    SD1.x / SDXL decoder (same graph, conv_in 4 -> 512)."""
    out: List[Tuple[str, Tuple[int, ...]]] = []

    def conv(name, cout, cin, k):
        out.append((f"{name}.weight", (cout, cin, k, k)))
        out.append((f"{name}.bias", (cout,)))

    def norm(name, c):
        out.append((f"{name}.weight", (c,)))
        out.append((f"{name}.bias", (c,)))

    def res(name, cin, cout):
        norm(f"{name}.norm1", cin); conv(f"{name}.conv1", cout, cin, 3)
        norm(f"{name}.norm2", cout); conv(f"{name}.conv2", cout, cout, 3)
        if cin != cout:
            conv(f"{name}.nin_shortcut", cout, cin, 1)

    top = CH * CH_MULT[-1]
    conv("conv_in", top, z_channels, 3)
    res("mid.block_1", top, top)
    norm("mid.attn_1.norm", top)
    for n in ("q", "k", "v", "proj_out"):
        conv(f"mid.attn_1.{n}", top, top, 1)
    res("mid.block_2", top, top)
    cin = top
    for lvl in reversed(range(4)):
        cout = CH * CH_MULT[lvl]
        for i in range(3):
            res(f"up.{lvl}.block.{i}", cin, cout)
            cin = cout
        if lvl != 0:
            conv(f"up.{lvl}.upsample.conv", cin, cin, 3)
    norm("norm_out", cin)
    conv("conv_out", 3, cin, 3)
    return out


def random_decoder_state_dict(seed: int = 0, z_channels: int = Z) -> Dict[str, torch.Tensor]:
    """PyTorch-default-style init (conv weight/bias ~ U(+-1/sqrt(fan_in)), GroupNorm 1/0), fp32, CPU."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    sd: Dict[str, torch.Tensor] = {}
    fan_in = 1
    for name, shape in decoder_param_shapes(z_channels):
        if len(shape) == 4:
            fan_in = shape[1] * shape[2] * shape[3]
            bound = 1.0 / math.sqrt(fan_in)
            sd[name] = (torch.rand(shape, generator=g) * 2 - 1) * bound
        elif ".norm" in name or name.startswith("norm_out"):
            sd[name] = torch.ones(shape) if name.endswith("weight") else torch.zeros(shape)
        else:
            sd[name] = (torch.rand(shape, generator=g) * 2 - 1) / math.sqrt(fan_in)
    return sd


class _DecoderBag(torch.nn.Module):
    """Holds a state dict under the original dotted keys (what the node reads via .state_dict())."""

    def __init__(self, sd: Dict[str, torch.Tensor]):
        super().__init__()
        self._sd = {k: torch.nn.Parameter(v, requires_grad=False) for k, v in sd.items()}

    def state_dict(self, *a, **k):          # noqa: D401
        return {k2: v.data for k2, v in self._sd.items()}

    def parameters(self, recurse: bool = True) -> Iterator[torch.nn.Parameter]:
        return iter(self._sd.values())


class _FirstStage:
    def __init__(self, decoder, post_quant_conv=None):
        self.decoder = decoder
        if post_quant_conv is not None:
            self.post_quant_conv = post_quant_conv


class SyntheticVAE:
    """The attributes of comfy.sd.VAE the node touches; ``output_device`` is where the IMAGE lands
    (ComfyUI: the intermediate device, normally CPU).  ``post_quant_conv``: the 1x1 conv an SD1.x / SDXL first-stage
    model applies to the latent before the decoder (Flux: None)."""

    def __init__(self, state_dict: Dict[str, torch.Tensor], device="cuda", output_device="cpu",
                 post_quant_conv: Optional[torch.nn.Module] = None):
        self.first_stage_model = _FirstStage(_DecoderBag(state_dict), post_quant_conv)
        self.device = torch.device(device)
        self.output_device = torch.device(output_device)


def synthetic_latent(b: int, h: int, w: int, seed: int = 1234) -> torch.Tensor:
    g = torch.Generator(device="cpu").manual_seed(seed)
    return torch.randn(b, Z, h, w, generator=g, dtype=torch.float32)


def upscaler_param_shapes(nb: int = 23, n_up: int = 2, shuffle: int = 1) -> List[Tuple[str, Tuple[int, ...]]]:
    """RRDBNet (ESRGAN: nf 64, gc 32) parameters in Real-ESRGAN key order: `n_up` upsampling convs, conv_first reading
    3 shuffle^2 channels (the pixel-unshuffle form); the defaults are the 4x model."""
    out: List[Tuple[str, Tuple[int, ...]]] = []

    def conv(name, cout, cin):
        out.append((name + ".weight", (cout, cin, 3, 3)))
        out.append((name + ".bias", (cout,)))
    conv("conv_first", 64, 3 * shuffle * shuffle)
    for i in range(nb):
        for r in (1, 2, 3):
            for j in range(4):
                conv(f"body.{i}.rdb{r}.conv{j + 1}", 32, 64 + 32 * j)
            conv(f"body.{i}.rdb{r}.conv5", 64, 192)
    for name in ["conv_body"] + [f"conv_up{k + 1}" for k in range(n_up)] + ["conv_hr"]:
        conv(name, 64, 64)
    conv("conv_last", 3, 64)
    return out


def random_upscaler_state_dict(seed: int = 0, nb: int = 23, n_up: int = 2, shuffle: int = 1) -> Dict[str, torch.Tensor]:
    """PyTorch-default-style init of an RRDBNet (config C5: random-init ESRGAN; `n_up` / `shuffle` as in
    `upscaler_param_shapes`), fp32, CPU."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    sd: Dict[str, torch.Tensor] = {}
    bound = 1.0
    for name, shape in upscaler_param_shapes(nb, n_up, shuffle):
        if len(shape) == 4:
            bound = 1.0 / math.sqrt(shape[1] * shape[2] * shape[3])
        sd[name] = (torch.rand(shape, generator=g) * 2 - 1) * bound
    return sd


def compact_param_shapes(nf: int = 64, nc: int = 32, s: int = 4) -> List[Tuple[str, Tuple[int, ...]]]:
    """Real-ESRGAN Compact (SRVGGNetCompact, PReLU) parameters: body.0 conv 3 -> nf, body.{2k+1} PReLU slopes,
    body.{2+2m} convs nf -> nf, body.{2nc+2} conv nf -> 3 s^2."""
    out: List[Tuple[str, Tuple[int, ...]]] = []
    for i in range(2 * nc + 3):
        if i % 2:
            out.append((f"body.{i}.weight", (nf,)))
            continue
        cout, cin = (3 * s * s if i == 2 * nc + 2 else nf), (3 if i == 0 else nf)
        out.append((f"body.{i}.weight", (cout, cin, 3, 3)))
        out.append((f"body.{i}.bias", (cout,)))
    return out


def random_compact_state_dict(seed: int = 0, nf: int = 64, nc: int = 32, s: int = 4) -> Dict[str, torch.Tensor]:
    """PyTorch-default-style conv init of a Compact model, PReLU slopes ~ U(-0.5, 0.5) per channel, fp32, CPU."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    sd: Dict[str, torch.Tensor] = {}
    bound = 1.0
    for name, shape in compact_param_shapes(nf, nc, s):
        if len(shape) == 4:
            bound = 1.0 / math.sqrt(shape[1] * shape[2] * shape[3])
        scale = 0.5 if len(shape) == 1 and name.endswith(".weight") else bound
        sd[name] = (torch.rand(shape, generator=g) * 2 - 1) * scale
    return sd


def span_param_shapes(nf: int = 48, s: int = 4, norm: bool = True) -> List[Tuple[str, Tuple[int, ...]]]:
    """SPAN (spandrel's "SPAN") state-dict keys in module order: Conv3XC conv_1 (3 -> nf), block_1 .. block_6 (c1_r, c2_r,
    c3_r: nf -> nf), conv_cat (1x1, 4 nf -> nf), Conv3XC conv_2, upsampler.0 (nf -> 3 s^2), and the buffer no_norm when
    the input normalisation is off.  Each Conv3XC holds sk, conv.0 / conv.1 / conv.2 (hidden width 2 cin / 2 cout) and
    eval_conv."""
    out: List[Tuple[str, Tuple[int, ...]]] = []

    def conv(name, cout, cin, k):
        out.append((f"{name}.weight", (cout, cin, k, k)))
        out.append((f"{name}.bias", (cout,)))

    def conv3xc(name, cin, cout):
        conv(f"{name}.sk", cout, cin, 1)
        conv(f"{name}.conv.0", 2 * cin, cin, 1)
        conv(f"{name}.conv.1", 2 * cout, 2 * cin, 3)
        conv(f"{name}.conv.2", cout, 2 * cout, 1)
        conv(f"{name}.eval_conv", cout, cin, 3)
    if not norm:
        out.append(("no_norm", (1,)))
    conv3xc("conv_1", 3, nf)
    for b in range(1, 7):
        for c in (1, 2, 3):
            conv3xc(f"block_{b}.c{c}_r", nf, nf)
    conv("conv_cat", nf, 4 * nf, 1)
    conv3xc("conv_2", nf, nf)
    conv("upsampler.0", 3 * s * s, nf, 3)
    return out


def random_span_state_dict(seed: int = 0, nf: int = 48, s: int = 4, norm: bool = True) -> Dict[str, torch.Tensor]:
    """Random SPAN weights with unit-gain convs (U(+-sqrt(3 / fan_in)), biases U(+-0.05)), fp32, CPU; with `norm`,
    conv_1's sk and conv.0 are scaled by 1/255 against the x 255 input.  eval_conv.* are random too: the library
    rebuilds them from conv.* and sk, as SPAN's own eval-mode forward does."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    sd: Dict[str, torch.Tensor] = {}
    bound = 1.0
    for name, shape in span_param_shapes(nf, s, norm):
        if name == "no_norm":
            sd[name] = torch.zeros(shape)
            continue
        if len(shape) == 4:
            bound = math.sqrt(3.0 / (shape[1] * shape[2] * shape[3]))
            if norm and name in ("conv_1.sk.weight", "conv_1.conv.0.weight"):
                bound /= 255.0
            sd[name] = (torch.rand(shape, generator=g) * 2 - 1) * bound
        else:
            sd[name] = (torch.rand(shape, generator=g) * 2 - 1) * 0.05
    return sd


SWINIR_UPSAMPLERS = ("pixelshuffle", "pixelshuffledirect", "nearest+conv", "")


def swinir_param_shapes(embed_dim: int = 180, depths=(6, 6, 6, 6, 6, 6), heads: int = 6, mlp_ratio: float = 2.0,
                        upsampler: str = "pixelshuffle", s: int = 4, resi_connection: str = "1conv",
                        patch_norm: bool = True, img_size: int = 64) -> List[Tuple[str, Tuple[int, ...]]]:
    """SwinIR (JingyunLiang/SwinIR network_swinir.py, spandrel's "SwinIR") state-dict keys in module order, 3 input channels,
    window 8, no ape, num_feat 64 in the tails.  Each Swin transformer layer holds its attn_mask buffer when it shifts
    (odd blocks; [(img_size / 8)^2, 64, 64]) and every layer its relative_position_index buffer [64, 64]."""
    if upsampler not in SWINIR_UPSAMPLERS:
        raise ValueError(f"upsampler must be one of {SWINIR_UPSAMPLERS}")
    C, ws = embed_dim, 8
    hidden = int(C * mlp_ratio)
    out: List[Tuple[str, Tuple[int, ...]]] = []

    def conv(name, cout, cin, k):
        out.append((f"{name}.weight", (cout, cin, k, k)))
        out.append((f"{name}.bias", (cout,)))

    def lin(name, cout, cin):
        out.append((f"{name}.weight", (cout, cin)))
        out.append((f"{name}.bias", (cout,)))

    def resi(name):
        if resi_connection == "1conv":
            conv(name, C, C, 3)
        else:
            conv(f"{name}.0", C // 4, C, 3)
            conv(f"{name}.2", C // 4, C // 4, 1)
            conv(f"{name}.4", C, C // 4, 3)
    conv("conv_first", C, 3, 3)
    if patch_norm:
        out.append(("patch_embed.norm.weight", (C,)))
        out.append(("patch_embed.norm.bias", (C,)))
    for i, depth in enumerate(depths):
        for j in range(depth):
            b = f"layers.{i}.residual_group.blocks.{j}"
            if j % 2:
                out.append((f"{b}.attn_mask", ((img_size // ws) ** 2, ws * ws, ws * ws)))
            out.append((f"{b}.norm1.weight", (C,)))
            out.append((f"{b}.norm1.bias", (C,)))
            out.append((f"{b}.attn.relative_position_bias_table", ((2 * ws - 1) ** 2, heads)))
            out.append((f"{b}.attn.relative_position_index", (ws * ws, ws * ws)))
            lin(f"{b}.attn.qkv", 3 * C, C)
            lin(f"{b}.attn.proj", C, C)
            out.append((f"{b}.norm2.weight", (C,)))
            out.append((f"{b}.norm2.bias", (C,)))
            lin(f"{b}.mlp.fc1", hidden, C)
            lin(f"{b}.mlp.fc2", C, hidden)
        resi(f"layers.{i}.conv")
    out.append(("norm.weight", (C,)))
    out.append(("norm.bias", (C,)))
    resi("conv_after_body")
    if upsampler == "pixelshuffle":
        conv("conv_before_upsample.0", 64, C, 3)
        for k in range(int(math.log2(s))):
            conv(f"upsample.{2 * k}", 256, 64, 3)
        conv("conv_last", 3, 64, 3)
    elif upsampler == "pixelshuffledirect":
        conv("upsample.0", 3 * s * s, C, 3)
    elif upsampler == "nearest+conv":
        conv("conv_before_upsample.0", 64, C, 3)
        conv("conv_up1", 64, 64, 3)
        if s == 4:
            conv("conv_up2", 64, 64, 3)
        conv("conv_hr", 64, 64, 3)
        conv("conv_last", 3, 64, 3)
    else:
        conv("conv_last", 3, C, 3)
    return out


def _swin_buffers(name: str, shape: Tuple[int, ...]) -> torch.Tensor:
    """SwinIR's relative_position_index and attn_mask buffers as the published module computes them at construction."""
    ws = 8
    if name.endswith("relative_position_index"):
        r = torch.arange(ws * ws)
        dy = (r[:, None] // ws - r[None, :] // ws) + ws - 1
        dx = (r[:, None] % ws - r[None, :] % ws) + ws - 1
        return dy * (2 * ws - 1) + dx
    res = int(round(math.sqrt(shape[0]))) * ws                      # attn_mask of an img_size x img_size input, shift 4
    img = torch.zeros(res, res)
    cnt = 0
    for hs in (slice(0, -ws), slice(-ws, -ws // 2), slice(-ws // 2, None)):
        for wsl in (slice(0, -ws), slice(-ws, -ws // 2), slice(-ws // 2, None)):
            img[hs, wsl] = cnt
            cnt += 1
    win = img.view(res // ws, ws, res // ws, ws).permute(0, 2, 1, 3).reshape(-1, ws * ws)
    m = win[:, None, :] - win[:, :, None]
    return m.masked_fill(m != 0, -100.0).masked_fill(m == 0, 0.0)


def random_swinir_state_dict(seed: int = 0, embed_dim: int = 180, depths=(6, 6, 6, 6, 6, 6), heads: int = 6,
                             mlp_ratio: float = 2.0, upsampler: str = "pixelshuffle", s: int = 4,
                             resi_connection: str = "1conv", patch_norm: bool = True) -> Dict[str, torch.Tensor]:
    """Random SwinIR weights, fp32, CPU, in spandrel's keys and shapes (swinir_param_shapes), buffers included: unit-gain
    convs and linears (U(+-sqrt(3 / fan_in))), proj and fc2 at half that gain, LayerNorm gains 1 +- 0.2 and shifts +-0.1,
    bias tables U(+-1), biases U(+-0.05)."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    sd: Dict[str, torch.Tensor] = {}
    for name, shape in swinir_param_shapes(embed_dim, depths, heads, mlp_ratio, upsampler, s, resi_connection, patch_norm):
        u = torch.rand(shape, generator=g) * 2 - 1
        if name.endswith(("relative_position_index", "attn_mask")):
            sd[name] = _swin_buffers(name, shape)
        elif name.endswith("relative_position_bias_table"):
            sd[name] = u
        elif "norm" in name.rsplit(".", 2)[-2] or name.startswith("norm."):
            sd[name] = 1.0 + 0.2 * u if name.endswith("weight") else 0.1 * u
        elif name.endswith("weight"):
            fan_in = math.prod(shape[1:])
            gain = 0.5 if (".attn.proj." in name or ".mlp.fc2." in name) else 1.0
            sd[name] = u * gain * math.sqrt(3.0 / fan_in)
        else:
            sd[name] = 0.05 * u
    return sd
