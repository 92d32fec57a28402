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


def upscaler_param_shapes(nb: int = 23) -> List[Tuple[str, Tuple[int, ...]]]:
    """RRDBNet (ESRGAN 4x: nf 64, gc 32) parameters in Real-ESRGAN key order."""
    out: List[Tuple[str, Tuple[int, ...]]] = []

    def conv(name, cout, cin):
        out.append((name + ".weight", (cout, cin, 3, 3)))
        out.append((name + ".bias", (cout,)))
    conv("conv_first", 64, 3)
    for i in range(nb):
        for r in (1, 2, 3):
            for j in range(4):
                conv(f"body.{i}.rdb{r}.conv{j + 1}", 32, 64 + 32 * j)
            conv(f"body.{i}.rdb{r}.conv5", 64, 192)
    for name in ("conv_body", "conv_up1", "conv_up2", "conv_hr"):
        conv(name, 64, 64)
    conv("conv_last", 3, 64)
    return out


def random_upscaler_state_dict(seed: int = 0, nb: int = 23) -> Dict[str, torch.Tensor]:
    """PyTorch-default-style init of an RRDBNet (config C5: random-init ESRGAN), fp32, CPU."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    sd: Dict[str, torch.Tensor] = {}
    bound = 1.0
    for name, shape in upscaler_param_shapes(nb):
        if len(shape) == 4:
            bound = 1.0 / math.sqrt(shape[1] * shape[2] * shape[3])
        sd[name] = (torch.rand(shape, generator=g) * 2 - 1) * bound
    return sd
