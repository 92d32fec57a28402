"""fp32 oracle of an SD1.x / SDXL VAE's decode side (TEST INFRASTRUCTURE ONLY).

The SD-family decoder is the Flux.1 graph of oracle/flux_decoder.py with ``z_channels = 4`` (conv_in 4 -> 512), and
ComfyUI's ``AutoencoderKL`` first-stage model applies ``post_quant_conv`` (1x1, 4 -> 4, with bias) to the latent before
the decoder.  ``SDFirstStage`` restates that; its ``features`` and ``conv_out`` mirror FluxDecoder's, so
hdr_oracle.simple_hdr_decode and the test metrics take it unchanged.  ``FakeComfySDVAE`` is the matching slice of
``comfy.sd.VAE``."""
import torch
from torch import nn

from oracle.flux_decoder import CH, CH_MULT, FakeComfyVAE, FluxDecoder

SD_Z_CHANNELS = 4


class SDFirstStage(nn.Module):
    """``decoder(post_quant_conv(z))`` with the state-dict keys of ComfyUI's first-stage model."""

    def __init__(self, z_channels: int = SD_Z_CHANNELS):
        super().__init__()
        self.decoder = FluxDecoder()
        self.decoder.conv_in = nn.Conv2d(z_channels, CH * CH_MULT[-1], 3, 1, 1)     # same key, 4 input channels
        self.post_quant_conv = nn.Conv2d(z_channels, z_channels, 1)

    @property
    def conv_out(self) -> nn.Conv2d:
        return self.decoder.conv_out

    def features(self, z):
        return self.decoder.features(self.post_quant_conv(z))

    def forward(self, z):
        return self.decoder(self.post_quant_conv(z))


def build_sd_decoder(seed: int = 0, dtype=torch.float32, device="cpu") -> SDFirstStage:
    """Random-init SD first stage under ``torch.manual_seed(seed)``, built on the CPU like oracle.build_decoder."""
    gen_state = torch.random.get_rng_state()
    try:
        torch.manual_seed(seed)
        m = SDFirstStage()
    finally:
        torch.random.set_rng_state(gen_state)
    return m.to(device=device, dtype=dtype).eval()


def make_sd_latent(b: int, h: int, w: int, seed: int = 1234, device="cpu") -> torch.Tensor:
    g = torch.Generator(device="cpu").manual_seed(seed)
    return torch.randn(b, SD_Z_CHANNELS, h, w, generator=g, dtype=torch.float32).to(device)


class FakeComfySDVAE(FakeComfyVAE):
    """``first_stage_model`` carries ``.post_quant_conv`` next to ``.decoder``; ``decode(z)`` =
    ``clamp((decoder(post_quant_conv(z))+1)/2, 0, 1).movedim(1, -1)``."""

    def __init__(self, first_stage: SDFirstStage):
        super().__init__(first_stage.decoder)
        self.first_stage_model = first_stage

    @torch.no_grad()
    def decode(self, samples_in: torch.Tensor) -> torch.Tensor:
        x = self.first_stage_model(samples_in.to(self.device).to(self.vae_dtype)).float()
        return torch.clamp((x + 1.0) / 2.0, 0.0, 1.0).to(self.output_device).movedim(1, -1)
