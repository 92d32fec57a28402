"""Comparison metrics and helpers shared by the GPU parity tests."""
import torch
import torch.nn.functional as F

SAT_BAND = 1e-3


def rel_l2(a: torch.Tensor, b: torch.Tensor) -> float:
    return float((a.double() - b.double()).norm() / b.double().norm())


def rel_trimmed(a, b, frac):
    e = ((a - b).double() ** 2).sum(dim=-1).flatten()
    k = e.numel() - int(frac * e.numel())
    return float(e.sort().values[:k].sum().sqrt() / b.double().norm())


class GpuModel(torch.nn.Module):
    """The oracle's tiling / recombination driven by the GPU network: isolates everything after the model."""

    def __init__(self, eng):
        super().__init__()
        self.eng = eng

    def forward(self, a):
        return self.eng.forward(a.movedim(1, -1).contiguous().to("cuda:0"), "none").cpu().movedim(-1, 1)


def saturation_band_mask(dec, pre_nchw: torch.Tensor, band: float = SAT_BAND) -> torch.Tensor:
    """Pixels [B,H,W] (bool) the logit-recovery modes are ill-conditioned at, decided BY RULE from the reference:
    the reference applies logit(clamp(s, 1e-7, 1 - 1e-7)) to s = clamp((conv_out + 1) / 2, 0, 1)
    (hdr_vae_decode.py:927-932, 1085-1102); d logit / ds = 1 / (s (1 - s)) exceeds 1e3 within `band` = 1e-3 of either
    clamp end (a 16-bit pipeline's error in s of ~2e-4 then moves the recovered value by > 0.2 of its 32-wide range,
    and because the squared error grows like 1 / distance^2 a single such pixel can outweigh a small image), and a value
    on the other side of the end is clamped to the +-16 bound.  A pixel is in the band when ANY
    of its three un-clamped reference values (conv_out + 1) / 2 lies within `band` of 0 or of 1.  Values solidly
    beyond an end (clamped in the reference AND in any faithful implementation) stay in the comparison."""
    conv = F.conv2d(pre_nchw.float(), dec.conv_out.weight.float(), dec.conv_out.bias.float(), padding=1)
    s = (conv + 1.0) / 2.0
    m = (s.abs() < band) | ((s - 1.0).abs() < band)
    return m.any(dim=1)


def rel_l2_outside(a_bhwc: torch.Tensor, b_bhwc: torch.Tensor, mask_bhw: torch.Tensor) -> float:
    """rel-L2 of a vs b over the pixels NOT in mask (the denominator is taken over the same pixels)."""
    keep = (~mask_bhw).unsqueeze(-1).to(a_bhwc.device)
    d = ((a_bhwc.double() - b_bhwc.double()) * keep).norm()
    n = (b_bhwc.double() * keep).norm()
    return float(d / n)
