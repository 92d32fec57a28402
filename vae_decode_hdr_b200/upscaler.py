"""Host side of the HDR upscaler path (libhdrvae.so `hdrvae_upscale*`): owns one model object per (upscaler weights,
device).  PyTorch is plumbing only (device memory, current stream); all arithmetic happens in the library."""
from __future__ import annotations

import ctypes as C
import re
from typing import Dict, Optional

import torch

from . import _native as N
from .engine import _DTYPE_ID, _require_cuda

REVERSAL = {"none": N.REVERSAL_NONE, "atanh": N.REVERSAL_ATANH, "logit": N.REVERSAL_LOGIT}
# hdr_upscale_with_model.py:64 — the node's enum; all five are implemented for local_fix (torch semantics for the
# first four, ComfyUI's own spherical-linear "bislerp" — the node's default — restated in oracle/upscaler_oracle.py)
UPSCALE_METHODS = ["nearest-exact", "bilinear", "area", "bicubic", "bislerp"]


def reversal_for_architecture(name: str) -> str:
    """hdr_upscale_with_model.py:266-279: which inverse activation the forward hook applies."""
    if name in ("ESRGAN", "RealESRGAN", "SwinIR", "HAT") or "VAE" in name:
        return "atanh"
    return "logit"


def is_compact_state_dict(state_dict) -> bool:
    """The Real-ESRGAN Compact (SRVGGNetCompact) key layout, as the library recognises it: `body.0.weight` and no
    `conv_first.*`.  The library then checks for SPAN (`conv_1.sk.weight`) and SwinIR (`SWIN_KEY`); every other model it
    runs is an RRDBNet (see `rrdbnet_scale`)."""
    return "body.0.weight" in state_dict and not any(k.startswith("conv_first.") for k in state_dict)


# The first Swin transformer layer's relative-position bias table: the key by which the library recognises SwinIR.  HAT
# state dicts have it too; the library refuses them by their own keys.
SWIN_KEY = "layers.0.residual_group.blocks.0.attn.relative_position_bias_table"
_HAT_MARKS = ("conv_block", "overlap_attn", "relative_position_index_SA")


def is_swinir_state_dict(state_dict) -> bool:
    """The SwinIR key layout as the library recognises it: `SWIN_KEY` and none of HAT's own keys (`conv_block`,
    `overlap_attn`, `relative_position_index_SA`)."""
    return SWIN_KEY in state_dict and not any(m in k for k in state_dict for m in _HAT_MARKS)


_OLD_TOP = re.compile(r"model\.(\d+)\.(weight|bias)$")


def rrdbnet_scale(state_dict) -> Optional[int]:
    """Scale of an RRDBNet state dict by the library's rules, without a device: s = 2^u / f for u upsampling convs (old
    arch: conv_last at top-level index 3u + 4; Real-ESRGAN names: conv_up1 / conv_up2 / conv_up3) and pixel-unshuffle
    factor f (conv_first reads 3 f^2 channels).  8 for three upsampling convs; None for a layout the library does not
    recognise (no conv_first, f not 1 / 2 / 4, s below 1, an old-arch conv_last index that fits no u)."""
    tops = [int(m.group(1)) for m in (_OLD_TOP.match(k) for k in state_dict) if m and m.group(1) != "1"]
    if tops:
        top = max(tops)
        if top < 4 or (top - 4) % 3:
            return None
        n_up, first = (top - 4) // 3, state_dict.get("model.0.weight")
    else:
        n_up = max([j for j in (1, 2, 3) if f"conv_up{j}.weight" in state_dict], default=0)
        first = state_dict.get("conv_first.weight")
    if n_up >= 3:
        return 8
    if first is None or len(first.shape) != 4 or first.shape[1] not in (3, 12, 48):
        return None
    f = {3: 1, 12: 2, 48: 4}[int(first.shape[1])]
    return (1 << n_up) // f if (1 << n_up) >= f else None


class HdrUpscalerEngine:
    """One upscaler model packed for the tcgen05 conv kernel on one GPU: an RRDBNet (ESRGAN: nf 64, gc 32; 0, 1 or 2
    upsampling convs, pixel-unshuffle factor 1, 2 or 4, scale 1, 2 or 4), a Real-ESRGAN Compact (SRVGGNetCompact,
    PReLU, 1x / 2x / 4x), a SPAN (nf <= 64, 1x / 2x / 4x; the library fuses every Conv3XC from its conv.* and sk
    tensors and ignores eval_conv.*) or a SwinIR (embed_dim <= 256, head dim <= 32, window 8, 1conv / 3conv, upsampler
    "pixelshuffle", "pixelshuffledirect" or "nearest+conv" at 2x / 4x, or "" at 1x; the stored relative_position_index
    and attn_mask buffers are not read).  `scale` is the model's, read from the library; `blocks` is the RRDB count, the
    Compact's body-conv count, SPAN's 6 or SwinIR's RSTB count."""

    def __init__(self, state_dict: Dict[str, torch.Tensor], device="cuda"):
        self.lib = N.load_library()
        self.device = _require_cuda(device)
        self._ctx = C.c_void_p()
        self._up = C.c_void_p()
        N.check(self.lib.hdrvae_create(C.byref(self._ctx), self.device.index), "hdrvae_create")
        N.check(self.lib.hdrvae_upscaler_create(self._ctx, C.byref(self._up)), "hdrvae_upscaler_create")
        self._workspace: Optional[torch.Tensor] = None
        keep, descs = [], []
        for name, t in state_dict.items():
            if not isinstance(t, torch.Tensor) or t.dim() == 0 or t.dim() > 4:
                continue
            if t.dtype not in _DTYPE_ID:
                t = t.float()
            t = t.detach().contiguous()
            keep.append(t)
            d = N.HdrvaeWeightDesc()
            d.name, d.data, d.dtype, d.ndim = name.encode(), t.data_ptr(), _DTYPE_ID[t.dtype], t.dim()
            for i, s in enumerate(t.shape):
                d.shape[i] = s
            descs.append(d)
        arr = (N.HdrvaeWeightDesc * len(descs))(*descs)
        with torch.cuda.device(self.device):
            torch.cuda.synchronize(self.device)
            N.check(self.lib.hdrvae_upscaler_load_weights(self._up, arr, len(descs)), "hdrvae_upscaler_load_weights")
        self.blocks = int(self.lib.hdrvae_upscaler_blocks(self._up))
        self.scale = int(self.lib.hdrvae_upscaler_scale(self._up))

    def set_conv_impl(self, impl: int) -> None:
        N.check(self.lib.hdrvae_set_conv_impl(self._ctx, impl), "hdrvae_set_conv_impl")

    def _ws(self, need: int) -> torch.Tensor:
        if self._workspace is None or self._workspace.numel() < need:
            self._workspace = None
            self._workspace = torch.empty(need, dtype=torch.uint8, device=self.device)
        return self._workspace

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def forward(self, x_bhwc: torch.Tensor, reversal: str = "atanh") -> torch.Tensor:
        """The network + reversal hook on a batch of equal tiles: [n,h,w,3] -> [n,s*h,s*w,3] (fp32, s = self.scale)."""
        if x_bhwc.dim() != 4 or x_bhwc.shape[-1] != 3:
            raise ValueError(f"expected [n,h,w,3], got {tuple(x_bhwc.shape)}")
        n, h, w, _ = x_bhwc.shape
        with torch.cuda.device(self.device):
            x = x_bhwc.to(self.device, torch.float32).contiguous()
            y = torch.empty((n, self.scale * h, self.scale * w, 3), dtype=torch.float32, device=self.device)
            need = C.c_size_t()
            N.check(self.lib.hdrvae_upscaler_forward_bytes(self._up, n, h, w, C.byref(need)), "hdrvae_upscaler_forward_bytes")
            ws = self._ws(int(need.value))
            N.check(self.lib.hdrvae_upscaler_forward(self._up, x.data_ptr(), n, h, w, REVERSAL[reversal], y.data_ptr(),
                                                     ws.data_ptr(), ws.numel(), self._stream()), "hdrvae_upscaler_forward")
        return y

    def upscale(self, image_bhwc: torch.Tensor, reversal: str = "atanh", small_blur: bool = False, local_fix: bool = False,
                upscale_method: str = "bilinear", out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """The whole node path on the GPU: [B,H,W,3] fp32 -> [B,s*H,s*W,3] fp32 (s = self.scale)."""
        if image_bhwc.dim() != 4 or image_bhwc.shape[-1] != 3:
            raise ValueError(f"expected an IMAGE tensor [B,H,W,3], got {tuple(image_bhwc.shape)}")
        if reversal not in ("atanh", "logit"):
            raise ValueError("reversal must be 'atanh' or 'logit'")
        if local_fix and upscale_method not in N.UPSCALE_METHODS:
            raise ValueError(f"unknown upscale_method {upscale_method!r} (available: {sorted(N.UPSCALE_METHODS)})")
        B, H, W, _ = image_bhwc.shape
        with torch.cuda.device(self.device):
            x = image_bhwc.to(self.device, torch.float32).contiguous()
            if out is None:
                out = torch.empty((B, self.scale * H, self.scale * W, 3), dtype=torch.float32, device=self.device)
            need = C.c_size_t()
            N.check(self.lib.hdrvae_upscale_workspace_bytes(self._up, B, H, W, C.byref(need)), "hdrvae_upscale_workspace_bytes")
            ws = self._ws(int(need.value))
            N.check(self.lib.hdrvae_upscale(self._up, x.data_ptr(), B, H, W, REVERSAL[reversal], int(bool(small_blur)),
                                            int(bool(local_fix)), N.UPSCALE_METHODS.get(upscale_method, 0), out.data_ptr(),
                                            ws.data_ptr(), ws.numel(), self._stream()), "hdrvae_upscale")
        return out

    def close(self) -> None:
        if getattr(self, "_up", None) is not None and self._up.value:
            self.lib.hdrvae_upscaler_destroy(self._up)
            self._up = C.c_void_p()
        if getattr(self, "_ctx", None) is not None and self._ctx.value:
            self.lib.hdrvae_destroy(self._ctx)
            self._ctx = C.c_void_p()
        self._workspace = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
