"""HDRVAEDecode — the ComfyUI node, same surface as the reference (hdr_vae_decode.py:23-60),
computing on libhdrvae.so (sm_100a) instead of PyTorch eager.

Kept verbatim from the reference: INPUT_TYPES (required samples/vae, optional hdr_mode enum in
the code's order with default "mathematical_recovery", conservative_ev_multiplier FLOAT 0.1-10),
RETURN_TYPES ("IMAGE",), RETURN_NAMES ("image",), FUNCTION "simple_hdr_decode", CATEGORY "latent",
and the float32 [B,H,W,3] contiguous output (:195,:354).

Differences, all documented in DESIGN.md:
  * one decoder pass instead of two + a third conv_out (SURVEY.md §0.5);
  * README-era mode names "moderate"/"aggressive" are accepted as aliases (SURVEY.md §0.2);
  * NORMALIZATION_FUNCTION is recomputed per call (the reference's sticky state, SURVEY.md §0.9, is a bug);
  * the non-deterministic bypass fallback (SURVEY.md §0.8) is replaced by a deterministic rule: the
    intelligent result is always returned and ``last_stats['accepted']`` tells whether the reference
    would have gone to its bypass.
"""
from __future__ import annotations

import logging
import os
import weakref
from collections import OrderedDict
from typing import Any, Dict, Optional, Tuple

import torch

from .engine import DEFAULT_MODE, HDR_MODES, HdrVaeEngine, quantiles

logger = logging.getLogger(__name__)


def _decoder_of(vae: Any):
    try:
        return vae.first_stage_model.decoder          # hdr_vae_decode.py:842
    except AttributeError as e:
        raise RuntimeError("HDRVAEDecode: vae.first_stage_model.decoder not found (not a Flux.1 / SD1.x / SDXL-style "
                           "AutoencoderKL VAE)") from e


def _post_quant_conv_of(vae: Any) -> Optional[torch.nn.Module]:
    """SD1.x / SDXL first-stage models apply post_quant_conv (1x1 conv, 4 -> 4 channels) to the latent before the decoder;
    Flux's has none (absent, None or nn.Identity)."""
    m = getattr(getattr(vae, "first_stage_model", None), "post_quant_conv", None)
    w = getattr(m, "weight", None)
    if isinstance(m, torch.nn.Module) and isinstance(w, torch.Tensor) and w.dim() == 4:
        return m
    return None


def _engine_state_dict(decoder, pqc: Optional[torch.nn.Module]) -> Dict[str, torch.Tensor]:
    """The decoder's state dict plus post_quant_conv.{weight,bias} (a bias-less conv sends zeros)."""
    sd = dict(decoder.state_dict())
    if pqc is not None:
        sd["post_quant_conv.weight"] = pqc.weight.detach()
        b = pqc.bias
        sd["post_quant_conv.bias"] = b.detach() if b is not None else pqc.weight.new_zeros(pqc.weight.shape[0])
    return sd


def _weights_key(decoder, pqc: Optional[torch.nn.Module] = None) -> Tuple:
    """Identity + in-place-modification fingerprint of EVERY parameter of the decoder and of post_quant_conv (storage
    address, version counter, size).  The id() half is safe against reuse because an engine never outlives its decoder
    (weakref.finalize below)."""
    ps = list(decoder.parameters()) + (list(pqc.parameters()) if pqc is not None else [])
    return (id(decoder), len(ps), hash(tuple((p.data_ptr(), p._version, p.numel()) for p in ps)))


# README.md:143-145 documents three inputs the code no longer has; the shipped example workflow still names them
# (workflow_examples/HDR_VAE_DECODE.json:499-504).  They are accepted and ignored so API-format prompts that carry them load.
LEGACY_IGNORED_INPUTS = ("max_range", "scale_factor", "enable_negatives")
MAX_CACHED_ENGINES = 2


_IN_COMFYUI: Optional[bool] = None


def _in_comfyui() -> bool:
    global _IN_COMFYUI
    if _IN_COMFYUI is None:          # probed once: a failed import is not cached by Python and would be retried per call
        try:
            import comfy.model_management  # noqa: F401
            _IN_COMFYUI = True
        except Exception:
            _IN_COMFYUI = False
    return _IN_COMFYUI


class HDRVAEDecode:
    """HDR VAE Decode (B200-native).  Drop-in for the reference node class of the same name."""

    # LRU of at most MAX_CACHED_ENGINES engines (packed weights + CUDA graphs + workspace each); an engine is closed
    # when it is evicted, when its weights change in place, or when its decoder is garbage-collected
    _engines: "OrderedDict[Tuple, HdrVaeEngine]" = OrderedDict()

    def __init__(self):
        self.logger = logger
        self.NORMALIZATION_FUNCTION = str()
        self.last_stats: Optional[Dict] = None
        self.profile_quantiles = False      # True: last_stats["out_quantiles"] = {q: value} of the output image

    @classmethod
    def INPUT_TYPES(cls):
        return {
            "required": {
                "samples": ("LATENT",),
                "vae": ("VAE",),
            },
            "optional": {
                "hdr_mode": (list(HDR_MODES),
                             {"default": DEFAULT_MODE,
                              "tooltip": "conservative: Gentle conservative_ev_multiplier expansion, safest for general use \n "
                                         "exposure: Natural exposure-based HDR for compositing workflows \n "
                                         "mathematical_recovery: Full mathematical recovery, maximum range"}),
                "conservative_ev_multiplier": ("FLOAT", {"default": 1.0, "min": 0.1, "max": 10.0, "step": 0.1,
                                                         "tooltip": "Expansion multiplier for the conservative mode."}),
            }
        }

    RETURN_TYPES = ("IMAGE",)
    RETURN_NAMES = ("image",)
    FUNCTION = "simple_hdr_decode"
    CATEGORY = "latent"

    # ------------------------------------------------------------------------------------------
    @staticmethod
    def _compute_device(vae: Any, latent: torch.Tensor) -> torch.device:
        for cand in (getattr(vae, "device", None), latent.device):
            if cand is not None and torch.device(cand).type == "cuda":
                return torch.device(cand)
        if not torch.cuda.is_available():
            raise RuntimeError("HDRVAEDecode (B200) needs a CUDA device; there is no CPU fallback")
        return torch.device("cuda", torch.cuda.current_device())

    @classmethod
    def _evict(cls, key) -> None:
        eng = cls._engines.pop(key, None)
        if eng is not None:
            eng.close()

    @classmethod
    def _engine_for(cls, vae: Any, device: torch.device) -> HdrVaeEngine:
        decoder, pqc = _decoder_of(vae), _post_quant_conv_of(vae)
        key = (_weights_key(decoder, pqc), str(device))
        eng = cls._engines.get(key)
        if eng is None:
            for k in [k for k in cls._engines if k[0][0] == id(decoder) and k[1] == str(device)]:
                cls._evict(k)                          # weights changed in place: repack
            eng = HdrVaeEngine(_engine_state_dict(decoder, pqc), device)
            cls._register(decoder, key, eng)
        else:
            cls._engines.move_to_end(key)
        return eng

    @classmethod
    def _register(cls, decoder, key, eng: HdrVaeEngine) -> None:
        cls._engines[key] = eng
        cls._engines.move_to_end(key)
        try:
            weakref.finalize(decoder, cls._evict, key)     # the engine dies with its decoder (no stale id() reuse)
        except TypeError:
            pass
        while len(cls._engines) > MAX_CACHED_ENGINES:
            cls._evict(next(iter(cls._engines)))

    @classmethod
    def adopt_engine(cls, vae: Any, device, engine: HdrVaeEngine) -> None:
        """Register an already-built engine for this vae's decoder (and post_quant_conv) weights (avoids a second
        repack)."""
        decoder = _decoder_of(vae)
        cls._register(decoder, (_weights_key(decoder, _post_quant_conv_of(vae)), str(torch.device(device))), engine)

    @classmethod
    def release_memory(cls, keep_weights: bool = True) -> None:
        """Give the GPU memory back: drop every engine's workspace (and, with keep_weights=False, the engines).  ComfyUI's
        model_management cannot see this memory; inside ComfyUI the workspace is released after every call unless
        HDRVAE_KEEP_WORKSPACE=1."""
        for k in list(cls._engines):
            if keep_weights:
                cls._engines[k].free_workspace()
            else:
                cls._evict(k)
        if torch.cuda.is_available():
            torch.cuda.empty_cache()

    def simple_hdr_decode(
        self,
        samples: Dict[str, torch.Tensor],
        vae: Any,
        hdr_mode: str = DEFAULT_MODE,
        conservative_ev_multiplier: float = 1.0,
        **legacy_inputs,
    ) -> Tuple[torch.Tensor]:
        unknown = [k for k in legacy_inputs if k not in LEGACY_IGNORED_INPUTS]
        if unknown:
            raise TypeError(f"simple_hdr_decode() got unexpected keyword argument(s) {unknown}")
        if legacy_inputs:
            self.logger.info("HDRVAEDecode: ignoring README-era inputs %s (the reference code has no such inputs, "
                             "hdr_vae_decode.py:40-55)", sorted(legacy_inputs))
        latent = samples["samples"]                    # hdr_vae_decode.py:78
        device = self._compute_device(vae, latent)
        engine = self._engine_for(vae, device)
        image, stats = engine.decode(latent, hdr_mode, conservative_ev_multiplier, want_stats=True)
        if self.profile_quantiles:
            # statistical profiling beyond the reference's min/max/mean: exact quantiles by GPU radix select
            qs = (0.01, 0.5, 0.99, 0.999)
            stats["out_quantiles"] = dict(zip(qs, quantiles(image, qs)))
        self.last_stats = stats
        self.NORMALIZATION_FUNCTION = {0: "", 1: "SIGMOID", 2: "TANH"}[stats["norm_function"]]
        if not stats["accepted"]:
            self.logger.warning("HDRVAEDecode: no value above 1.0 in the intelligent result; the reference would "
                                "fall back to its non-deterministic bypass decode here (returning the deterministic "
                                "intelligent result)")
        self.logger.debug("OUTPUT: range=[%.3f, %.3f], HDR pixels: %d, Negative pixels: %d", stats["out_min"],
                          stats["out_max"], stats["hdr_pixels"], stats["negative_pixels"])
        out_dev = getattr(vae, "output_device", None)
        if out_dev is None:
            out_dev = latent.device
        out_dev = torch.device(out_dev)
        if out_dev != image.device:
            if out_dev.type == "cpu":
                # pinned staging (torch's caching host allocator recycles it): D2H at link speed
                host = torch.empty(image.shape, dtype=image.dtype, pin_memory=True)
                host.copy_(image, non_blocking=True)
                torch.cuda.current_stream(image.device).synchronize()
                image = host
            else:
                image = image.to(out_dev)
        keep = os.environ.get("HDRVAE_KEEP_WORKSPACE")
        if keep == "0" or (keep is None and _in_comfyui()):
            engine.free_workspace()                    # hand the workspace back to the host application's allocator
            torch.cuda.empty_cache()
        return (image,)
