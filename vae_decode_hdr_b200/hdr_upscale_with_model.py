"""`HDRUpscaleWithModel` — drop-in for the reference node of the same name
(/root/reference/hdr_upscale_with_model.py:50-279): same INPUT_TYPES / RETURN_TYPES / FUNCTION / CATEGORY, same
argument meaning, IMAGE in ([B,H,W,3] float32) -> IMAGE out ([B,sH,sW,3] float32, s = the model's scale).

What changes is where the work happens: the model, the reversal hook, the tiled feather blend and the YCbCr
recombination all run in libhdrvae.so on the GPU (vae_decode_hdr_b200/csrc/upscaler.cu).  There is no CPU path: without
a CUDA device or without the library the node raises.

Model loading stays what it is in ComfyUI (folder_paths + spandrel, :73-77); the node only reads
`descriptor.model.state_dict()`, `descriptor.scale` and `descriptor.architecture.name`.  Four architectures run:
RRDBNet (ESRGAN: nf 64, gc 32) at 1x, 2x and 4x -- the plain form with 0, 1 or 2 upsampling convs and the pixel-unshuffle
form (RealESRGAN_x2plus) --, Real-ESRGAN Compact (SRVGGNetCompact with PReLU) at 1x, 2x and 4x, SPAN (nf <= 64) at
1x, 2x and 4x, which gets the logit reversal like every architecture outside the reference's atanh list, and SwinIR
(window 8, embed_dim <= 256) at 1x, 2x and 4x, which gets atanh.  An RRDBNet of another scale (8x), or one whose
`descriptor.scale` disagrees with its weights, fails before any GPU work; any other architecture (HAT among them) is
rejected by the library with an error naming the tensor that does not fit; a Compact, SPAN or SwinIR model whose
`descriptor.scale` disagrees with its weights is an error too.
"""
from __future__ import annotations

import logging
import os
from collections import OrderedDict
from typing import Any, Tuple

import torch

from .upscaler import (SWIN_KEY, UPSCALE_METHODS, HdrUpscalerEngine, is_compact_state_dict, reversal_for_architecture,
                       rrdbnet_scale)


def _model_filenames():
    try:
        import folder_paths  # provided by ComfyUI
        return folder_paths.get_filename_list("upscale_models")
    except Exception:
        return []


class HDRUpscaleWithModel:
    # LRU of at most MAX_ENGINES engines keyed on the model FILE (resolved path, mtime, size) and the device: the node
    # reloads the model through spandrel on every execution (:149-152), so object identity never repeats
    _engines: "OrderedDict[Any, HdrUpscalerEngine]" = OrderedDict()
    MAX_ENGINES = 2
    logger = logging.getLogger("HDRUpscaleWithModel")

    @classmethod
    def INPUT_TYPES(s):
        # hdr_upscale_with_model.py:59-66
        return {"required": {
            "image": ("IMAGE",),
            "model_name": (_model_filenames(),),
            "small_blur": ("BOOLEAN", {"default": False, "tooltip": "Apply small blur to avoid hot-pixels."}),
            "local_fix": ("BOOLEAN", {"default": False, "tooltip": "Apply local masking to suppress extreme hotspots in dark areas."}),
            "upscale_method": (list(UPSCALE_METHODS), {"default": "bislerp", "tooltip": "method used by the local_fix"}),
        }}

    RETURN_TYPES = ("IMAGE",)
    FUNCTION = "upscale"
    CATEGORY = "HDR/Upscale"

    # hdr_upscale_with_model.py:73-77 — unchanged: ComfyUI's model folder + spandrel's loader
    @staticmethod
    def _model_path(model_name) -> str:
        import folder_paths
        return folder_paths.get_full_path("upscale_models", model_name)

    def _load_model_internal(self, model_name):
        from spandrel import ModelLoader
        return ModelLoader().load_from_file(self._model_path(model_name))

    @staticmethod
    def _compute_device(image: torch.Tensor) -> torch.device:
        if image.device.type == "cuda":
            return image.device
        if not torch.cuda.is_available():
            raise RuntimeError("HDRUpscaleWithModel (B200) needs a CUDA device; there is no CPU fallback")
        return torch.device("cuda", torch.cuda.current_device())

    @staticmethod
    def _file_key(path: str, device: torch.device):
        try:
            st = os.stat(path)
            return (os.path.realpath(path), st.st_mtime_ns, st.st_size, str(device))
        except (OSError, TypeError):
            return (str(path), 0, 0, str(device))

    @staticmethod
    def _new_engine(descriptor, device: torch.device) -> HdrUpscalerEngine:
        """Packs the descriptor's weights; the engine's scale (read from the weights) must be `descriptor.scale`."""
        scale = getattr(descriptor, "scale", 4)
        sd = descriptor.model.state_dict()
        # (SWIN_KEY: SwinIR, or HAT, which the library refuses by name; neither has an RRDBNet's scale rule)
        if not is_compact_state_dict(sd) and SWIN_KEY not in sd:
            # RRDBNet: the scale follows from the key layout, so both checks fail before any weights reach the GPU (an
            # unrecognised layout goes on to the library, whose error names the tensor that does not fit)
            weights = rrdbnet_scale(sd)
            if weights is not None and weights not in (1, 2, 4):
                raise RuntimeError(f"HDRUpscaleWithModel (B200) implements RRDBNet / ESRGAN at scales 1, 2 and 4; these "
                                   f"weights upscale {weights}x (descriptor scale {scale})")
            if weights is not None and weights != scale:
                raise RuntimeError(f"HDRUpscaleWithModel (B200): the model descriptor gives scale {scale}, its weights "
                                   f"are a {weights}x network")
        engine = HdrUpscalerEngine(sd, device)
        if engine.scale != scale:
            engine.close()
            raise RuntimeError(f"HDRUpscaleWithModel (B200): the model descriptor gives scale {scale}, its weights are a "
                               f"{engine.scale}x network")
        return engine

    @classmethod
    def _engine_for(cls, key, load_descriptor, device: torch.device):
        """-> (engine, scale, architecture name).  `load_descriptor()` is only called on a cache miss."""
        hit = cls._engines.get(key)
        if hit is not None:
            cls._engines.move_to_end(key)
            return hit
        descriptor = load_descriptor()
        engine = cls._new_engine(descriptor, device)
        entry = (engine, engine.scale, descriptor.architecture.name)
        cls._engines[key] = entry
        while len(cls._engines) > cls.MAX_ENGINES:
            _, (old, _, _) = cls._engines.popitem(last=False)
            old.close()
        return entry

    @classmethod
    def release_memory(cls) -> None:
        while cls._engines:
            _, (eng, _, _) = cls._engines.popitem(last=False)
            eng.close()

    def upscale(self, image, model_name, small_blur=False, local_fix=False, upscale_method="bislerp") -> Tuple[torch.Tensor]:
        device = self._compute_device(image)
        try:
            key = self._file_key(self._model_path(model_name), device)
        except ImportError:                 # no folder_paths (outside ComfyUI): nothing stable to key on, do not cache
            key = None
        if key is None:
            descriptor = self._load_model_internal(model_name)
            engine = self._new_engine(descriptor, device)
            try:
                out = engine.upscale(image, reversal_for_architecture(descriptor.architecture.name), bool(small_blur),
                                     bool(local_fix), upscale_method)
            finally:
                engine.close()
            return (out if image.device.type == "cuda" else out.to(image.device),)
        engine, _scale, arch = self._engine_for(key, lambda: self._load_model_internal(model_name), device)
        reversal = reversal_for_architecture(arch)                             # :266-279
        out = engine.upscale(image, reversal, bool(small_blur), bool(local_fix), upscale_method)
        if image.device.type != "cuda":
            out = out.to(image.device)
        return (out,)
