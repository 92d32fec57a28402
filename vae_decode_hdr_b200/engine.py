"""Host-side engine: owns one hdrvae context per (decoder weights, device) and the device workspace.

PyTorch is used for plumbing only: device memory (torch.empty), the current CUDA stream and
(in sharding.py) torch.distributed.  All arithmetic happens in libhdrvae.so.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Tuple

import torch

from . import _native as N

# hdr_vae_decode.py:48 — the enum as it is in code, in the code's order
HDR_MODES = ["conservative", "exposure", "adaptive_recovery", "mathematical_recovery"]
DEFAULT_MODE = "mathematical_recovery"
# README.md:37,78-81 / BASELINE.json names -> (code mode, smart-expansion factor); SURVEY.md §0.2
MODE_ALIASES = {"moderate": ("conservative", 3.0), "aggressive": ("mathematical_recovery", 1.0)}
_MODE_ID = {m: i for i, m in enumerate(HDR_MODES)}
_DTYPE_ID = {torch.float32: N.F32, torch.bfloat16: N.BF16, torch.float16: N.F16}
_ID_DTYPE = {v: k for k, v in _DTYPE_ID.items()}
PRECISIONS = {"fp16": N.PRECISION_F16, "bf16": N.PRECISION_BF16, "high": N.PRECISION_HIGH}


def resolve_mode(hdr_mode: str) -> Tuple[int, float]:
    """-> (mode id of include/hdrvae.h, smart-expansion factor).  The factor is 1.0 for the code names:
    simple_hdr_decode never forwards conservative_ev_multiplier (hdr_vae_decode.py:97 vs :1107)."""
    m = str(hdr_mode).lower()
    factor = 1.0
    if m in MODE_ALIASES:
        m, factor = MODE_ALIASES[m]
    if m not in _MODE_ID:
        raise ValueError(f"unknown hdr_mode {hdr_mode!r}; expected one of {HDR_MODES + list(MODE_ALIASES)}")
    return _MODE_ID[m], factor


def _require_cuda(device: torch.device) -> torch.device:
    if not torch.cuda.is_available():
        raise RuntimeError("vae_decode_hdr_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    device = torch.device(device)
    if device.type != "cuda":
        raise RuntimeError(f"vae_decode_hdr_b200 computes on CUDA devices only, got {device}")
    if device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    return device


class HdrVaeEngine:
    """One libhdrvae context: packed decoder weights + workspace on one GPU."""

    def __init__(self, state_dict: Dict[str, torch.Tensor], device="cuda", precision: str = "fp16"):
        """precision: "fp16" (default: 16-bit tensor-core operands, meets the 1e-2 image tolerance), "bf16" (same speed,
        documented 2e-2), or "high" (fp16 hi + lo split operands, 3 MMAs per product: image rel-L2 <= 1e-3 at ~3x the conv
        time; single-GPU decode only).  The residual / conv streams are fp32 in all three (include/hdrvae.h)."""
        if precision not in PRECISIONS:
            raise ValueError(f"precision must be one of {list(PRECISIONS)}")
        self.precision = precision
        self.lib = N.load_library()
        self.device = _require_cuda(device)
        self._ctx = C.c_void_p()
        N.check(self.lib.hdrvae_create(C.byref(self._ctx), self.device.index), "hdrvae_create")
        self._workspace: Optional[torch.Tensor] = None
        # the library captures the whole decode into a CUDA graph, which needs a non-default stream
        self._side = torch.cuda.Stream(device=self.device)
        self._load(state_dict)

    # -- weights -------------------------------------------------------------------------------
    def _load(self, state_dict: Dict[str, torch.Tensor]) -> None:
        keep, descs = [], []
        for name, t in state_dict.items():
            if not isinstance(t, torch.Tensor) or t.dim() == 0 or t.dim() > 4:
                continue
            if t.dtype not in _DTYPE_ID:
                t = t.float()
            t = t.detach().contiguous()
            keep.append(t)
            d = N.HdrvaeWeightDesc()
            d.name = name.encode()
            d.data = t.data_ptr()
            d.dtype = _DTYPE_ID[t.dtype]
            d.ndim = t.dim()
            for i, s in enumerate(t.shape):
                d.shape[i] = s
            descs.append(d)
        arr = (N.HdrvaeWeightDesc * len(descs))(*descs)
        with torch.cuda.device(self.device):
            torch.cuda.synchronize(self.device)
            N.check(self.lib.hdrvae_load_weights(self._ctx, arr, len(descs), PRECISIONS[self.precision]),
                    "hdrvae_load_weights")
        self.operand_dtype = _ID_DTYPE[self.lib.hdrvae_operand_dtype(self._ctx)]
        # channels of the latents this engine decodes: 16 for Flux.1, 4 for SD1.x / SDXL (post_quant_conv's input when the
        # state dict carries post_quant_conv.{weight,bias}, else conv_in's)
        self.latent_channels = self.lib.hdrvae_latent_channels(self._ctx)
        self.features_dtype = _ID_DTYPE[self.lib.hdrvae_features_dtype(self._ctx)]

    def set_conv_impl(self, impl: int) -> None:
        N.check(self.lib.hdrvae_set_conv_impl(self._ctx, impl), "hdrvae_set_conv_impl")

    def set_cta_group(self, cta_group: int) -> None:
        """0 = default (CTA pairs, tcgen05 cta_group::2), 1 = single-CTA kernel, 2 = pairs."""
        N.check(self.lib.hdrvae_set_cta_group(self._ctx, cta_group), "hdrvae_set_cta_group")

    # -- workspace -----------------------------------------------------------------------------
    def workspace_bytes(self, B: int, h: int, w: int) -> int:
        n = C.c_size_t()
        N.check(self.lib.hdrvae_workspace_bytes(self._ctx, B, h, w, C.byref(n)), "hdrvae_workspace_bytes")
        return int(n.value)

    def _ws(self, B: int, h: int, w: int) -> torch.Tensor:
        need = self.workspace_bytes(B, h, w)
        if self._workspace is None or self._workspace.numel() < need:
            self._workspace = None
            self._workspace = torch.empty(need, dtype=torch.uint8, device=self.device)
        return self._workspace

    def free_workspace(self) -> None:
        """Drop the persistent workspace (the next decode allocates it again; captured CUDA graphs stay valid only if
        the allocator returns the same block, otherwise the library re-captures)."""
        self._workspace = None

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def _check_latent(self, latent: torch.Tensor) -> Tuple[int, int, int]:
        if latent.dim() != 4 or latent.shape[1] != self.latent_channels:
            raise ValueError(f"expected a latent [B,{self.latent_channels},h,w] for this VAE, got {tuple(latent.shape)}")
        B, _, h, w = latent.shape
        if B == 0 or h == 0 or w == 0:
            raise ValueError(f"empty latent batch {tuple(latent.shape)}")
        return B, h, w

    # -- the hot path ----------------------------------------------------------------------------
    def decode(self, latent: torch.Tensor, hdr_mode: str = DEFAULT_MODE, ev_multiplier: float = 1.0,
               want_stats: bool = True, out: Optional[torch.Tensor] = None):
        """latent: float32 [B,latent_channels,h,w] on this engine's device -> (float32 [B,8h,8w,3], stats dict|None)."""
        B, h, w = self._check_latent(latent)
        mode, factor = resolve_mode(hdr_mode)
        with torch.cuda.device(self.device):
            z = latent.to(device=self.device, dtype=torch.float32).contiguous()
            ws = self._ws(B, h, w)
            if out is None:
                out = torch.empty((B, 8 * h, 8 * w, 3), dtype=torch.float32, device=self.device)
            st = N.HdrvaeStats() if want_stats else None
            cur = torch.cuda.current_stream(self.device)
            run_on = cur
            if cur.cuda_stream == 0:        # legacy default stream: hop to the engine's stream (graph capture)
                run_on = self._side
                run_on.wait_stream(cur)
                for t in (z, ws, out):
                    t.record_stream(run_on)
            N.check(self.lib.hdrvae_decode(self._ctx, z.data_ptr(), B, h, w, mode, factor, float(ev_multiplier),
                                           out.data_ptr(), C.byref(st) if want_stats else None, ws.data_ptr(),
                                           ws.numel(), run_on.cuda_stream), "hdrvae_decode")
            if run_on is not cur:
                cur.wait_stream(run_on)
        return out, (st.as_dict() if want_stats else None)

    def decode_begin_block(self, latent: torch.Tensor) -> torch.Tensor:
        """Decoder + epilogue phase A.  Returns the device-resident raw statistics block (hdrvae_raw_stats, 96 bytes)
        as a uint8 VIEW of the workspace, for the cross-rank exchange."""
        B, h, w = self._check_latent(latent)
        with torch.cuda.device(self.device):
            z = latent.to(device=self.device, dtype=torch.float32).contiguous()
            ws = self._ws(B, h, w)
            raw = C.c_void_p()
            N.check(self.lib.hdrvae_decode_begin(self._ctx, z.data_ptr(), B, h, w, ws.data_ptr(), ws.numel(),
                                                 C.byref(raw), self._stream()), "hdrvae_decode_begin")
            self._pending = (B, h, w)
            off = raw.value - ws.data_ptr()
        return ws[off:off + C.sizeof(N.HdrvaeRawStats)]

    def decode_begin(self, latent: torch.Tensor):
        """Same, returning the block as three tensor VIEWS (vmin float32[4], vmax float32[4], vsum float64[8])."""
        blk = self.decode_begin_block(latent)
        return blk[0:16].view(torch.float32), blk[16:32].view(torch.float32), blk[32:32 + 64].view(torch.float64)

    def decode_finish(self, hdr_mode: str = DEFAULT_MODE, ev_multiplier: float = 1.0, want_stats: bool = True):
        B, h, w = self._pending
        mode, factor = resolve_mode(hdr_mode)
        with torch.cuda.device(self.device):
            ws = self._ws(B, h, w)
            out = torch.empty((B, 8 * h, 8 * w, 3), dtype=torch.float32, device=self.device)
            st = N.HdrvaeStats() if want_stats else None
            N.check(self.lib.hdrvae_decode_finish(self._ctx, B, h, w, mode, factor, float(ev_multiplier),
                                                  out.data_ptr(), C.byref(st) if want_stats else None,
                                                  ws.data_ptr(), ws.numel(), self._stream()), "hdrvae_decode_finish")
        return out, (st.as_dict() if want_stats else None)

    # -- spatial row tiling (one image split over ranks): step program driven by sharding.py ----------------
    def rows_workspace_bytes(self, h: int, w: int, world: int) -> int:
        n = C.c_size_t()
        N.check(self.lib.hdrvae_rows_workspace_bytes(self._ctx, h, w, world, C.byref(n)), "hdrvae_rows_workspace_bytes")
        return int(n.value)

    def rows_begin(self, latent_full: torch.Tensor, rank: int, world: int, hdr_mode: str, ev_multiplier: float,
                   workspace: Optional[torch.Tensor] = None):
        """-> (state handle, workspace uint8 tensor, out tensor [1, 8h/world, 8w, 3])."""
        B, h, w = self._check_latent(latent_full)
        if B != 1:
            raise ValueError("row tiling decodes one image (shard batches with decode_batch_sharded)")
        if h % world:
            raise ValueError(f"latent height {h} must be a multiple of the number of ranks {world}")
        mode, factor = resolve_mode(hdr_mode)
        with torch.cuda.device(self.device):
            z = latent_full.to(device=self.device, dtype=torch.float32).contiguous()
            need = self.rows_workspace_bytes(h, w, world)
            ws = workspace if workspace is not None else torch.empty(need, dtype=torch.uint8, device=self.device)
            # `workspace` may also be a (device pointer, bytes) pair: a library-owned, IPC-shared allocation (sharding.RowsDirect)
            ws_ptr, ws_bytes = (ws if isinstance(ws, tuple) else (ws.data_ptr(), ws.numel()))
            out = torch.empty((1, 8 * h // world, 8 * w, 3), dtype=torch.float32, device=self.device)
            state = C.c_void_p()
            N.check(self.lib.hdrvae_rows_begin(self._ctx, z.data_ptr(), h, w, rank, world, mode, factor, float(ev_multiplier),
                                               out.data_ptr(), ws_ptr, ws_bytes, C.byref(state)), "hdrvae_rows_begin")
        return state, ws, out, z

    def rows_run(self, state) -> "N.HdrvaeExchange":
        ex = N.HdrvaeExchange()
        with torch.cuda.device(self.device):
            N.check(self.lib.hdrvae_rows_run(state, C.byref(ex), self._stream()), "hdrvae_rows_run")
        return ex

    def rows_end(self, state, want_stats: bool = True):
        st = N.HdrvaeStats() if want_stats else None
        with torch.cuda.device(self.device):
            N.check(self.lib.hdrvae_rows_end(state, C.byref(st) if want_stats else None, self._stream()), "hdrvae_rows_end")
        return st.as_dict() if want_stats else None

    def decode_features(self, latent: torch.Tensor) -> torch.Tensor:
        """Decoder only -> NHWC [B,8h,8w,128] in the operand dtype (fp16 by default) = the tensor the reference's
        hook captures (:850-855)."""
        B, h, w = self._check_latent(latent)
        with torch.cuda.device(self.device):
            z = latent.to(device=self.device, dtype=torch.float32).contiguous()
            ws = self._ws(B, h, w)
            feat = torch.empty((B, 8 * h, 8 * w, 128), dtype=self.features_dtype, device=self.device)
            N.check(self.lib.hdrvae_decode_features(self._ctx, z.data_ptr(), B, h, w, feat.data_ptr(), ws.data_ptr(),
                                                    ws.numel(), self._stream()), "hdrvae_decode_features")
        return feat

    # -- fused epilogue on caller activations -------------------------------------------------------
    def epilogue(self, pre_nhwc: torch.Tensor, conv_w: torch.Tensor, conv_b: torch.Tensor,
                 hdr_mode: str = DEFAULT_MODE, ev_multiplier: float = 1.0, debug: bool = False):
        """pre_nhwc: [B,H,W,128] float32 or bfloat16 on device.  -> (image, stats[, post3, pre3, argmax3])."""
        if pre_nhwc.dim() != 4 or pre_nhwc.shape[-1] != 128:
            raise ValueError(f"expected activations [B,H,W,128], got {tuple(pre_nhwc.shape)}")
        if pre_nhwc.dtype not in _DTYPE_ID:
            raise ValueError("activations must be float32, float16 or bfloat16")
        B, H, W, _ = pre_nhwc.shape
        if B == 0 or H == 0 or W == 0:
            raise ValueError("empty activation batch")
        mode, factor = resolve_mode(hdr_mode)
        with torch.cuda.device(self.device):
            pre = pre_nhwc.to(self.device).contiguous()
            cw = conv_w.to(self.device, torch.float32).contiguous()
            cb = conv_b.to(self.device, torch.float32).contiguous()
            n = C.c_size_t()
            N.check(self.lib.hdrvae_epilogue_scratch_bytes(B, H, W, C.byref(n)), "hdrvae_epilogue_scratch_bytes")
            scratch = torch.empty(n.value, dtype=torch.uint8, device=self.device)
            out = torch.empty((B, H, W, 3), dtype=torch.float32, device=self.device)
            post3 = pre3 = am3 = None
            if debug:
                post3 = torch.empty_like(out)
                pre3 = torch.empty_like(out)
                am3 = torch.empty((B, H, W, 3), dtype=torch.int32, device=self.device)
            st = N.HdrvaeStats()
            N.check(self.lib.hdrvae_epilogue(
                self._ctx, pre.data_ptr(), _DTYPE_ID[pre.dtype], B, H, W, cw.data_ptr(), cb.data_ptr(), mode, factor,
                float(ev_multiplier), out.data_ptr(), C.byref(st), post3.data_ptr() if debug else None,
                pre3.data_ptr() if debug else None, am3.data_ptr() if debug else None, scratch.data_ptr(),
                scratch.numel(), self._stream()), "hdrvae_epilogue")
        if debug:
            return out, st.as_dict(), post3, pre3, am3
        return out, st.as_dict()

    # -- kernel-level entry points (unit parity tests) ------------------------------------------------
    def conv2d(self, x_nhwc: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor], ksize: int,
               upsample2x: bool = False, residual: Optional[torch.Tensor] = None, out_dtype=torch.float32,
               round_tf32: bool = False, want_stats: bool = False, impl: int = N.CONV_TCGEN05, *,
               cin: Optional[int] = None, x_chan_off: int = 0, out: Optional[torch.Tensor] = None, out_chan_off: int = 0,
               out2: Optional[torch.Tensor] = None, out2_chan_off: Optional[int] = None, out2_scale: float = 1.0,
               residual2: Optional[torch.Tensor] = None, res_scale: float = 1.0, lrelu: float = 0.0,
               prelu: Optional[torch.Tensor] = None, act: int = N.ACT_NONE):
        """x_nhwc dtype selects the MMA kind: float16/bfloat16 -> kind::f16, float32 -> kind::tf32.

        The keyword arguments are the upscalers' conv features (include/hdrvae.h, hdrvae_conv_extra):
          cin / x_chan_off: the conv reads channels [x_chan_off, x_chan_off + cin) of x_nhwc [B,H,W,X] (X is the pixel
                           stride); without cin it reads all of them, densely;
          out / out_chan_off: write round_up(Cout, 4) channels from out_chan_off on into this device tensor
                           [B,OH,OW,Y] (its dtype is the output's) and return it; residual / residual2 share its layout;
          out2 / out2_chan_off / out2_scale: second, 16-bit output y * out2_scale into a slice of out2 [B,OH,OW,Y2]
                           (without out2_chan_off, out2 has y's pixel stride and channel offset);
          residual2 (float32), res_scale: t = conv + bias + res_scale * residual + residual2;
          lrelu, prelu (Cout slopes), act (N.ACT_SILU / N.ACT_GATE): the activation of t.
        The device tensors given here are used in place (no copies), so they may alias one another as in the upscalers."""
        B, H, W, xc = x_nhwc.shape
        cout = weight.shape[0]
        OH, OW = (2 * H, 2 * W) if upsample2x else (H, W)
        sliced = cin is not None
        cin = xc if cin is None else cin
        if not 0 <= x_chan_off <= xc - cin:
            raise ValueError(f"channels [{x_chan_off}, {x_chan_off + cin}) lie outside x's {xc}")
        for name, t in (("x_nhwc", x_nhwc if sliced else None), ("out", out), ("out2", out2), ("residual2", residual2),
                        ("residual", residual if out is not None else None), ("prelu", prelu)):
            if t is not None and (t.device != self.device or not t.is_contiguous()):
                raise ValueError(f"{name} must be a contiguous tensor on {self.device} when used in place")
        ext = N.HdrvaeConvExtra()
        if sliced:
            ext.x_channels = xc
        if out is not None:
            if tuple(out.shape[:3]) != (B, OH, OW):
                raise ValueError(f"out {tuple(out.shape)} does not match the output grid {(B, OH, OW)}")
            ext.y_channels, ext.y_chan_off = out.shape[3], out_chan_off
        if out2 is not None:
            if tuple(out2.shape[:3]) != (B, OH, OW):
                raise ValueError(f"out2 {tuple(out2.shape)} does not match the output grid {(B, OH, OW)}")
            ext.y2, ext.y2_dtype, ext.y2_scale = out2.data_ptr(), _DTYPE_ID[out2.dtype], out2_scale
            if out2_chan_off is not None:
                ext.y2_channels, ext.y2_chan_off = out2.shape[3], out2_chan_off
            elif out2.shape[3] != (out.shape[3] if out is not None else cout):
                raise ValueError("out2 without out2_chan_off must have y's pixel stride")
        if residual2 is not None:
            if residual2.dtype != torch.float32:
                raise ValueError("residual2 must be float32")
            ext.residual2 = residual2.data_ptr()
        if prelu is not None:
            if prelu.dtype != torch.float32 or prelu.numel() != cout:
                raise ValueError(f"prelu must hold {cout} float32 slopes")
            ext.act_slope = prelu.data_ptr()
        ext.res_scale, ext.lrelu, ext.act = res_scale, lrelu, act
        with torch.cuda.device(self.device):
            x = x_nhwc if sliced else x_nhwc.to(self.device).contiguous()
            wt = weight.to(self.device, torch.float32).contiguous()
            bs = bias.to(self.device, torch.float32).contiguous() if bias is not None else None
            rs = residual if out is not None or residual is None else residual.to(self.device).contiguous()
            y = out if out is not None else torch.empty((B, OH, OW, cout), dtype=out_dtype, device=self.device)
            chunks = self.lib.hdrvae_conv2d_stats_chunks(H, W, int(upsample2x))
            part = torch.zeros((B, chunks, 32, 2), dtype=torch.float32, device=self.device) if want_stats else None
            nch = C.c_int(0)
            N.check(self.lib.hdrvae_conv2d(
                self._ctx, x.data_ptr() + x_chan_off * x.element_size(), _DTYPE_ID[x.dtype], B, H, W, cin, wt.data_ptr(),
                bs.data_ptr() if bs is not None else None, cout, ksize, int(upsample2x),
                rs.data_ptr() if rs is not None else None, _DTYPE_ID[rs.dtype] if rs is not None else 0, y.data_ptr(),
                _DTYPE_ID[y.dtype], int(round_tf32), part.data_ptr() if want_stats else None, C.byref(nch), impl,
                self._stream(), C.byref(ext)), "hdrvae_conv2d")
        if want_stats:      # the library packs the partials with the chunk count it actually used (<= the capacity asked for)
            part = part.flatten()[:B * nch.value * 64].view(B, nch.value, 32, 2)
        return (y, part) if want_stats else y

    def groupnorm_silu(self, x_nhwc: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, silu: bool = True,
                       out_dtype=torch.float16, partials: Optional[torch.Tensor] = None):
        B, H, W, Cc = x_nhwc.shape
        with torch.cuda.device(self.device):
            x = x_nhwc.to(self.device).contiguous()
            g = gamma.to(self.device, torch.float32).contiguous()
            b = beta.to(self.device, torch.float32).contiguous()
            y = torch.empty(x.shape, dtype=out_dtype, device=self.device)
            N.check(self.lib.hdrvae_groupnorm_silu(
                self._ctx, x.data_ptr(), _DTYPE_ID[x.dtype], B, H * W, Cc, g.data_ptr(), b.data_ptr(), int(silu),
                y.data_ptr(), _DTYPE_ID[out_dtype], partials.data_ptr() if partials is not None else None,
                partials.shape[1] if partials is not None else 0, self._stream()), "hdrvae_groupnorm_silu")
        return y

    def attention(self, q: torch.Tensor, k: torch.Tensor, v: torch.Tensor) -> torch.Tensor:
        B, T, d = q.shape
        assert d == 512 and q.dtype in (torch.float16, torch.bfloat16)
        with torch.cuda.device(self.device):
            q, k, v = (t.to(self.device, q.dtype).contiguous() for t in (q, k, v))
            o = torch.empty_like(q)
            N.check(self.lib.hdrvae_attention(self._ctx, q.data_ptr(), k.data_ptr(), v.data_ptr(), _DTYPE_ID[q.dtype], B, T,
                                              o.data_ptr(), self._stream()), "hdrvae_attention")
        return o

    def close(self) -> None:
        if getattr(self, "_ctx", None) is not None and self._ctx.value:
            self.lib.hdrvae_destroy(self._ctx)
            self._ctx = C.c_void_p()
        self._workspace = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def quantiles(x: torch.Tensor, qs) -> list:
    """Exact quantiles (lower interpolation = order statistic of rank floor(q*(n-1))) of a CUDA float32 tensor by
    radix select on the GPU; == torch.quantile(x.flatten(), q, interpolation="lower"), bit-exact."""
    lib = N.load_library()
    dev = _require_cuda(x.device)
    qs = [float(q) for q in qs]
    if not 1 <= len(qs) <= 8:
        raise ValueError("1..8 quantiles")
    if x.numel() == 0:
        raise ValueError("quantiles of an empty tensor")
    with torch.cuda.device(dev):
        xf = x.to(torch.float32).contiguous()
        qa = (C.c_double * len(qs))(*qs)
        out = (C.c_float * len(qs))()
        N.check(lib.hdrvae_quantiles(xf.data_ptr(), xf.numel(), qa, len(qs), out,
                                     torch.cuda.current_stream(dev).cuda_stream), "hdrvae_quantiles")
    return [float(v) for v in out]


def pack_half(image_bhwc: torch.Tensor, exr_scanline_order: bool = False) -> torch.Tensor:
    """float32 [B,H,W,3] on a CUDA device -> float16 bits (RNE, overflow -> inf), as
    ndarray.astype(np.float16) in linear_exr_export.py:155,165.  exr_scanline_order: per image row the
    B, G, R planes ([B,H,3,W]) instead of interleaved RGB."""
    lib = N.load_library()
    dev = _require_cuda(image_bhwc.device)
    if image_bhwc.dim() != 4 or image_bhwc.shape[-1] != 3:
        raise ValueError(f"expected IMAGE [B,H,W,3], got {tuple(image_bhwc.shape)}")
    B, H, W, _ = image_bhwc.shape
    with torch.cuda.device(dev):
        img = image_bhwc.to(torch.float32).contiguous()
        shape = (B, H, 3, W) if exr_scanline_order else (B, H, W, 3)
        out = torch.empty(shape, dtype=torch.float16, device=dev)
        if img.numel():
            N.check(lib.hdrvae_pack_half(img.data_ptr(), B, H, W, int(exr_scanline_order), out.data_ptr(),
                                         torch.cuda.current_stream(dev).cuda_stream), "hdrvae_pack_half")
    return out
