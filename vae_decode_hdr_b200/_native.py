"""ctypes binding of libhdrvae.so (include/hdrvae.h) — the only road from Python to the kernels.

This is the stub a maintainer of the reference would add next to hdr_vae_decode.py
(see INTEGRATION.md).  There is no CPU path: if the library is missing or no B200 is
visible, every entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import Dict

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libhdrvae.so")
CSRC_DIR = os.path.join(_HERE, "csrc")

MODE_CONSERVATIVE, MODE_EXPOSURE, MODE_ADAPTIVE_RECOVERY, MODE_MATHEMATICAL_RECOVERY = range(4)
NORM_NONE, NORM_SIGMOID, NORM_TANH = range(3)
F32, BF16, F16 = range(3)
PRECISION_BF16, PRECISION_F16, PRECISION_HIGH = 0, 1, 2
CONV_TCGEN05, CONV_DIRECT = 0, 1
RAW_NMIN, RAW_NMAX, RAW_NSUM = 4, 4, 8
ACT_NONE, ACT_SILU, ACT_GATE = range(3)
ABI_VERSION = 2


class HdrvaeStats(C.Structure):
    _fields_ = [(n, C.c_double) for n in (
        "pre_min", "pre_max", "pre_mean", "pre_std", "post_min", "post_max", "post_mean", "post_std",
        "conv_min", "conv_max", "conv_mean", "pre3_min", "pre3_max", "rec_min", "rec_max", "aligned_max",
        "out_min", "out_max")] + [(n, C.c_int64) for n in (
        "hdr_pixels", "negative_pixels", "highlight_count", "intelligent_hdr_pixels")] + [
        ("intelligent_max", C.c_double), ("norm_function", C.c_int32), ("has_hdr", C.c_int32),
        ("accepted", C.c_int32), ("reserved", C.c_int32)]

    def as_dict(self) -> Dict:
        return {n: getattr(self, n) for n, _ in self._fields_ if n != "reserved"}


class HdrvaeWeightDesc(C.Structure):
    _fields_ = [("name", C.c_char_p), ("data", C.c_void_p), ("dtype", C.c_int32), ("ndim", C.c_int32),
                ("shape", C.c_int64 * 4)]


class HdrvaeExchange(C.Structure):
    _fields_ = [("kind", C.c_int32), ("n_halo", C.c_int32),
                ("halo_first_row_off", C.c_uint64 * 2), ("halo_last_row_off", C.c_uint64 * 2),
                ("halo_top_off", C.c_uint64 * 2), ("halo_bottom_off", C.c_uint64 * 2), ("halo_row_bytes", C.c_uint64 * 2),
                ("allreduce_off", C.c_uint64), ("allreduce_count", C.c_uint64),
                ("n_gather", C.c_int32), ("reserved", C.c_int32),
                ("gather_off", C.c_uint64 * 2), ("gather_bytes_per_rank", C.c_uint64 * 2), ("raw_stats_off", C.c_uint64)]


EX_END, EX_HALO, EX_ALLREDUCE_F64, EX_ALLGATHER, EX_RAW_STATS = 0, 1, 2, 4, 8


class HdrvaeIpcHandle(C.Structure):
    _fields_ = [("bytes", C.c_ubyte * 64)]


class HdrvaeRawStats(C.Structure):
    _fields_ = [("vmin", C.c_float * RAW_NMIN), ("vmax", C.c_float * RAW_NMAX), ("vsum", C.c_double * RAW_NSUM)]


class HdrvaeConvExtra(C.Structure):
    _fields_ = [("x_channels", C.c_int32), ("y_channels", C.c_int32), ("y_chan_off", C.c_int32), ("y2_dtype", C.c_int32),
                ("y2", C.c_void_p), ("y2_scale", C.c_float), ("y2_channels", C.c_int32), ("y2_chan_off", C.c_int32),
                ("res_scale", C.c_float), ("residual2", C.c_void_p), ("act_slope", C.c_void_p), ("lrelu", C.c_float),
                ("act", C.c_int32)]


# every symbol include/hdrvae.h declares: name -> (restype, argtypes)
_vp, _i, _f, _sz = C.c_void_p, C.c_int, C.c_float, C.c_size_t
SIGNATURES = {
    "hdrvae_last_error": (C.c_char_p, []),
    "hdrvae_abi_version": (_i, []),
    "hdrvae_create": (_i, [C.POINTER(_vp), _i]),
    "hdrvae_destroy": (_i, [_vp]),
    "hdrvae_set_conv_impl": (_i, [_vp, _i]),
    "hdrvae_launch_count": (C.c_longlong, []),
    "hdrvae_profile_begin": (_i, []),
    "hdrvae_profile_end": (_i, [C.c_char_p]),
    "hdrvae_load_weights": (_i, [_vp, C.POINTER(HdrvaeWeightDesc), _i, _i]),
    "hdrvae_latent_channels": (_i, [_vp]),
    "hdrvae_workspace_bytes": (_i, [_vp, _i, _i, _i, C.POINTER(_sz)]),
    "hdrvae_decode": (_i, [_vp, _vp, _i, _i, _i, _i, _f, _f, _vp, C.POINTER(HdrvaeStats), _vp, _sz, _vp]),
    "hdrvae_decode_begin": (_i, [_vp, _vp, _i, _i, _i, _vp, _sz, C.POINTER(_vp), _vp]),
    "hdrvae_decode_finish": (_i, [_vp, _i, _i, _i, _i, _f, _f, _vp, C.POINTER(HdrvaeStats), _vp, _sz, _vp]),
    "hdrvae_raw_stats_merge": (_i, [_vp, _i, _vp, _vp]),
    "hdrvae_rows_workspace_bytes": (_i, [_vp, _i, _i, _i, C.POINTER(_sz)]),
    "hdrvae_rows_begin": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _f, _f, _vp, _vp, _sz, C.POINTER(_vp)]),
    "hdrvae_rows_run": (_i, [_vp, C.POINTER(HdrvaeExchange), _vp]),
    "hdrvae_rows_end": (_i, [_vp, C.POINTER(HdrvaeStats), _vp]),
    "hdrvae_peer_alloc": (_i, [_vp, _sz, C.POINTER(_vp), C.POINTER(HdrvaeIpcHandle)]),
    "hdrvae_peer_open": (_i, [_vp, C.POINTER(HdrvaeIpcHandle), C.POINTER(_vp)]),
    "hdrvae_peer_close": (_i, [_vp, _vp]),
    "hdrvae_peer_free": (_i, [_vp, _vp]),
    "hdrvae_rows_set_peers": (_i, [_vp, C.POINTER(_vp), _i]),
    "hdrvae_rows_run_direct": (_i, [_vp, _vp]),
    "hdrvae_decode_features": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _sz, _vp]),
    "hdrvae_epilogue_scratch_bytes": (_i, [_i, _i, _i, C.POINTER(_sz)]),
    "hdrvae_epilogue": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp, _i, _f, _f, _vp, C.POINTER(HdrvaeStats),
                             _vp, _vp, _vp, _vp, _sz, _vp]),
    "hdrvae_operand_dtype": (_i, [_vp]),
    "hdrvae_features_dtype": (_i, [_vp]),
    "hdrvae_set_cta_group": (_i, [_vp, _i]),
    "hdrvae_conv2d": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _i, _i, _i, _vp, _i, _vp, _i, _i, _vp,
                           C.POINTER(_i), _i, _vp, C.POINTER(HdrvaeConvExtra)]),
    "hdrvae_conv2d_stats_chunks": (_i, [_i, _i, _i]),
    "hdrvae_groupnorm_silu": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp, _i, _vp, _i, _vp, _i, _vp]),
    "hdrvae_attention": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp]),
    "hdrvae_quantiles": (_i, [_vp, C.c_longlong, C.POINTER(C.c_double), _i, C.POINTER(C.c_float), _vp]),
    "hdrvae_pack_half": (_i, [_vp, _i, _i, _i, _i, _vp, _vp]),
    "hdrvae_upscaler_create": (_i, [_vp, C.POINTER(_vp)]),
    "hdrvae_upscaler_destroy": (_i, [_vp]),
    "hdrvae_upscaler_load_weights": (_i, [_vp, C.POINTER(HdrvaeWeightDesc), _i]),
    "hdrvae_upscaler_blocks": (_i, [_vp]),
    "hdrvae_upscaler_scale": (_i, [_vp]),
    "hdrvae_upscaler_forward_bytes": (_i, [_vp, _i, _i, _i, C.POINTER(_sz)]),
    "hdrvae_upscaler_forward": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp, _sz, _vp]),
    "hdrvae_upscale_workspace_bytes": (_i, [_vp, _i, _i, _i, C.POINTER(_sz)]),
    "hdrvae_upscale": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _sz, _vp]),
}
REVERSAL_NONE, REVERSAL_ATANH, REVERSAL_LOGIT = 0, 1, 2
UPSCALE_METHODS = {"nearest-exact": 0, "bilinear": 1, "area": 2, "bicubic": 3, "bislerp": 4}

_lib = None


def build_library(force: bool = False) -> str:
    """Compile libhdrvae.so in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    if force:
        subprocess.run(["make", "-C", CSRC_DIR, "clean"], check=True, capture_output=True)
    r = subprocess.run(["make", "-C", CSRC_DIR, "-j8"], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("building libhdrvae.so failed:\n" + r.stdout[-4000:] + r.stderr[-4000:])
    return LIB_PATH


def load_library() -> C.CDLL:
    """dlopen libhdrvae.so and bind every declared symbol; raises if it is missing (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `make -C {CSRC_DIR}` (or __graft_entry__.build()); "
            "vae_decode_hdr_b200 has no CPU or PyTorch fallback")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)       # AttributeError if the .so lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    if lib.hdrvae_abi_version() != ABI_VERSION:
        raise RuntimeError("libhdrvae.so ABI version mismatch")
    _lib = lib
    return lib


def last_error() -> str:
    return load_library().hdrvae_last_error().decode("utf-8", "replace")


def check(rc: int, what: str) -> None:
    if rc != 0:
        raise RuntimeError(f"{what} failed ({rc}): {last_error()}")
