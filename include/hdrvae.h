/*
 * hdrvae.h — C ABI of libhdrvae.so: the B200 (sm_100a) HDR decode path for Flux.1 and SD1.x / SDXL VAEs.
 *
 * The reference (netocg/vae-decode-hdr) has no native code and no FFI: the whole
 * path is PyTorch eager driven from hdr_vae_decode.py.  Each entry point below
 * names the reference interface it replaces (file:line in /root/reference).  The
 * reference-side binding a maintainer would add is the ctypes stub shown in
 * INTEGRATION.md (vae_decode_hdr_b200/_native.py is that stub).
 *
 * Conventions
 *   - plain C types only; every function returns 0 on success, <0 on error and
 *     records a message retrievable with hdrvae_last_error() (thread local).
 *     The Python host raises RuntimeError; there is NO CPU fallback.
 *   - device pointers are raw CUDA pointers owned by the caller (PyTorch
 *     allocations).  The library owns only what lives inside an hdrvae_ctx.
 *   - all work is enqueued on the caller's stream (cudaStream_t passed as void*);
 *     no hidden host threads.  Functions that fill a host-side hdrvae_stats
 *     synchronise that stream once at the end; pass stats == NULL to stay async.
 *   - activations inside the library are NHWC bf16; the boundary tensors keep the
 *     reference layouts: latent float32 NCHW in, IMAGE float32 BHWC out
 *     (hdr_vae_decode.py:78 and :195,:354).
 */
#ifndef HDRVAE_H_
#define HDRVAE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HDRVAE_ABI_VERSION 2

typedef struct hdrvae_ctx hdrvae_ctx;

/* hdr_mode enum as it is in code, same order (hdr_vae_decode.py:48). */
enum {
  HDRVAE_MODE_CONSERVATIVE = 0,          /* smart_hdr_expansion        :941-980  */
  HDRVAE_MODE_EXPOSURE = 1,              /* exposure_based_hdr         :982-1007 */
  HDRVAE_MODE_ADAPTIVE_RECOVERY = 2,     /* adaptive branch            :1114-1147 */
  HDRVAE_MODE_MATHEMATICAL_RECOVERY = 3  /* mathematical branch        :1149-1159 */
};

/* Normalisation detected by analyze_conv_out (hdr_vae_decode.py:890-897). */
enum { HDRVAE_NORM_NONE = 0, HDRVAE_NORM_SIGMOID = 1, HDRVAE_NORM_TANH = 2 };

/* element types for hdrvae_weight_desc / activations handed across the ABI */
enum { HDRVAE_F32 = 0, HDRVAE_BF16 = 1, HDRVAE_F16 = 2 };

/* 16-bit tensor-core operand type of the decoder (kind::f16, fp32 accumulate in TMEM).  In both modes the
 * un-normalised residual / conv streams stay fp32 in HBM; the convs that read them directly get a 16-bit
 * copy scaled by 2^-4 from the producing conv's epilogue.
 *   F16  (default): fp16 operands (GroupNorm outputs, weights, attention operands are bounded) — meets the
 *                   1e-2 end-to-end tolerance;
 *   BF16          : bf16 operands, same speed, ~8x larger operand rounding (DESIGN.md "Precision");
 *   HIGH          : every tensor-core operand as an fp16 hi + lo pair (x = hi + lo to ~2^-22): the K dimension of every
 *                   GEMM-shaped op is the concatenation [hi | lo | hi] x [hi | hi | lo], i.e. 3 MMAs per product, fp32
 *                   accumulation; features and conv_out in fp32.  Meets rel-L2 <= 1e-3 on the image (BASELINE.json's
 *                   "TF32 path at <= 1e-3": tf32 itself has fp16's 10-bit mantissa and cannot) at ~3x the conv time.
 *                   Single-GPU decode only (no row tiling). */
enum { HDRVAE_PRECISION_BF16 = 0, HDRVAE_PRECISION_F16 = 1, HDRVAE_PRECISION_HIGH = 2 };

/* conv implementation selector (debug/validation): the tcgen05 implicit-GEMM
 * kernel is the product path; the CUDA-core direct kernel exists to validate it
 * on the GPU and is never selected implicitly. */
enum { HDRVAE_CONV_TCGEN05 = 0, HDRVAE_CONV_DIRECT = 1 };
/* Upscaler: reversal hook kinds (hdr_upscale_with_model.py:79-107, :266-279) and the resampling methods of
 * local_fix (:241; the torch-expressible ones and ComfyUI's own "bislerp"). */
enum { HDRVAE_REVERSAL_NONE = 0, HDRVAE_REVERSAL_ATANH = 1, HDRVAE_REVERSAL_LOGIT = 2 };
enum { HDRVAE_UPSCALE_NEAREST_EXACT = 0, HDRVAE_UPSCALE_BILINEAR = 1, HDRVAE_UPSCALE_AREA = 2, HDRVAE_UPSCALE_BICUBIC = 3,
       HDRVAE_UPSCALE_BISLERP = 4 /* ComfyUI's spherical-linear resampler, the node's default (hdr_upscale_with_model.py:65) */ };

/*
 * Scalars the reference computes with ~25 full-tensor reductions + host syncs
 * (hdr_vae_decode.py:862-879, 1063-1066, 100-102, 188-191); here they come out
 * of the fused epilogue in one struct.  "pre" = input of decoder.conv_out
 * ([B,128,H,W]), "post" = clamp((conv_out+1)/2,0,1), "conv" = conv_out only,
 * "pre3" = 128->3 channel MAX-pool, "rec" = logit/atanh recovered map.
 */
typedef struct hdrvae_stats {
  double pre_min, pre_max, pre_mean, pre_std;     /* :862-865 (std unbiased) */
  double post_min, post_max, post_mean, post_std; /* :867-870 */
  double conv_min, conv_max, conv_mean;           /* :877-879 */
  double pre3_min, pre3_max;                      /* :1065-1066 */
  double rec_min, rec_max;                        /* :1098 */
  double aligned_max;                             /* :1116 (adaptive mode; else NaN) */
  double out_min, out_max;                        /* :188-189 */
  int64_t hdr_pixels;                             /* :190  sum(out > 1.0) */
  int64_t negative_pixels;                        /* :191  sum(out < 0.0) */
  int64_t highlight_count;                        /* :961  sum(pre3 > 1.0) */
  int64_t intelligent_hdr_pixels;                 /* :100  sum(decoded > 1.0) before the multiplier */
  double intelligent_max;                         /* :102 */
  int32_t norm_function;                          /* HDRVAE_NORM_* :890-897 */
  int32_t has_hdr;                                /* :1078 pre3_max > 1.001 */
  int32_t accepted;                               /* :106  hdr_pixels>0 || max>1.1 (0 => reference would bypass) */
  int32_t reserved;
} hdrvae_stats;

/* One tensor of vae.first_stage_model.decoder.state_dict() (hdr_vae_decode.py:842):
 * name is the state-dict key ("up.1.block.0.nin_shortcut.weight", ...), data a
 * host or device pointer to a contiguous tensor of `dtype`. */
typedef struct hdrvae_weight_desc {
  const char* name;
  const void* data;
  int32_t dtype;      /* HDRVAE_F32 / HDRVAE_BF16 / HDRVAE_F16 */
  int32_t ndim;
  int64_t shape[4];
} hdrvae_weight_desc;

/* Raw, all-reducible statistics block between epilogue phase A and phase B
 * (multi-GPU batch sharding: MIN-, MAX- and SUM-reduce the three arrays across
 * ranks; SURVEY.md §0.7 / §8e). */
#define HDRVAE_RAW_NMIN 4
#define HDRVAE_RAW_NMAX 4
#define HDRVAE_RAW_NSUM 8
typedef struct hdrvae_raw_stats {
  float vmin[HDRVAE_RAW_NMIN];   /* pre, post, conv, pre3 */
  float vmax[HDRVAE_RAW_NMAX];   /* pre, post, conv, pre3 */
  double vsum[HDRVAE_RAW_NSUM];  /* pre Σx, pre Σx², post Σx, post Σx², conv Σx, n_pre, n_post, highlight_count */
} hdrvae_raw_stats;

const char* hdrvae_last_error(void);
int hdrvae_abi_version(void);

/* ---- context ------------------------------------------------------------- */
int hdrvae_create(hdrvae_ctx** out, int device);
int hdrvae_destroy(hdrvae_ctx* ctx);
/* HDRVAE_CONV_TCGEN05 (default) or HDRVAE_CONV_DIRECT (validation only; also env HDRVAE_CONV_IMPL=direct). */
int hdrvae_set_conv_impl(hdrvae_ctx* ctx, int impl);
/* HDRVAE_F16 or HDRVAE_BF16: element type of hdrvae_decode_features' output (set by hdrvae_load_weights). */
int hdrvae_operand_dtype(hdrvae_ctx* ctx);
/* element type of the tensor hdrvae_decode_features returns: the operand type, or HDRVAE_F32 in the HIGH precision mode */
int hdrvae_features_dtype(hdrvae_ctx* ctx);
/* tcgen05 cta_group of the GEMM/conv kernel: 0 = default (2: CTA pairs, M = 256 MMAs), 1 = single CTAs, 2 = pairs. */
int hdrvae_set_cta_group(hdrvae_ctx* ctx, int cta_group);

/* Diagnostics: per-op CUDA-event timing of everything the library launches between begin and end
 * (the reference's only instrumentation is logging with host syncs, hdr_vae_decode.py:81-84,188-193). */
long long hdrvae_launch_count(void);   /* kernels launched by the library so far (process-wide) */
int hdrvae_profile_begin(void);
int hdrvae_profile_end(const char* path_or_null);

/* Replaces the reference's reads of vae.first_stage_model.decoder.* modules
 * (hdr_vae_decode.py:448,505-516,842,855,876): one-time repack of the state
 * dict into K-major bf16 GEMM operands (3x3 taps, upsample phase weights,
 * fused q/k/v) owned by the context.
 * The decoder's latent channel count C_z is the input-channel count of conv_in.weight (Flux.1: 16, SD1.x / SDXL: 4;
 * 1..64).  Optionally the descriptors "post_quant_conv.weight" [C_z, C_lat, 1, 1] and "post_quant_conv.bias" [C_z]
 * (both or neither; 1 <= C_lat <= 64): the 1x1 conv of vae.first_stage_model that SD-family AutoencoderKL applies to the
 * latent before the decoder.  The decode entry points then take latents of C_lat channels and apply it first. */
int hdrvae_load_weights(hdrvae_ctx* ctx, const hdrvae_weight_desc* descs, int n, int precision);

/* Channels C_lat of the latents the decode entry points take (post_quant_conv's input channels, else conv_in's):
 * 16 for Flux.1, 4 for SD1.x / SDXL.  <0 before hdrvae_load_weights succeeded. */
int hdrvae_latent_channels(const hdrvae_ctx* ctx);

/* Bytes of caller-provided device workspace hdrvae_decode needs for a latent
 * batch [B,C_lat,h,w].  The workspace pointer must be 256-byte aligned (what
 * cudaMalloc and torch's allocator return). */
int hdrvae_workspace_bytes(hdrvae_ctx* ctx, int B, int h, int w, size_t* bytes);

/* ---- the hot path ---------------------------------------------------------
 * Replaces HDRVAEDecode.simple_hdr_decode's happy path (hdr_vae_decode.py:62-195):
 * analyze_conv_out (:837) + intelligent_hdr_decode (:1009) + multiplier (:180) +
 * _format_tensor passthrough (:209-212,:354), with ONE decoder pass.
 *   latent_nchw : device float32 [B,C_lat,h,w]         (:78; C_lat = hdrvae_latent_channels)
 *   out_bhwc    : device float32 [B,8h,8w,3] contiguous (:195)
 *   expansion_factor : smart_hdr_expansion factor (1.0 for "conservative" as the
 *                 reference calls it, 3.0 for the README "moderate" alias)
 *   ev_multiplier    : conservative_ev_multiplier (:180-182)
 */
int hdrvae_decode(hdrvae_ctx* ctx, const float* latent_nchw, int B, int h, int w, int mode,
                  float expansion_factor, float ev_multiplier, float* out_bhwc,
                  hdrvae_stats* stats, void* workspace, size_t workspace_bytes, void* stream);

/* Same path split around the batch-global scalars for multi-GPU batch sharding
 * (SURVEY.md §8e): begin = decoder + epilogue phase A, leaves a device-resident
 * hdrvae_raw_stats at *raw_stats_dev (inside the workspace) that the host
 * all-reduces; finish = scalar finalisation + phase B. */
int hdrvae_decode_begin(hdrvae_ctx* ctx, const float* latent_nchw, int B, int h, int w,
                        void* workspace, size_t workspace_bytes, void** raw_stats_dev, void* stream);
int hdrvae_decode_finish(hdrvae_ctx* ctx, int B, int h, int w, int mode, float expansion_factor,
                         float ev_multiplier, float* out_bhwc, hdrvae_stats* stats, void* workspace,
                         size_t workspace_bytes, void* stream);

/* Batch sharding, the exchange step: merge `n` gathered hdrvae_raw_stats blocks (device memory, 96 bytes each, rank
 * order — the result of ONE all-gather of every rank's block) into *dst (device; must not alias `blocks`), MIN / MAX /
 * SUM in rank order, so every rank derives bit-identical batch-global statistics (hdr_vae_decode.py:862-865,1098,1116
 * take them over the whole batch tensor). */
int hdrvae_raw_stats_merge(const void* blocks, int n, void* dst, void* stream);

/* ---- spatial row tiling across GPUs (BASELINE config C4; SURVEY.md 8e) --------------------------------------
 * One image, latent rows split evenly over `world` ranks (h % world == 0).  Every rank runs the same step
 * program on its slab; between steps the HOST performs the exchange the library describes (NCCL in
 * vae_decode_hdr_b200/sharding.py, plain copies when ranks are emulated in one process):
 *   HALO      : the first / last interior row of up to two conv outputs goes to the upper / lower neighbour's halo row
 *               (33 of these per decode, one per 3x3-conv input);
 *   ALLREDUCE : SUM of `allreduce_count` doubles = the GroupNorm (sum, sum of squares) of every (image, group), so
 *               that tiling does not change the normalisation;
 *   ALLGATHER : in-place all-gather of `gather_bytes_per_rank` bytes per rank (attention K and V: mid.attn_1 is global);
 *   RAW_STATS : MIN/MAX/SUM all-reduce of the hdrvae_raw_stats block (batch-global HDR statistics).
 * All offsets are byte offsets into the rank's workspace (identical on every rank). */
enum { HDRVAE_EX_END = 0, HDRVAE_EX_HALO = 1, HDRVAE_EX_ALLREDUCE_F64 = 2, HDRVAE_EX_ALLGATHER = 4, HDRVAE_EX_RAW_STATS = 8 };
typedef struct hdrvae_exchange {
  int32_t kind;                 /* bitmask of HDRVAE_EX_* ; HDRVAE_EX_END: the program is finished */
  int32_t n_halo;               /* 0..2 buffers */
  uint64_t halo_first_row_off[2], halo_last_row_off[2];   /* send: first interior row (up), last interior row (down) */
  uint64_t halo_top_off[2], halo_bottom_off[2];           /* receive: halo row above (from up), below (from down) */
  uint64_t halo_row_bytes[2];
  uint64_t allreduce_off, allreduce_count;
  int32_t n_gather, reserved;
  uint64_t gather_off[2], gather_bytes_per_rank[2];
  uint64_t raw_stats_off;
} hdrvae_exchange;
typedef struct hdrvae_rows hdrvae_rows;

int hdrvae_rows_workspace_bytes(hdrvae_ctx* ctx, int h, int w, int world, size_t* bytes);
/* latent_full_nchw: device float32 [1,C_lat,h,w] (the whole latent, every rank has it; 16 MB at 4096^2 for Flux);
 * out_rows: device float32 [1, 8h/world, 8w, 3] = this rank's rows of the IMAGE. */
int hdrvae_rows_begin(hdrvae_ctx* ctx, const float* latent_full_nchw, int h, int w, int rank, int world, int mode,
                      float expansion_factor, float ev_multiplier, float* out_rows, void* workspace,
                      size_t workspace_bytes, hdrvae_rows** state);
/* Enqueue work up to the next exchange point; *ex describes what the host must exchange before calling again. */
int hdrvae_rows_run(hdrvae_rows* state, hdrvae_exchange* ex, void* stream);
/* Device-driven transport (no host round trips, no NCCL on the data path): every rank allocates its workspace through
 * the library (hdrvae_peer_alloc: zero-initialised device memory + a CUDA IPC handle), the host exchanges the 64-byte
 * handles by any means (one all-gather of bytes), every rank maps every other rank's workspace (hdrvae_peer_open) and hands
 * the `world` pointers (its own at [rank]) to hdrvae_rows_set_peers.  hdrvae_rows_run_direct then enqueues the WHOLE
 * program on `stream`: at every exchange point a push kernel stores the halo rows / GroupNorm sums / K,V rows / statistics
 * straight into the peers' workspaces over NVLink behind a two-phase flag handshake, and a wait kernel folds the received
 * sums in rank order (csrc/rows_p2p.cu).  Results equal the host-driven exchange up to the fp64 order of 64 sums.  One
 * process per GPU only: ranks that share a GPU would wait on one another's kernels. */
typedef struct hdrvae_ipc_handle { unsigned char bytes[64]; } hdrvae_ipc_handle;
int hdrvae_peer_alloc(hdrvae_ctx* ctx, size_t bytes, void** dev_ptr, hdrvae_ipc_handle* handle);
int hdrvae_peer_open(hdrvae_ctx* ctx, const hdrvae_ipc_handle* handle, void** mapped);
int hdrvae_peer_close(hdrvae_ctx* ctx, void* mapped);
int hdrvae_peer_free(hdrvae_ctx* ctx, void* dev_ptr);
int hdrvae_rows_set_peers(hdrvae_rows* state, void* const* workspaces_of_all_ranks, int world);
int hdrvae_rows_run_direct(hdrvae_rows* state, void* stream);
/* After HDRVAE_EX_END: copy the statistics (global: pre/post/conv/pre3; local slab: out_*, pixel counts) and free. */
int hdrvae_rows_end(hdrvae_rows* state, hdrvae_stats* stats, void* stream);

/* ---- HDR upscaler: replaces HDRUpscaleWithModel.upscale (hdr_upscale_with_model.py:148-263) for four of the
 * architectures spandrel loads from models/upscale_models (:73-77):
 *   - ESRGAN / RRDBNet (nf 64, gc 32, any block count) with u = 0, 1 or 2 upsampling convs (nearest 2x + conv) and
 *     pixel-unshuffle factor f = 1, 2 or 4 (conv_first reads 3 f^2 channels: RealESRGAN_x2plus has u 2, f 2), scale
 *     s = 2^u / f in {1, 2, 4}; 8x (a third upsampling conv) and the pixel-shuffle upsampler variant are rejected.  A
 *     tile side that is not a multiple of f is reflect-padded (the pad must be shorter than the side) and the output
 *     cropped, as spandrel does;
 *   - Real-ESRGAN Compact (SRVGGNetCompact with PReLU: realesr-general-x4v3, realesr-animevideov3, the 2x / 1x
 *     "compact" models): 3 input channels, nf a multiple of 8 in 8..64, any body depth, scale s = 1, 2 or 4;
 *   - SPAN (spandrel's "SPAN"): 3 input channels, nf a multiple of 8 in 8..64, blocks block_1 .. block_6, any Conv3XC
 *     hidden width, scale s = 1, 2 or 4, with or without the input normalisation (buffer no_norm).  Every Conv3XC is
 *     fused from conv.0 / conv.1 / conv.2 and sk at load time, as its eval-mode forward does; eval_conv.* is ignored;
 *   - SwinIR (spandrel's "SwinIR"): 3 input channels, embed_dim C <= 256, head dimension C / heads <= 32, window 8 (shift 4
 *     in odd blocks), any RSTB count and depths, any MLP width, resi_connection "1conv" or "3conv", with or without
 *     patch_embed.norm, no absolute_pos_embed; upsampler "pixelshuffle", "pixelshuffledirect" or "nearest+conv" at
 *     s = 2 or 4, or "" at s = 1.  A tile is reflect-padded to a multiple of 8 (the pad must be shorter than the side), the
 *     shifted-window mask is computed for the padded size, and the output is cropped.  The stored relative_position_index
 *     and attn_mask buffers are not read.  HAT (conv_block / overlap_attn / relative_position_index_SA keys), 3x and 8x
 *     are rejected.
 * The layout is recognised by its keys (Compact: body.0.weight and no conv_first; SPAN: conv_1.sk.weight; SwinIR:
 * layers.0.residual_group.blocks.0.attn.relative_position_bias_table); anything else is rejected with a
 * message naming the tensor and its shape.  The model object is created against a decode context (device, SM count,
 * conv implementation).  s below is the model's scale (hdrvae_upscaler_scale).
 *   load_weights : the model's state dict, host or device pointers.  RRDBNet in either key layout (Real-ESRGAN
 *                  "conv_first / body.N.rdbK.convJ / conv_body / conv_up1 / conv_up2 / conv_hr / conv_last" or
 *                  BasicSR-spandrel "model.0 / model.1.sub.N.RDBK.convJ.0 / ...", whose top-level convs sit at 0,
 *                  3 + 3k (upsampling conv k + 1), 3u + 2 (conv_hr) and 3u + 4 (conv_last)); Compact as
 *                  "body.0 / body.1 (PReLU) / ... / body.{2nc+2}"; SPAN as "conv_1 / block_K.cJ_r / conv_2" (each
 *                  ".sk / .conv.0 / .conv.1 / .conv.2 / .eval_conv") / "conv_cat" / "upsampler.0" [/ "no_norm"]; SwinIR
 *                  in the network_swinir.py names ("conv_first / layers.i.residual_group.blocks.j.* / layers.i.conv /
 *                  norm / conv_after_body / ...");
 *   blocks       : RRDB blocks, the Compact's body convs nc (0 allowed), 6 (SPAN) or the RSTB count (SwinIR); < 0
 *                  without a model;
 *   scale        : 2^u / f for RRDBNet, s for Compact, SPAN and SwinIR; < 0 before the weights are loaded;
 *   forward      : the network (+ reversal hook) on n equal tiles, x [n,h,w,3] -> y [n,s*h,s*w,3], float32 device
 *                  (kernel-level parity entry: what `upscale_model(a)` with the forward hook returns, :92-105; for
 *                  Compact that includes the nearest-upsampled input the network adds);
 *   upscale      : the whole node: image [B,H,W,3] float32 -> out [B,s*H,s*W,3]; two passes (input as is / clamped to
 *                  [-1,1], :181-186) through 512-pixel tiles with 64 overlap and feather blending (:110-146,
 *                  comfy.utils.tiled_scale), Y from the first and Cb/Cr from the second pass, clamp(Y,0,8), 3x3 median
 *                  (:189-218), optional output median (small_blur, :219-224) and local hot-spot fix (:229-258). */
typedef struct hdrvae_upscaler hdrvae_upscaler;
int hdrvae_upscaler_create(hdrvae_ctx* ctx, hdrvae_upscaler** out);
int hdrvae_upscaler_destroy(hdrvae_upscaler* up);
int hdrvae_upscaler_load_weights(hdrvae_upscaler* up, const hdrvae_weight_desc* descs, int n);
int hdrvae_upscaler_blocks(hdrvae_upscaler* up);
int hdrvae_upscaler_scale(hdrvae_upscaler* up);
int hdrvae_upscaler_forward_bytes(hdrvae_upscaler* up, int n, int h, int w, size_t* bytes);
int hdrvae_upscaler_forward(hdrvae_upscaler* up, const float* x_bhwc, int n, int h, int w, int reversal,
                            float* y_bhwc, void* workspace, size_t workspace_bytes, void* stream);
int hdrvae_upscale_workspace_bytes(hdrvae_upscaler* up, int B, int H, int W, size_t* bytes);
int hdrvae_upscale(hdrvae_upscaler* up, const float* image_bhwc, int B, int H, int W, int reversal, int small_blur,
                   int local_fix, int upscale_method, float* out_bhwc, void* workspace, size_t workspace_bytes,
                   void* stream);

/* Decoder only: latent -> SiLU(norm_out(h)), the tensor the reference's forward
 * hook captures (hdr_vae_decode.py:850-855), as device NHWC [B,8h,8w,128] of hdrvae_operand_dtype(ctx) (fp16 by default). */
int hdrvae_decode_features(hdrvae_ctx* ctx, const float* latent_nchw, int B, int h, int w,
                           void* features_nhwc, void* workspace, size_t workspace_bytes,
                           void* stream);

/* Fused HDR epilogue on caller-supplied activations (the 1e-5 parity entry):
 * replaces analyze_conv_out's statistics + conv_out (:862-879), the MAX-pool
 * (:1042-1056), srgb_to_linear (:1163), the recovery block (:1076-1102), the mode
 * formulas (:1106-1159) and the multiplier (:180-182).
 *   pre_nhwc : device [B,H,W,128], dtype HDRVAE_F32, HDRVAE_F16 or HDRVAE_BF16
 *   conv_w   : device float32 [3,128,3,3] (OIHW, as in the state dict), conv_b [3]
 *   dbg_post3 / dbg_pre3 / dbg_argmax3 : optional device outputs [B,H,W,3]
 *               (float32, float32, int32): clamp((conv+1)/2), MAX-pool, first-max index
 *   scratch  : device, >= hdrvae_epilogue_scratch_bytes(B,H,W)
 */
int hdrvae_epilogue_scratch_bytes(int B, int H, int W, size_t* bytes);
int hdrvae_epilogue(hdrvae_ctx* ctx, const void* pre_nhwc, int dtype, int B, int H, int W,
                    const float* conv_w, const float* conv_b, int mode, float expansion_factor,
                    float ev_multiplier, float* out_bhwc, hdrvae_stats* stats, float* dbg_post3,
                    float* dbg_pre3, int32_t* dbg_argmax3, void* scratch, size_t scratch_bytes,
                    void* stream);

/* ---- kernel-level entry points (unit parity tests and micro-benchmarks) ----
 * Generic NHWC convolution on the tcgen05 implicit-GEMM kernel (or the CUDA-core validation kernel):
 * replaces one nn.Conv2d of ComfyUI's Decoder as driven by vae.decode (:859,:1022).
 *   x [B,H,W,Cin] of x_dtype: HDRVAE_F16 / HDRVAE_BF16 (kind::f16) or HDRVAE_F32 (read as tf32, kind::tf32);
 *   w OIHW float32 [Cout,Cin,k,k] (k = 1 or 3, pad k/2), bias float32 [Cout] or NULL (device pointers);
 *   residual [B,OH,OW,Cout] of res_dtype or NULL; upsample2x != 0: nearest-2x upsample folded into the load
 *   (OH=2H, OW=2W); y [B,OH,OW,Cout] of y_dtype; round_tf32: round a float32 y to tf32 (RN);
 *   gn_partials: optional device float32 [B][chunks][32][2] receiving the GroupNorm (sum, sum of squares)
 *   partials of y, chunks = hdrvae_conv2d_stats_chunks(H, W, upsample2x) (also stored to *gn_chunks).
 *   extra: NULL, or the channel slices, second output and epilogue of the upscalers' convs (hdrvae_conv_extra).
 * Without extra (or with its x_channels / y_channels 0) Cin must be a multiple of 64 and Cout of 32 and the tensors are
 * dense.  With x_channels, Cin is free (x_channels % 8 == 0, x_channels >= Cin); with y_channels, Cout is free
 * (y_chan_off % 4 == 0, y_channels % 4 == 0, y_chan_off + round_up(Cout, 4) <= y_channels) and the residuals share
 * y's addressing. */
enum { HDRVAE_ACT_NONE = 0, HDRVAE_ACT_SILU = 1, HDRVAE_ACT_GATE = 2, HDRVAE_ACT_GELU = 3 };
typedef struct hdrvae_conv_extra {
  int32_t x_channels;        /* pixel stride of x in elements (0: Cin); the conv reads the first Cin channels */
  int32_t y_channels;        /* pixel stride of y (0: Cout) ... */
  int32_t y_chan_off;        /* ... and the first channel of y written; round_up(Cout, 4) channels are stored */
  int32_t y2_dtype;          /* HDRVAE_F16 / HDRVAE_BF16 */
  void* y2;                  /* optional second output y * y2_scale (0: 1), 16-bit, [B,OH,OW,y2_channels] ... */
  float y2_scale;
  int32_t y2_channels;       /* ... (0: y's pixel stride and channel offset) */
  int32_t y2_chan_off;
  float res_scale;           /* t = conv + bias + res_scale * residual + residual2 (0: 1) */
  const float* residual2;    /* optional float32 in y's layout */
  const float* act_slope;    /* optional per-channel PReLU slopes, Cout floats */
  float lrelu;               /* LeakyReLU slope (0: none) */
  int32_t act;               /* HDRVAE_ACT_*: SiLU, the gate y = (t + residual terms)(sigmoid(t) - 1/2) of SPAN, or
                                GELU (erf form, nn.GELU()) applied last */
} hdrvae_conv_extra;
int hdrvae_conv2d(hdrvae_ctx* ctx, const void* x, int x_dtype, int B, int H, int W, int Cin, const float* w,
                  const float* bias, int Cout, int ksize, int upsample2x, const void* residual, int res_dtype,
                  void* y, int y_dtype, int round_tf32, float* gn_partials, int* gn_chunks, int impl,
                  void* stream, const hdrvae_conv_extra* extra);
int hdrvae_conv2d_stats_chunks(int H, int W, int upsample2x);

/* GroupNorm(32 groups, eps 1e-6, affine) [+ SiLU] on NHWC: replaces norm1/norm2/norm_out + swish of
 * ComfyUI's Decoder.  x of x_dtype (float32 stream or 16-bit), y of y_dtype (HDRVAE_F16/BF16), gamma/beta
 * float32 [C].  gn_partials/gn_chunks: statistics partials emitted by hdrvae_conv2d for x (skips the
 * statistics pass), or NULL/0. */
int hdrvae_groupnorm_silu(hdrvae_ctx* ctx, const void* x, int x_dtype, int B, int HW, int C, const float* gamma,
                          const float* beta, int apply_silu, void* y, int y_dtype, const float* gn_partials,
                          int gn_chunks, void* stream);

/* Single-head attention over T tokens, d = 512 (mid.attn_1 core; the reference reaches it through vae.decode,
 * hdr_vae_decode.py:859,:1022): q,k,v,o device [B,T,512] of dtype HDRVAE_F16 or HDRVAE_BF16; softmax(q k^T / sqrt(512)) v.
 * ONE fused flash-style kernel launch for all B images (csrc/attention.cu: S and O in tensor memory, P written back to
 * tensor memory as the PV operand, online soft-max with lazy rescaling; hdrvae_set_cta_group(ctx, 1) selects its
 * single-CTA build); the CUDA-core validation build (hdrvae_set_conv_impl) computes it as separate GEMMs.  The entry
 * itself allocates a scratch copy of the operands in the decoder's layout (q|k interleaved, v transposed). */
int hdrvae_attention(hdrvae_ctx* ctx, const void* q, const void* k, const void* v, int dtype, int B, int T,
                     void* o, void* stream);

/* LayerNorm over the C <= 256 channels of each of n_tokens fp32 tokens x [n_tokens][C] (eps 1e-5, fp32 statistics,
 * torch.nn.LayerNorm): y = (x - mean) / sqrt(var + eps) * gamma + beta, gamma / beta float32 [C].  y_dtype HDRVAE_F32
 * (y [n_tokens][C]) or HDRVAE_F16 (y [n_tokens][y_channels], y_channels >= C a multiple of 8; channels C .. y_channels - 1
 * are written as zero).  The SwinIR upscaler's norm1 / norm2 / norm / patch_embed.norm. */
int hdrvae_layernorm(hdrvae_ctx* ctx, const float* x, long long n_tokens, int C, const float* gamma, const float* beta,
                     void* y, int y_dtype, int y_channels, void* stream);

/* SwinIR's (shifted) window attention, window 8, head dim padded to 32: qkv fp16 [B][H][W][3 * heads * 32] holds per pixel
 * q (pre-scaled by head_dim^-0.5), k and v, each head-major with 32 channels per head (zero beyond the head dim); bias_table
 * float32 [225][heads] is the relative-position bias table; shift 0 or 4.  H and W are multiples of 8.  The windows tile
 * the image rolled by (-shift, -shift) (torch.roll, as the Swin transformer layer does); with a shift, keys of another
 * region of calculate_mask's partition of the H x W image get -100.  o fp16 [B][H][W][heads * 32]: softmax(q k^T + bias
 * (+ mask)) v written back at the un-shifted pixel of each query, head-major. */
int hdrvae_window_attention(hdrvae_ctx* ctx, const void* qkv, int B, int H, int W, int heads, const float* bias_table,
                            int shift, void* o, void* stream);

/* Exact quantiles by radix select over a device float32 array (statistical profiling; BASELINE.json north_star).
 * The reference computes none (SURVEY.md 0.6): defined as torch.quantile(x, q, interpolation="lower") =
 * the element of 0-based rank floor(q * (n - 1)); bit-exact.  q: host doubles in [0,1] (1..8 of them),
 * out_host: host float32 [nq]; synchronises the stream. */
int hdrvae_quantiles(const float* data, long long n, const double* q, int nq, float* out_host, void* stream);

/* fp32 -> fp16 round-to-nearest-even pack for LinearEXRExport
 * (linear_exr_export.py:155,165: ndarray.astype(np.float16); overflow -> inf).
 * layout 0: same order as the input; layout 1: EXR scanline order
 * (per image row: B plane, G plane, R plane). image [B,H,W,3] float32 device. */
int hdrvae_pack_half(const float* image_bhwc, int B, int H, int W, int layout, uint16_t* out,
                     void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HDRVAE_H_ */
