// HDR upscaler path: replaces HDRUpscaleWithModel.upscale of the reference
// (/root/reference/hdr_upscale_with_model.py:148-263): two passes of the model (ESRGAN / RRDBNet at 1x, 2x or 4x, or
// Real-ESRGAN Compact or SPAN at 1x, 2x or 4x) through overlapping 512-pixel tiles with the atanh / logit reversal hook on every tile output
// (:79-107, :110-146), feather blending (restated comfy.utils.tiled_scale), then the luma / chroma recombination in YCbCr
// with a 3x3 median on Y (:187-224) and the optional local hot-spot fix (:229-258).  Everything after the model reads
// the float4 tile-output layout [n][s h][s w] that both forwards leave, with the model's scale s.
//
// The RRDB convs run on the tcgen05 implicit-GEMM kernel of gemm_tc.cu with narrow (32 / 64 column) tiles:
//   * a dense block keeps one 192-channel fp16 buffer per pixel [x | g1 | g2 | g3 | g4]; conv k reads the channel
//     prefix 64 + 32(k-1) through a TMA map whose channel extent is exactly that prefix (the tail of the last
//     128-byte K block is zero-filled by TMA, the packed weights hold zeros there) and writes its LeakyReLU'd 32
//     channels into the next slice: the concat never exists as a copy;
//   * conv5 adds the fp32 residual stream (0.2 conv + x; at the end of an RRDB 0.04 conv + 0.2 x2 + x0 with two
//     residual operands) and writes, besides the fp32 stream, the fp16 operand copy into the next block's buffer;
//   * the u (0, 1 or 2) nearest-2x upsamples are folded into the loads of conv_up1 / conv_up2 (4 phase convs each);
//   * conv_last (64 -> 3) computes 32 columns and stores 4;
//   * a pixel-unshuffle RRDBNet (RealESRGAN_x2plus: f = 2) reads its tile reflect-padded to a multiple of f and unshuffled
//     into 3 f^2 channels (up_extract_tiles_kernel<f>); the scale is 2^u / f, and a padded tile's output is cropped.
// The Compact convs (SRVGGNetCompact: conv, PReLU, ..., conv to 3 s^2 channels) run on the same kernel with the
// per-channel PReLU in the epilogue; up_shuffle_base_kernel then applies the pixel shuffle and adds the nearest-upsampled
// fp32 input (the network's base).
// SPAN (conv_1, six SPAB blocks, conv_2, conv_cat, upsampler.0) runs on the same kernel too: every Conv3XC is fused into
// one 3x3 conv at load time, SiLU and SPAN's attention gate are epilogue operations, and the four tensors conv_cat reads
// are channel slices of one fp16 buffer, so that conv_cat is a plain 1x1 conv (up_forward_span).
// SwinIR (up_forward_swinir) runs its linears and convs on the same kernel (fc1 with the GELU epilogue) and its LayerNorm,
// shifted-window attention and fp16 pixel shuffle in swin.cu, on the tile reflect-padded to a multiple of the 8-pixel window.
// Everything after the model (hook, feather blend, YCbCr, median, local fix) is elementwise / stencil work in
// fp32 with the reference's operation order (no FMA contraction) so that it is bit-comparable to the oracle.
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "engine.cuh"

namespace hdrvae {

// ------------------------------------------------------------------------------------------------ kernels
// fp16 channels per pixel of the network input for pixel-unshuffle factor f: 3 f^2 rounded up to a 16-byte pixel stride
// (the TMA row stride); the conv reads the first 3 f^2 of them (ConvIO::x_channels)
__host__ __device__ constexpr int up_in_channels(int f) { return f == 1 ? 8 : f == 2 ? 16 : 48; }

// image fp32 BHWC (3 channels) -> fp16 network input [n][h'][w'][up_in_channels(F)] of tiles of h x w at the origins of
// `tiles`: clamp to [-1, 1] (flag or tile table .w), minus `mean` (SPAN's and SwinIR's normalisation; zero for the
// other models, where it leaves every value as it is), reflect pad of the tile's bottom / right edge to
// F h' x F w' (torch "reflect": row h + k reads row h - 2 - k), pixel unshuffle by F (channel c F^2 + i F + j = channel c
// at pixel (y F + i, x F + j)), channels beyond 3 F^2 zero.  The clamp is elementwise, so it commutes with pad and
// unshuffle.  h' = ceil(h / F) for RRDBNet, and h rounded up to a multiple of 8 (SwinIR's window, F = 1); F = 1 without
// a pad is the plain [n][h][w][8] copy.
template <int F>
__global__ void up_extract_tiles_kernel(const float* __restrict__ img, int H, int W, const int4* __restrict__ tiles /*b,y0,x0,_*/,
                                        int n, int h, int w, int hq, int wq, int clamp1, float3 mean, uint4* __restrict__ out) {
  constexpr int CX = up_in_channels(F), F2 = F * F;
  const long long total = (long long)n * hq * wq;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int x = (int)(i % wq);
    const int y = (int)((i / wq) % hq);
    const int t = (int)(i / ((long long)wq * hq));
    const int4 tl = tiles[t];                     // image, y0, x0, clamp flag
    __align__(16) __half v[CX];
#pragma unroll
    for (int c = 0; c < CX; ++c) v[c] = __float2half_rn(0.f);
#pragma unroll
    for (int a = 0; a < F; ++a) {
      int yy = y * F + a;
      if (yy >= h) yy = 2 * (h - 1) - yy;
#pragma unroll
      for (int b = 0; b < F; ++b) {
        int xx = x * F + b;
        if (xx >= w) xx = 2 * (w - 1) - xx;
        const float* src = img + (((long long)tl.x * H + tl.y + yy) * W + tl.z + xx) * 3;
        float r = src[0], g = src[1], bl = src[2];
        if (clamp1 || tl.w) { r = fminf(fmaxf(r, -1.f), 1.f); g = fminf(fmaxf(g, -1.f), 1.f); bl = fminf(fmaxf(bl, -1.f), 1.f); }
        r = __fsub_rn(r, mean.x); g = __fsub_rn(g, mean.y); bl = __fsub_rn(bl, mean.z);
        v[a * F + b] = __float2half_rn(r);
        v[F2 + a * F + b] = __float2half_rn(g);
        v[2 * F2 + a * F + b] = __float2half_rn(bl);
      }
    }
#pragma unroll
    for (int k = 0; k < CX / 8; ++k) out[i * (CX / 8) + k] = reinterpret_cast<const uint4*>(v)[k];
  }
}

// top-left [oh][ow] window of each of n float4 images [ih][iw]: the output of a reflect-padded tile cut to s h x s w
__global__ void up_crop_kernel(const float4* __restrict__ in, int ih, int iw, int n, int oh, int ow, float4* __restrict__ out) {
  const long long total = (long long)n * oh * ow;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int x = (int)(i % ow);
    const int y = (int)((i / ow) % oh);
    const int t = (int)(i / ((long long)ow * oh));
    out[i] = in[((long long)t * ih + y) * iw + x];
  }
}

__global__ void up_scale_f32_kernel(float* p, int n, float s) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] *= s;
}

__device__ __forceinline__ float up_reversal(float v, int kind) {
  if (kind == 1) {                                    // atanh(clamp(v, -1 + 1e-6, 1 - 1e-6))   (:101-105)
    v = fminf(fmaxf(v, -1.f + 1e-6f), 1.f - 1e-6f);
    return atanhf(v);
  }
  if (kind == 2) {                                    // logit(clamp(v, 1e-7, 1 - 1e-7))          (:93-98)
    v = fminf(fmaxf(v, 1e-7f), 1.f - 1e-7f);
    return logf(__fdiv_rn(v, 1.f - v));
  }
  return v;
}

// Compact tail: y = pixel_shuffle(conv, s) + nearest_upsample(x, s).  conv is the last conv's fp32 output [n][h][w][cl]
// (channel c s^2 + i s + j of input pixel (y, x) -> channel c of output pixel (y s + i, x s + j)); the base is the tile's
// fp32 input pixel, clamped to [-1, 1] for the second pass's tiles (tile table .w) like the network's own input.  Writes
// the float4 [n][s h][s w] tile-output layout of the RRDBNet forward (.w = 0).  img == null: the plain pixel shuffle
// (SPAN, which adds no base).
__global__ void up_shuffle_base_kernel(const float* __restrict__ conv, int cl, const float* __restrict__ img, int H, int W,
                                       const int4* __restrict__ tiles, int n, int h, int w, int s, float4* __restrict__ out) {
  const int OH = h * s, OW = w * s, s2 = s * s;
  const long long total = (long long)n * OH * OW;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int X = (int)(i % OW);
    const int Y = (int)((i / OW) % OH);
    const int t = (int)(i / ((long long)OW * OH));
    const int y = Y / s, x = X / s;
    const float* c = conv + (((long long)t * h + y) * w + x) * cl + (Y - y * s) * s + (X - x * s);
    if (img == nullptr) {
      out[i] = make_float4(c[0], c[s2], c[2 * s2], 0.f);
      continue;
    }
    const int4 tl = tiles[t];                     // image, y0, x0, clamp flag
    const float* src = img + (((long long)tl.x * H + tl.y + y) * W + tl.z + x) * 3;
    float r = src[0], g = src[1], b = src[2];
    if (tl.w) { r = fminf(fmaxf(r, -1.f), 1.f); g = fminf(fmaxf(g, -1.f), 1.f); b = fminf(fmaxf(b, -1.f), 1.f); }
    out[i] = make_float4(__fadd_rn(c[0], r), __fadd_rn(c[s2], g), __fadd_rn(c[2 * s2], b), 0.f);
  }
}

// model output [n][s h][s w][4] fp32 -> reversal hook -> [n][s h][s w][3] (kernel-level parity entry)
__global__ void up_finish_tiles_kernel(const float4* __restrict__ in, long long n_px, int kind, float* __restrict__ out) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n_px; i += (long long)gridDim.x * blockDim.x) {
    const float4 v = in[i];
    out[i * 3 + 0] = up_reversal(v.x, kind);
    out[i * 3 + 1] = up_reversal(v.y, kind);
    out[i * 3 + 2] = up_reversal(v.z, kind);
  }
}

struct UpTile {             // one tile of comfy.utils.tiled_scale, output coordinates
  int b, oy, ox, oh, ow;    // image index, origin and size on the upscaled grid
  long long off, off2;      // float4 offsets of the tile's model output: pass 1 (input as is), pass 2 (input clamped)
};

// feather weight of output row/col `i` of a tile of length `len` (restated tiled_scale: ramps (t+1)/feather applied
// to both ends, successively, in fp32; a dimension not longer than the feather is left unmasked)
__device__ __forceinline__ float up_feather(float m, int i, int len, int feather) {
  if (feather >= len) return m;
  if (i < feather) m = __fmul_rn(m, (float)((double)(i + 1) / (double)feather));
  if (len - 1 - i < feather) m = __fmul_rn(m, (float)((double)(len - i) / (double)feather));
  return m;
}

// Blend of one pass: for every output pixel the tiles covering it, in the reference's accumulation order
// (itertools.product: y outer, x inner): out += reversal(ps) * mask; div += mask; result out / div.
__device__ __forceinline__ void up_blend_px(const float4* __restrict__ tiles_out, const UpTile* __restrict__ tl, int t0, int t1,
                                            int single, int second, int b, int y, int x, int feather, int kind, float* rgb) {
  if (single) {
    const UpTile t = tl[t0 + b];
    const float4 v = tiles_out[(second ? t.off2 : t.off) + (long long)y * t.ow + x];
    rgb[0] = up_reversal(v.x, kind); rgb[1] = up_reversal(v.y, kind); rgb[2] = up_reversal(v.z, kind);
    return;
  }
  float acc[3] = {0.f, 0.f, 0.f}, div = 0.f;
  for (int i = t0; i < t1; ++i) {
    const UpTile t = tl[i];
    if (t.b != b || y < t.oy || y >= t.oy + t.oh || x < t.ox || x >= t.ox + t.ow) continue;
    const int ly = y - t.oy, lx = x - t.ox;
    float m = 1.f;
    m = up_feather(m, ly, t.oh, feather);
    m = up_feather(m, lx, t.ow, feather);
    const float4 v = tiles_out[(second ? t.off2 : t.off) + (long long)ly * t.ow + lx];
    acc[0] = __fadd_rn(acc[0], __fmul_rn(up_reversal(v.x, kind), m));
    acc[1] = __fadd_rn(acc[1], __fmul_rn(up_reversal(v.y, kind), m));
    acc[2] = __fadd_rn(acc[2], __fmul_rn(up_reversal(v.z, kind), m));
    div = __fadd_rn(div, m);
  }
  rgb[0] = __fdiv_rn(acc[0], div); rgb[1] = __fdiv_rn(acc[1], div); rgb[2] = __fdiv_rn(acc[2], div);
}

__device__ __forceinline__ void up_rgb_to_ycbcr(const float* rgb, float* ycc) {
  // kornia.color.rgb_to_ycbcr, left-to-right fp32
  const float y = __fadd_rn(__fadd_rn(__fmul_rn(0.299f, rgb[0]), __fmul_rn(0.587f, rgb[1])), __fmul_rn(0.114f, rgb[2]));
  ycc[0] = y;
  ycc[1] = __fadd_rn(__fmul_rn(__fsub_rn(rgb[2], y), 0.564f), 0.5f);
  ycc[2] = __fadd_rn(__fmul_rn(__fsub_rn(rgb[0], y), 0.713f), 0.5f);
}

// Both passes blended -> (clamp(Y_unclamped, 0, 8), Cb_clamped, Cr_clamped) per pixel   (:189-213)
__global__ void up_blend_ycc_kernel(const float4* __restrict__ tiles_out,
                                    const UpTile* __restrict__ tl, int n_tiles, int single, int B, int OH, int OW,
                                    int feather, int kind, float* __restrict__ ycc /*[B][OH][OW][3]*/) {
  const long long total = (long long)B * OH * OW;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int x = (int)(i % OW);
    const int y = (int)((i / OW) % OH);
    const int b = (int)(i / ((long long)OW * OH));
    float ru[3], rc[3], yu[3], yc[3];
    up_blend_px(tiles_out, tl, 0, n_tiles, single, 0, b, y, x, feather, kind, ru);
    up_blend_px(tiles_out, tl, 0, n_tiles, single, 1, b, y, x, feather, kind, rc);
    up_rgb_to_ycbcr(ru, yu);
    up_rgb_to_ycbcr(rc, yc);
    ycc[i * 3 + 0] = fminf(fmaxf(yu[0], 0.f), 8.f);
    ycc[i * 3 + 1] = yc[1];
    ycc[i * 3 + 2] = yc[2];
  }
}

__device__ __forceinline__ void up_sort2(float& a, float& b) { const float lo = fminf(a, b), hi = fmaxf(a, b); a = lo; b = hi; }
__device__ __forceinline__ float up_median9(float* v) {
  // 19-exchange median-of-9 network
  up_sort2(v[1], v[2]); up_sort2(v[4], v[5]); up_sort2(v[7], v[8]);
  up_sort2(v[0], v[1]); up_sort2(v[3], v[4]); up_sort2(v[6], v[7]);
  up_sort2(v[1], v[2]); up_sort2(v[4], v[5]); up_sort2(v[7], v[8]);
  up_sort2(v[0], v[3]); up_sort2(v[5], v[8]); up_sort2(v[4], v[7]);
  up_sort2(v[3], v[6]); up_sort2(v[1], v[4]); up_sort2(v[2], v[5]);
  up_sort2(v[4], v[7]); up_sort2(v[4], v[2]); up_sort2(v[6], v[4]);
  up_sort2(v[4], v[2]);
  return v[4];
}

// zero-padded 3x3 median of channel `c` of an interleaved [B][H][W][3] tensor (kornia.filters.median_blur)
__device__ __forceinline__ float up_median_at(const float* __restrict__ t, int b, int y, int x, int c, int H, int W) {
  float v[9];
#pragma unroll
  for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
    for (int dx = -1; dx <= 1; ++dx) {
      const int yy = y + dy, xx = x + dx;
      v[(dy + 1) * 3 + dx + 1] = (yy >= 0 && yy < H && xx >= 0 && xx < W) ? t[(((long long)b * H + yy) * W + xx) * 3 + c] : 0.f;
    }
  return up_median9(v);
}

// median on Y, then the reference's un-clamped ycbcr_to_rgb (:20-48)
__global__ void up_recombine_kernel(const float* __restrict__ ycc, int B, int H, int W, float* __restrict__ out) {
  const long long total = (long long)B * H * W;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int x = (int)(i % W);
    const int y = (int)((i / W) % H);
    const int b = (int)(i / ((long long)W * H));
    const float Y = up_median_at(ycc, b, y, x, 0, H, W);
    const float cb = __fsub_rn(ycc[i * 3 + 1], 0.5f), cr = __fsub_rn(ycc[i * 3 + 2], 0.5f);
    out[i * 3 + 0] = __fadd_rn(Y, __fmul_rn(1.403f, cr));
    out[i * 3 + 1] = __fsub_rn(__fsub_rn(Y, __fmul_rn(0.714f, cr)), __fmul_rn(0.344f, cb));
    out[i * 3 + 2] = __fadd_rn(Y, __fmul_rn(1.773f, cb));
  }
}

// per-channel zero-padded 3x3 median of an RGB image (small_blur output filter, :219-224)
__global__ void up_median_rgb_kernel(const float* __restrict__ in, int B, int H, int W, float* __restrict__ out) {
  const long long total = (long long)B * H * W * 3;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % 3);
    const long long px = i / 3;
    const int x = (int)(px % W);
    const int y = (int)((px / W) % H);
    const int b = (int)(px / ((long long)W * H));
    out[i] = up_median_at(in, b, y, x, c, H, W);
  }
}

// local hot-spot fix (:229-258): mask = upscaled luma of the ORIGINAL image < 0.1; out = s (1 - mask) + clamp(s, -1, 1) mask
__global__ void up_local_fix_kernel(const float* __restrict__ img, int B, int H, int W, int scale, int method,
                                    float* __restrict__ s /*[B][H*scale][W*scale][3], in place*/) {
  const int OH = H * scale, OW = W * scale;
  const long long total = (long long)B * OH * OW;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int x = (int)(i % OW);
    const int y = (int)((i / OW) % OH);
    const int b = (int)(i / ((long long)OW * OH));
    auto luma = [&](int yy, int xx) {
      const float* p = img + (((long long)b * H + yy) * W + xx) * 3;
      return __fadd_rn(__fadd_rn(__fmul_rn(0.299f, p[0]), __fmul_rn(0.587f, p[1])), __fmul_rn(0.114f, p[2]));
    };
    float ys;
    if (method == HDRVAE_UPSCALE_BISLERP) {
      // comfy.utils.bislerp on the 1-channel luma (restated in oracle/upscaler_oracle.py): separable, width pass first.
      // Per axis: the two source pixels bilinear interpolation (align_corners = False) would blend, c1 = floor(src),
      // c2 = min(c1 + 1, last), ratio r = frac(src) with src = max((dst + 0.5) / scale - 0.5, 0) — exact in fp32 for
      // power-of-two scales — then a SPHERICAL interpolation of the channel vectors; for scalars: same sign -> the first
      // pixel, opposite signs -> linear, a zero -> sine weights times the linearly interpolated magnitude.
      auto slerp1 = [](float b1, float b2, float r) {
        const float n1 = fabsf(b1), n2 = fabsf(b2);
        const float u1 = n1 == 0.f ? 0.f : b1 / n1, u2 = n2 == 0.f ? 0.f : b2 / n2;
        const float dot = u1 * u2;
        if (dot > 1.f - 1e-5f) return b1;
        if (dot < 1e-5f - 1.f) return __fadd_rn(__fmul_rn(b1, __fsub_rn(1.f, r)), __fmul_rn(b2, r));
        const float omega = acosf(dot), so = sinf(omega);
        float res = (sinf((1.f - r) * omega) / so) * u1 + (sinf(r * omega) / so) * u2;
        return res * (n1 * (1.f - r) + n2 * r);
      };
      const float fy = fmaxf((y + 0.5f) / scale - 0.5f, 0.f), fx = fmaxf((x + 0.5f) / scale - 0.5f, 0.f);
      const int y1 = min((int)fy, H - 1), x1 = min((int)fx, W - 1);
      const int y2 = min(y1 + 1, H - 1), x2 = min(x1 + 1, W - 1);
      const float ry = fy - floorf(fy), rx = fx - floorf(fx);
      const float t1 = slerp1(luma(y1, x1), luma(y1, x2), rx);
      const float t2 = slerp1(luma(y2, x1), luma(y2, x2), rx);
      ys = slerp1(t1, t2, ry);
    } else if (method == HDRVAE_UPSCALE_NEAREST_EXACT || method == HDRVAE_UPSCALE_AREA) {
      // nearest-exact: floor((dst + 0.5) / scale); "area" = adaptive average pooling, whose window for an integer
      // upscale factor is exactly that one source pixel
      ys = luma(min((int)floorf((y + 0.5f) / scale), H - 1), min((int)floorf((x + 0.5f) / scale), W - 1));
    } else if (method == HDRVAE_UPSCALE_BICUBIC) {
      // torch upsample_bicubic2d, align_corners = False: cubic convolution, A = -0.75, border indices clamped
      auto coef = [](float t, float* c) {
        const float A = -0.75f;
        auto c1 = [A](float x) { return ((A + 2.f) * x - (A + 3.f)) * x * x + 1.f; };
        auto c2 = [A](float x) { return ((A * x - 5.f * A) * x + 8.f * A) * x - 4.f * A; };
        c[0] = c2(t + 1.f); c[1] = c1(t); c[2] = c1(1.f - t); c[3] = c2(2.f - t);
      };
      const float fy = (y + 0.5f) / scale - 0.5f, fx = (x + 0.5f) / scale - 0.5f;
      const int iy = (int)floorf(fy), ix = (int)floorf(fx);
      float cy[4], cx[4];
      coef(fy - iy, cy); coef(fx - ix, cx);
      ys = 0.f;
#pragma unroll
      for (int a = 0; a < 4; ++a) {
        const int yy = min(max(iy - 1 + a, 0), H - 1);
        float rowv = 0.f;
#pragma unroll
        for (int b2 = 0; b2 < 4; ++b2) rowv += cx[b2] * luma(yy, min(max(ix - 1 + b2, 0), W - 1));
        ys += cy[a] * rowv;
      }
    } else {   // bilinear, align_corners = False (torch.nn.functional.interpolate)
      const float fy = fmaxf((y + 0.5f) / scale - 0.5f, 0.f), fx = fmaxf((x + 0.5f) / scale - 0.5f, 0.f);
      const int y0 = min((int)fy, H - 1), x0 = min((int)fx, W - 1);
      const int y1 = min(y0 + 1, H - 1), x1 = min(x0 + 1, W - 1);
      const float wy = fy - y0, wx = fx - x0;
      ys = (1.f - wy) * ((1.f - wx) * luma(y0, x0) + wx * luma(y0, x1)) + wy * ((1.f - wx) * luma(y1, x0) + wx * luma(y1, x1));
    }
    const float mask = ys < 0.1f ? 1.f : 0.f;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float v = s[i * 3 + c];
      s[i * 3 + c] = __fadd_rn(__fmul_rn(v, __fsub_rn(1.f, mask)), __fmul_rn(fminf(fmaxf(v, -1.f), 1.f), mask));
    }
  }
}

static inline int up_grid(long long n) { return (int)std::min<long long>((n + 255) / 256, 148 * 32); }

}  // namespace hdrvae

using namespace hdrvae;

// ------------------------------------------------------------------------------------------------ model
enum UpArch { UP_RRDB, UP_COMPACT, UP_SPAN, UP_SWINIR };   // ESRGAN / RRDBNet, Real-ESRGAN SRVGGNetCompact, SPAN, SwinIR
enum UpSwinTail { SW_NONE, SW_PIXELSHUFFLE, SW_DIRECT, SW_NEAREST };   // SwinIR upsampler "", "pixelshuffle",
                                                                       // "pixelshuffledirect", "nearest+conv"
struct UpSwinBlock {              // one Swin transformer layer (STL) of SwinIR
  float *ln1_g = nullptr, *ln1_b = nullptr, *ln2_g = nullptr, *ln2_b = nullptr;
  float* table = nullptr;         // relative-position bias table [225][heads]
  PackedConv qkv, proj, fc1, fc2; // qkv: 3 heads 32 columns (q scaled by hd^-0.5, heads padded to 32); proj reads that layout
};
struct UpSwin {
  int C = 0, CP = 0;              // embed_dim and the pixel stride of its fp16 operands (C rounded up to 8)
  int heads = 0, hidden = 0, HP = 0;   // heads, MLP width and its fp16 pixel stride
  int c4 = 0, c4p = 0;            // 3conv: conv.0 / conv.2 width C / 4 and its pixel stride
  bool conv3 = false, patch_norm = false;
  UpSwinTail tail = SW_NONE;
  int n_up = 0;                   // 2x stages of the pixelshuffle / nearest+conv tails
  std::vector<int> depths;        // blocks per RSTB
  std::vector<UpSwinBlock> blocks;
  float *pn_g = nullptr, *pn_b = nullptr, *norm_g = nullptr, *norm_b = nullptr;   // patch_embed.norm, norm
};

struct hdrvae_upscaler {
  hdrvae_ctx* ctx = nullptr;      // device / SM count / conv implementation come from the decode context
  hdrvae_ctx store;               // owns this model's device allocations
  bool loaded = false;
  UpArch arch = UP_RRDB;
  float3 mean = {0.f, 0.f, 0.f};  // subtracted from the network input (SPAN's normalisation; its 255 is in conv_1's weights)
  int scale = 4;                  // output pixels per input pixel along each axis (RRDBNet: 2^n_up / shuffle)
  int nb = 0;                     // RRDB blocks (RRDBNet), body convs (Compact) or SPAB blocks (SPAN: 6)
  int n_up = 2;                   // RRDBNet: nearest-2x + conv upsampling stages (0, 1 or 2)
  int shuffle = 1;                // RRDBNet: pixel-unshuffle factor of the input (1, 2 or 4; conv_first reads 3 f^2 channels)
  std::vector<PackedConv> convs;  // every conv in launch order.  RRDBNet: conv_first, conv1 .. conv5 of each dense block
                                  // (3 per RRDB), conv_body, conv_up1 / conv_up2 (n_up of them), conv_hr, conv_last.
                                  // Compact: first conv, nb body convs, last conv (nf -> 3 s^2).  SPAN: the fused conv_1,
                                  // block_k.c{1,2,3}_r (k = 1..6), conv_2, then conv_cat (1x1, 4 nf -> nf) and upsampler.0
  std::vector<float*> slopes;     // Compact: PReLU slopes applied after convs[k], k <= nb (cout_pad floats, zero-padded)
                                  // SwinIR: conv_first, each RSTB's conv (or conv.0/2/4), conv_after_body (1 or 3), then the
                                  // tail: conv_before_upsample.0, upsample.{2k} | conv_up1/2, conv_hr, conv_last, or upsample.0
                                  // or conv_last alone
  UpSwin sw;                      // SwinIR: dimensions and the transformer layers (their linears are not in `convs`)
};

namespace hdrvae {

// channels per pixel of the Compact last conv's fp32 output: 3 s^2 rounded up to the epilogue's 4-column stores
static int up_last_channels(const hdrvae_upscaler* up) { return (3 * up->scale * up->scale + 3) / 4 * 4; }

// network grid of a tile of h x w: the reflect-padded tile pixel-unshuffled by the model's factor f (RRDBNet), or the
// tile reflect-padded to a multiple of SwinIR's 8-pixel window
static constexpr int kSwinWin = 8;
static int up_net_side(const hdrvae_upscaler* up, int side) {
  if (up->arch == UP_SWINIR) return (side + kSwinWin - 1) / kSwinWin * kSwinWin;
  return (side + up->shuffle - 1) / up->shuffle;
}

// torch's reflect pad needs pad < side; a tile side for which the pad to a multiple of f (or of the window) fails is refused
static int up_check_sides(const hdrvae_upscaler* up, int h, int w) {
  const int f = up->arch == UP_SWINIR ? kSwinWin : up->shuffle;
  for (int side : {h, w}) {
    const int pad = (f - side % f) % f;
    if (up->arch == UP_SWINIR)
      HDRVAE_REQUIRE(pad < side, "upscaler: a tile side of %d pixels is too short for the reflect pad of %d pixels that "
                     "SwinIR's %d-pixel windows need (the pad must be shorter than the side)", side, pad, f);
    else
      HDRVAE_REQUIRE(pad < side, "upscaler: a tile side of %d pixels is too short for the reflect pad of %d pixels that the "
                     "model's %dx pixel unshuffle needs (the pad must be shorter than the side)", side, pad, f);
  }
  return 0;
}

struct UpPlan {                   // workspace of one forward over n tiles of h x w
  size_t img8, cat0, cat1, f_feat, f_a, f_b, f_c, u0, u1, u2, u3;   // RRDBNet
  size_t act0, act1, last;                                          // Compact (SPAN: last)
  size_t sp_r0, sp_r1, sp_d, sp_t0, sp_t1, sp_cat;                  // SPAN
  size_t sw_f, sw_b0, sw_b1, sw_a16, sw_b16, sw_qkv, sw_o, sw_hid, sw_t0, sw_t1, sw_u0, sw_ua, sw_ub, sw_big, sw_last,
         sw_out;                                                    // SwinIR
  size_t total;
};
static UpPlan up_make_plan(const hdrvae_upscaler* up, int n, int h, int w) {
  UpPlan pl;
  size_t off = 0;
  auto take = [&](size_t bytes) { const size_t o = off; off += (bytes + 1023) / 1024 * 1024; return o; };
  const size_t P = (size_t)n * up_net_side(up, h) * up_net_side(up, w);   // pixels of the network's input grid
  pl.img8 = take(P * up_in_channels(up->shuffle) * 2);
  switch (up->arch) {
    case UP_COMPACT: {
      // fp16 activations at a pixel stride of cout_pad (the convs read the first nf channels), ping-pong
      const size_t cp = (size_t)up->convs[0].cout_pad;
      pl.act0 = take(P * cp * 2);
      pl.act1 = take(P * cp * 2);
      pl.last = take(P * up_last_channels(up) * 4);
      break;
    }
    case UP_SPAN: {
      const size_t nf = (size_t)up->convs[0].cout;
      pl.sp_r0 = take(P * nf * 4);      // fp32 block stream (the gate's residual), ping-pong
      pl.sp_r1 = take(P * nf * 4);
      pl.sp_d = take(P * nf * 2);       // fp16 operand copy of a block output
      pl.sp_t0 = take(P * nf * 2);      // SiLU'd c1_r / c2_r outputs
      pl.sp_t1 = take(P * nf * 2);
      pl.sp_cat = take(P * 4 * nf * 2); // [f | b6 | b1 | b5_2]: conv_cat's input, the channel order of torch.cat
      pl.last = take(P * up_last_channels(up) * 4);
      break;
    }
    case UP_SWINIR: {
      const UpSwin& sw = up->sw;
      const size_t s2 = (size_t)up->scale * up->scale;
      pl.sw_f = take(P * sw.C * 4);                 // conv_first's output (the long skip), fp32
      pl.sw_b0 = take(P * sw.C * 4);                // RSTB input / output stream, fp32
      pl.sw_b1 = take(P * sw.C * 4);                // the STL stream inside an RSTB, fp32
      pl.sw_a16 = take(P * sw.CP * 2);              // LayerNorm outputs and the stream's fp16 copy
      pl.sw_b16 = take(P * sw.CP * 2);              // conv_after_body's output (the tail's input), fp16
      pl.sw_qkv = take(P * sw.heads * 3 * 32 * 2);  // q | k | v, 32 channels per head
      pl.sw_o = take(P * sw.heads * 32 * 2);        // attention output, 32 channels per head
      pl.sw_hid = take(P * sw.HP * 2);              // GELU(fc1)
      pl.sw_t0 = take(sw.conv3 ? P * sw.c4p * 2 : 0);   // 3conv: conv.0 / conv.2 outputs
      pl.sw_t1 = take(sw.conv3 ? P * sw.c4p * 2 : 0);
      const bool up64 = sw.tail == SW_PIXELSHUFFLE || sw.tail == SW_NEAREST;
      pl.sw_u0 = take(up64 ? P * 64 * 2 : 0);       // conv_before_upsample
      pl.sw_ua = take(up64 ? P * s2 * 64 * 2 : 0);  // 64-channel fp16 stages of the tail, ping-pong
      pl.sw_ub = take(up64 ? P * s2 * 64 * 2 : 0);
      pl.sw_big = take(sw.tail == SW_PIXELSHUFFLE ? P * (s2 / 4) * 256 * 2 : 0);   // upsample.{2k}'s 256 channels
      pl.sw_last = take(sw.tail == SW_DIRECT ? P * up_last_channels(up) * 4 : sw.tail == SW_NONE ? P * 16 : 0);
      pl.sw_out = take(P * s2 * 16);                // float4 output of the padded tile (cropped into out4)
      break;
    }
    case UP_RRDB:
      pl.cat0 = take(P * 192 * 2);
      pl.cat1 = take(P * 192 * 2);
      pl.f_feat = take(P * 64 * 4);
      pl.f_a = take(P * 64 * 4);
      pl.f_b = take(P * 64 * 4);
      pl.f_c = take(P * 64 * 4);
      // fp16 operands of the upsampling stages: conv_body's copy (h' w'), conv_up1's (4 h' w'), conv_up2's (16 h' w'), conv_hr's
      pl.u0 = take(P * 64 * 2);
      pl.u1 = take(up->n_up >= 1 ? P * 4 * 64 * 2 : 0);
      pl.u2 = take(up->n_up >= 2 ? P * 16 * 64 * 2 : 0);
      pl.u3 = take((P << (2 * up->n_up)) * 64 * 2);
      break;
  }
  pl.total = off;
  return pl;
}

// RRDBNet forward on n tiles of h x w (fp16 network input [n][h'][w'][cx] in pl.img8, h' = ceil(h / f)) -> fp32
// [n][s h][s w][4] at `out4`.  The network runs at h' x w' and conv_last at 2^u h' x 2^u w' = f s h' x f s w'; when the
// tile was padded (f h' > h) conv_last writes into the dense-block buffer cat0 (dead by then) and the top-left window is
// copied to out4.
static int up_forward_rrdb(hdrvae_upscaler* up, int n, int h, int w, uint8_t* ws, const UpPlan& pl, float* out4, cudaStream_t s) {
  hdrvae_ctx* ctx = up->ctx;
  const int impl = ctx->conv_impl;
  const int hq = up_net_side(up, h), wq = up_net_side(up, w);
  const int u = up->n_up, hu = hq << u, wu = wq << u;
  const bool crop = up->shuffle * hq != h || up->shuffle * wq != w;
  uint16_t* cat[2] = {reinterpret_cast<uint16_t*>(ws + pl.cat0), reinterpret_cast<uint16_t*>(ws + pl.cat1)};
  float* feat = reinterpret_cast<float*>(ws + pl.f_feat);
  float* fb[3] = {reinterpret_cast<float*>(ws + pl.f_a), reinterpret_cast<float*>(ws + pl.f_b), reinterpret_cast<float*>(ws + pl.f_c)};
  const PackedConv* conv = up->convs.data();          // walked in the order up_pack_rrdb packed them
  int cur = 0;                                        // cat[cur] holds the fp16 copy of the current stream in channels 0..63
  {
    ConvIO io; io.x = ws + pl.img8; io.x_channels = up_in_channels(up->shuffle); io.y = feat; io.y_dtype = DT_F32;
    io.y2 = cat[cur]; io.y2_channels = 192; io.y2_chan_off = 0;
    HDRVAE_TRY(run_conv(ctx, *conv++, io, n, hq, wq, impl, s));
  }
  // fp32 stream buffers: x0 (the RRDB input) lives in feat (first block) or fb[xi]; x1 -> fb[P], x2 -> fb[Q] and the
  // block output overwrites x1's buffer (dead by then), which makes it the next block's x0
  const float* x0 = feat;
  int xi = -1;
  for (int r = 0; r < up->nb; ++r) {
    const int P = (xi + 1) % 3, Q = (xi + 2) % 3;
    float* outs[3] = {fb[P], fb[Q], fb[P]};
    const float* xin = x0;
    for (int k = 0; k < 3; ++k) {
      for (int j = 0; j < 4; ++j) {
        ConvIO io; io.x = cat[cur]; io.x_channels = 192; io.y = cat[cur]; io.y_dtype = DT_F16; io.y_channels = 192;
        io.y_chan_off = 64 + 32 * j; io.lrelu = 0.2f;
        HDRVAE_TRY(run_conv(ctx, *conv++, io, n, hq, wq, impl, s));
      }
      ConvIO io; io.x = cat[cur]; io.x_channels = 192; io.y_dtype = DT_F32; io.y = outs[k];
      io.y2 = cat[cur ^ 1]; io.y2_channels = 192; io.y2_chan_off = 0;
      io.residual = xin; io.res_dtype = DT_F32;
      // k < 2: x_{k+1} = 0.2 conv5 + x_k (weights and bias packed x 0.2); end of the RRDB:
      // (0.2 conv5 + x2) 0.2 + x0 = 0.04 conv5 + 0.2 x2 + x0 (weights and bias packed x 0.04)
      if (k == 2) { io.res_scale = 0.2f; io.residual2 = x0; }
      HDRVAE_TRY(run_conv(ctx, *conv++, io, n, hq, wq, impl, s));
      xin = outs[k];
      cur ^= 1;
    }
    x0 = outs[2];
    xi = P;
  }
  // trunk conv + long skip: t = conv_body(x) + feat; only its fp16 copy is needed (operand of the first upsampling conv,
  // or of conv_hr when there is none)
  {
    ConvIO io; io.x = cat[cur]; io.x_channels = 192; io.y = fb[(xi + 2) % 3]; io.y_dtype = DT_F32;
    io.residual = feat; io.res_dtype = DT_F32; io.y2 = ws + pl.u0;
    HDRVAE_TRY(run_conv(ctx, *conv++, io, n, hq, wq, impl, s));
  }
  uint8_t* hr_in = ws + pl.u0;
  if (u >= 1) {
    ConvIO io; io.x = ws + pl.u0; io.y = ws + pl.u1; io.y_dtype = DT_F16; io.lrelu = 0.2f;
    HDRVAE_TRY(run_conv(ctx, *conv++, io, n, hq, wq, impl, s));
    hr_in = ws + pl.u1;
  }
  if (u >= 2) {
    ConvIO io; io.x = ws + pl.u1; io.y = ws + pl.u2; io.y_dtype = DT_F16; io.lrelu = 0.2f;
    HDRVAE_TRY(run_conv(ctx, *conv++, io, n, 2 * hq, 2 * wq, impl, s));
    hr_in = ws + pl.u2;
  }
  {
    ConvIO io; io.x = hr_in; io.y = ws + pl.u3; io.y_dtype = DT_F16; io.lrelu = 0.2f;
    HDRVAE_TRY(run_conv(ctx, *conv++, io, n, hu, wu, impl, s));
  }
  float* last_out = crop ? reinterpret_cast<float*>(ws + pl.cat0) : out4;     // cat0: 384 bytes per h' w' pixel >= 16 4^u
  {
    ConvIO io; io.x = ws + pl.u3; io.y = last_out; io.y_dtype = DT_F32; io.y_channels = 4; io.n_store = 4;
    HDRVAE_TRY(run_conv(ctx, *conv++, io, n, hu, wu, impl, s));
  }
  if (crop) {
    const int oh = up->scale * h, ow = up->scale * w;
    const long long opx = (long long)n * oh * ow;
    ProfScope prof("upscaler crop padded tiles", 0.0, opx * 32.0, s);
    up_crop_kernel<<<up_grid(opx), 256, 0, s>>>(reinterpret_cast<const float4*>(last_out), hu, wu, n, oh, ow,
                                                reinterpret_cast<float4*>(out4));
    HDRVAE_LAUNCHED();
  }
  return 0;
}

// Compact forward on n tiles (fp16 [n][h][w][8] in pl.img8) -> the last conv's fp32 [n][h][w][up_last_channels] in pl.last
static int up_forward_compact(hdrvae_upscaler* up, int n, int h, int w, uint8_t* ws, const UpPlan& pl, cudaStream_t s) {
  hdrvae_ctx* ctx = up->ctx;
  const int cp = up->convs[0].cout_pad;
  uint8_t* act[2] = {ws + pl.act0, ws + pl.act1};
  const size_t nconv = up->convs.size();
  for (size_t k = 0; k < nconv; ++k) {
    ConvIO io;
    io.x = k == 0 ? ws + pl.img8 : act[(k - 1) & 1];
    io.x_channels = k == 0 ? 8 : cp;
    if (k + 1 < nconv) {
      io.y = act[k & 1]; io.y_dtype = DT_F16; io.y_channels = cp; io.act_slope = up->slopes[k];
    } else {
      io.y = ws + pl.last; io.y_dtype = DT_F32; io.y_channels = up_last_channels(up);
    }
    HDRVAE_TRY(run_conv(ctx, up->convs[k], io, n, h, w, ctx->conv_impl, s));
  }
  return 0;
}

// SPAN forward on n tiles (fp16 [n][h][w][8] x - mean in pl.img8) -> upsampler.0's fp32 [n][h][w][up_last_channels] in
// pl.last.  Every conv is one launch of the conv kernel; conv_1 carries the normalisation's 255 in its weights.  The
// four tensors conv_cat reads are written straight into their channel slices of one fp16 buffer (conv_1 and block_1's
// c3_r as their fp16 operand copy, block_6's c1_r and conv_2 as their output), and the convs that read a slice (block_1,
// block_2, block_6's c2_r) address it through the A operand's base pointer at the slice's first channel with the
// buffer's pixel stride.  The block stream x, which the gate adds, stays fp32.
static int up_forward_span(hdrvae_upscaler* up, int n, int h, int w, uint8_t* ws, const UpPlan& pl, cudaStream_t s) {
  hdrvae_ctx* ctx = up->ctx;
  const int impl = ctx->conv_impl;
  const int nf = up->convs[0].cout, c4 = 4 * nf;
  uint16_t* cat = reinterpret_cast<uint16_t*>(ws + pl.sp_cat);
  float* r[2] = {reinterpret_cast<float*>(ws + pl.sp_r0), reinterpret_cast<float*>(ws + pl.sp_r1)};
  uint8_t* d = ws + pl.sp_d;
  uint8_t* t[2] = {ws + pl.sp_t0, ws + pl.sp_t1};
  {
    ConvIO io; io.x = ws + pl.img8; io.x_channels = 8; io.y = r[0]; io.y_dtype = DT_F32; io.y_channels = nf;
    io.y2 = cat; io.y2_channels = c4; io.y2_chan_off = 0;                                   // f
    HDRVAE_TRY(run_conv(ctx, up->convs[0], io, n, h, w, impl, s));
  }
  const void* xin = cat;                  // the block input's fp16 operand and its pixel stride
  int xch = c4, cur = 0;
  for (int b = 0; b < 6; ++b) {
    const PackedConv* c = &up->convs[1 + 3 * b];
    {
      ConvIO io; io.x = xin; io.x_channels = xch; io.y_dtype = DT_F16; io.act = ACT_SILU;
      if (b == 5) { io.y = cat; io.y_channels = c4; io.y_chan_off = 3 * nf; }           // b5_2: block_6's SiLU'd out1
      else { io.y = t[0]; io.y_channels = nf; }
      HDRVAE_TRY(run_conv(ctx, c[0], io, n, h, w, impl, s));
    }
    {
      ConvIO io; io.x = b == 5 ? static_cast<const void*>(cat + 3 * nf) : t[0]; io.x_channels = b == 5 ? c4 : nf;
      io.y = t[1]; io.y_dtype = DT_F16; io.y_channels = nf; io.act = ACT_SILU;
      HDRVAE_TRY(run_conv(ctx, c[1], io, n, h, w, impl, s));
    }
    {
      // out = (c3_r + x)(sigmoid(c3_r) - 1/2) into the other fp32 stream buffer, its fp16 copy for the next conv
      ConvIO io; io.x = t[1]; io.x_channels = nf; io.y = r[cur ^ 1]; io.y_dtype = DT_F32; io.y_channels = nf;
      io.residual = r[cur]; io.res_dtype = DT_F32; io.act = ACT_GATE;
      if (b == 0) { io.y2 = cat; io.y2_channels = c4; io.y2_chan_off = 2 * nf; xin = cat + 2 * nf; xch = c4; }   // b1
      else { io.y2 = d; io.y2_channels = nf; xin = d; xch = nf; }
      HDRVAE_TRY(run_conv(ctx, c[2], io, n, h, w, impl, s));
      cur ^= 1;
    }
  }
  {
    ConvIO io; io.x = d; io.x_channels = nf; io.y = cat; io.y_dtype = DT_F16; io.y_channels = c4; io.y_chan_off = nf;   // b6
    HDRVAE_TRY(run_conv(ctx, up->convs[19], io, n, h, w, impl, s));
  }
  {
    ConvIO io; io.x = cat; io.x_channels = c4; io.y = t[0]; io.y_dtype = DT_F16; io.y_channels = nf;
    HDRVAE_TRY(run_conv(ctx, up->convs[20], io, n, h, w, impl, s));
  }
  ConvIO io; io.x = t[0]; io.x_channels = nf; io.y = ws + pl.last; io.y_dtype = DT_F32; io.y_channels = up_last_channels(up);
  return run_conv(ctx, up->convs[21], io, n, h, w, impl, s);
}

// SwinIR forward on n tiles of h x w (fp16 [n][hp][wp][8] x - mean in pl.img8, hp / wp: h / w reflect-padded to a multiple
// of 8) -> fp32 [n][s h][s w][4] at out4.  Tokens are the NHWC pixels of the padded tile in raster order, so patch embed /
// unembed are no-ops.  Per STL: LayerNorm -> qkv (1x1 conv) -> window attention (shift 4 in odd blocks) -> proj + the
// residual, in place on the fp32 stream -> LayerNorm -> fc1 + GELU -> fc2 + the residual (the last STL of an RSTB also
// writes the stream's fp16 copy, the RSTB conv's operand).  The RSTB conv (or the 3conv triple) adds the RSTB input.
// After the last RSTB: norm, conv_after_body + conv_first's output, then the tail on the padded grid; the +mean of the
// output is in the last conv's bias (or, for the 1x form, in the base add of the input).  A padded tile's output is cut
// out of the padded grid's with up_crop_kernel.
static int up_forward_swinir(hdrvae_upscaler* up, const float* img, int H, int W, const int4* tiles, int n, int h, int w,
                             uint8_t* ws, const UpPlan& pl, float* out4, cudaStream_t s) {
  hdrvae_ctx* ctx = up->ctx;
  const int impl = ctx->conv_impl;
  const UpSwin& sw = up->sw;
  const int hp = up_net_side(up, h), wp = up_net_side(up, w), sc = up->scale;
  const long long P = (long long)n * hp * wp;
  const bool crop = hp != h || wp != w;
  float* F = reinterpret_cast<float*>(ws + pl.sw_f);
  float* B0 = reinterpret_cast<float*>(ws + pl.sw_b0);
  float* S = reinterpret_cast<float*>(ws + pl.sw_b1);
  uint8_t* a16 = ws + pl.sw_a16;
  uint8_t* b16 = ws + pl.sw_b16;
  const PackedConv* conv = up->convs.data();          // walked in the order up_pack_swinir packed them
  {
    ConvIO io; io.x = ws + pl.img8; io.x_channels = 8; io.y = F; io.y_dtype = DT_F32; io.y_channels = sw.C;
    HDRVAE_TRY(run_conv(ctx, *conv++, io, n, hp, wp, impl, s));
  }
  const float* rin = F;                               // RSTB input (fp32 stream)
  if (sw.patch_norm) {
    HDRVAE_TRY(launch_layernorm(F, P, sw.C, sw.pn_g, sw.pn_b, B0, DT_F32, sw.C, s));
    rin = B0;
  }
  // 3x3 conv (or conv.0 / conv.2 / conv.4 with LeakyReLU 0.2 between) of the fp16 tensor x, + the fp32 residual -> fp32 y
  // [P][C] (the residual shares y's addressing), and its fp16 copy y16 [P][CP] when given
  auto res_conv = [&](const void* x, const float* residual, float* y, void* y16) -> int {
    if (sw.conv3) {
      ConvIO io; io.x = x; io.x_channels = sw.CP; io.y = ws + pl.sw_t0; io.y_dtype = DT_F16; io.y_channels = sw.c4p;
      io.lrelu = 0.2f;
      HDRVAE_TRY(run_conv(ctx, *conv++, io, n, hp, wp, impl, s));
      ConvIO io2; io2.x = ws + pl.sw_t0; io2.x_channels = sw.c4p; io2.y = ws + pl.sw_t1; io2.y_dtype = DT_F16;
      io2.y_channels = sw.c4p; io2.lrelu = 0.2f;
      HDRVAE_TRY(run_conv(ctx, *conv++, io2, n, hp, wp, impl, s));
      x = ws + pl.sw_t1;
    }
    ConvIO io; io.x = x; io.x_channels = sw.conv3 ? sw.c4p : sw.CP; io.y = y; io.y_dtype = DT_F32; io.y_channels = sw.C;
    io.residual = residual; io.res_dtype = DT_F32;
    if (y16 != nullptr) { io.y2 = y16; io.y2_channels = sw.CP; io.y2_chan_off = 0; }
    return run_conv(ctx, *conv++, io, n, hp, wp, impl, s);
  };
  size_t bi = 0;
  for (size_t r = 0; r < sw.depths.size(); ++r) {
    for (int j = 0; j < sw.depths[r]; ++j, ++bi) {
      const UpSwinBlock& b = sw.blocks[bi];
      const float* xin = j == 0 ? rin : S;
      HDRVAE_TRY(launch_layernorm(xin, P, sw.C, b.ln1_g, b.ln1_b, a16, DT_F16, sw.CP, s));
      {
        ConvIO io; io.x = a16; io.x_channels = sw.CP; io.y = ws + pl.sw_qkv; io.y_dtype = DT_F16;
        HDRVAE_TRY(run_conv(ctx, b.qkv, io, n, hp, wp, impl, s));
      }
      HDRVAE_TRY(launch_window_attention(ws + pl.sw_qkv, n, hp, wp, sw.heads, b.table, (j & 1) ? kSwinWin / 2 : 0,
                                         ws + pl.sw_o, s));
      {
        ConvIO io; io.x = ws + pl.sw_o; io.x_channels = sw.heads * 32; io.y = S; io.y_dtype = DT_F32; io.y_channels = sw.C;
        io.residual = xin; io.res_dtype = DT_F32;
        HDRVAE_TRY(run_conv(ctx, b.proj, io, n, hp, wp, impl, s));
      }
      HDRVAE_TRY(launch_layernorm(S, P, sw.C, b.ln2_g, b.ln2_b, a16, DT_F16, sw.CP, s));
      {
        ConvIO io; io.x = a16; io.x_channels = sw.CP; io.y = ws + pl.sw_hid; io.y_dtype = DT_F16; io.y_channels = sw.HP;
        io.act = ACT_GELU;
        HDRVAE_TRY(run_conv(ctx, b.fc1, io, n, hp, wp, impl, s));
      }
      {
        ConvIO io; io.x = ws + pl.sw_hid; io.x_channels = sw.HP; io.y = S; io.y_dtype = DT_F32; io.y_channels = sw.C;
        io.residual = S; io.res_dtype = DT_F32;
        if (j + 1 == sw.depths[r]) { io.y2 = a16; io.y2_channels = sw.CP; io.y2_chan_off = 0; }
        HDRVAE_TRY(run_conv(ctx, b.fc2, io, n, hp, wp, impl, s));
      }
    }
    // RSTB end: conv(stream) + RSTB input, in place on B0 (the first RSTB's input may be conv_first's output F, kept)
    HDRVAE_TRY(res_conv(a16, rin, B0, nullptr));
    rin = B0;
  }
  HDRVAE_TRY(launch_layernorm(rin, P, sw.C, sw.norm_g, sw.norm_b, a16, DT_F16, sw.CP, s));
  HDRVAE_TRY(res_conv(a16, F, S, b16));                   // conv_after_body + conv_first's output (fp16 copy: the tail's input)
  float* o4 = crop ? reinterpret_cast<float*>(ws + pl.sw_out) : out4;   // [n][s hp][s wp] float4
  const int hs = sc * hp, wsd = sc * wp;
  switch (sw.tail) {
    case SW_PIXELSHUFFLE:
    case SW_NEAREST: {
      uint8_t* cur = ws + pl.sw_u0;
      uint8_t* pp[2] = {ws + pl.sw_ua, ws + pl.sw_ub};
      {
        ConvIO io; io.x = b16; io.x_channels = sw.CP; io.y = cur; io.y_dtype = DT_F16; io.lrelu = 0.01f;   // nn.LeakyReLU()
        HDRVAE_TRY(run_conv(ctx, *conv++, io, n, hp, wp, impl, s));
      }
      for (int k = 0; k < sw.n_up; ++k) {
        const int gh = hp << k, gw = wp << k;
        uint8_t* nxt = pp[k & 1];
        if (sw.tail == SW_PIXELSHUFFLE) {
          ConvIO io; io.x = cur; io.y = ws + pl.sw_big; io.y_dtype = DT_F16;
          HDRVAE_TRY(run_conv(ctx, *conv++, io, n, gh, gw, impl, s));
          HDRVAE_TRY(launch_pixel_shuffle2_f16(ws + pl.sw_big, n, gh, gw, 64, nxt, s));
        } else {
          ConvIO io; io.x = cur; io.y = nxt; io.y_dtype = DT_F16; io.lrelu = 0.2f;     // nearest 2x folded into the load
          HDRVAE_TRY(run_conv(ctx, *conv++, io, n, gh, gw, impl, s));
        }
        cur = nxt;
      }
      if (sw.tail == SW_NEAREST) {
        uint8_t* nxt = pp[sw.n_up & 1];
        ConvIO io; io.x = cur; io.y = nxt; io.y_dtype = DT_F16; io.lrelu = 0.2f;
        HDRVAE_TRY(run_conv(ctx, *conv++, io, n, hs, wsd, impl, s));
        cur = nxt;
      }
      ConvIO io; io.x = cur; io.y = o4; io.y_dtype = DT_F32; io.y_channels = 4; io.n_store = 4;
      HDRVAE_TRY(run_conv(ctx, *conv++, io, n, hs, wsd, impl, s));
      break;
    }
    case SW_DIRECT: {
      const int cl = up_last_channels(up);
      ConvIO io; io.x = b16; io.x_channels = sw.CP; io.y = ws + pl.sw_last; io.y_dtype = DT_F32; io.y_channels = cl;
      HDRVAE_TRY(run_conv(ctx, *conv++, io, n, hp, wp, impl, s));
      const long long opx = P * sc * sc;
      ProfScope prof("upscaler pixel shuffle", 0.0, (double)P * cl * 4 + opx * 16, s);
      up_shuffle_base_kernel<<<up_grid(opx), 256, 0, s>>>(reinterpret_cast<const float*>(ws + pl.sw_last), cl, nullptr, H, W,
                                                          tiles, n, hp, wp, sc, reinterpret_cast<float4*>(o4));
      HDRVAE_LAUNCHED();
      break;
    }
    case SW_NONE: {
      // x + conv_last(res): conv_last on the padded grid, cut to the tile, then the base add of the (clamped) input pixel
      float* last = reinterpret_cast<float*>(ws + pl.sw_last);
      ConvIO io; io.x = b16; io.x_channels = sw.CP; io.y = crop ? o4 : last; io.y_dtype = DT_F32; io.y_channels = 4;
      io.n_store = 4;
      HDRVAE_TRY(run_conv(ctx, *conv++, io, n, hp, wp, impl, s));
      const long long opx = (long long)n * h * w;
      if (crop) {
        ProfScope prof("upscaler crop padded tiles", 0.0, opx * 32.0, s);
        up_crop_kernel<<<up_grid(opx), 256, 0, s>>>(reinterpret_cast<const float4*>(o4), hp, wp, n, h, w,
                                                    reinterpret_cast<float4*>(last));
        HDRVAE_LAUNCHED();
      }
      ProfScope prof("upscaler pixel shuffle + base", 0.0, opx * 28.0 + opx * 16, s);
      up_shuffle_base_kernel<<<up_grid(opx), 256, 0, s>>>(last, 4, img, H, W, tiles, n, h, w, 1,
                                                          reinterpret_cast<float4*>(out4));
      HDRVAE_LAUNCHED();
      return 0;
    }
  }
  if (crop) {
    const long long opx = (long long)n * sc * sc * h * w;
    ProfScope prof("upscaler crop padded tiles", 0.0, opx * 32.0, s);
    up_crop_kernel<<<up_grid(opx), 256, 0, s>>>(reinterpret_cast<const float4*>(o4), hs, wsd, n, sc * h, sc * w,
                                                reinterpret_cast<float4*>(out4));
    HDRVAE_LAUNCHED();
  }
  return 0;
}

// The network on n tiles of h x w cut from img [.][H][W][3] at the origins of `tiles` (image, y0, x0, clamp to [-1, 1])
// -> fp32 [n][s h][s w][4] at out4
static int up_run_model(hdrvae_upscaler* up, const float* img, int H, int W, const int4* tiles, int n, int h, int w,
                        uint8_t* ws, const UpPlan& pl, float* out4, cudaStream_t s) {
  {
    const int f = up->shuffle;
    const int hq = up_net_side(up, h), wq = up_net_side(up, w);
    const long long npx = (long long)n * hq * wq;
    ProfScope prof("upscaler extract tiles", 0.0, (double)npx * (f * f * 12 + up_in_channels(f) * 2), s);
    uint4* x = reinterpret_cast<uint4*>(ws + pl.img8);
    const float3 m = up->mean;
    if (f == 1) up_extract_tiles_kernel<1><<<up_grid(npx), 256, 0, s>>>(img, H, W, tiles, n, h, w, hq, wq, 0, m, x);
    else if (f == 2) up_extract_tiles_kernel<2><<<up_grid(npx), 256, 0, s>>>(img, H, W, tiles, n, h, w, hq, wq, 0, m, x);
    else up_extract_tiles_kernel<4><<<up_grid(npx), 256, 0, s>>>(img, H, W, tiles, n, h, w, hq, wq, 0, m, x);
    HDRVAE_LAUNCHED();
  }
  switch (up->arch) {
    case UP_RRDB: return up_forward_rrdb(up, n, h, w, ws, pl, out4, s);
    case UP_COMPACT: HDRVAE_TRY(up_forward_compact(up, n, h, w, ws, pl, s)); break;
    case UP_SPAN: HDRVAE_TRY(up_forward_span(up, n, h, w, ws, pl, s)); break;
    case UP_SWINIR: return up_forward_swinir(up, img, H, W, tiles, n, h, w, ws, pl, out4, s);
  }
  const int sc = up->scale, cl = up_last_channels(up);
  const long long opx = (long long)n * sc * sc * h * w;
  // SPAN adds no base: the plain shuffle
  const bool base = up->arch == UP_COMPACT;
  ProfScope prof(base ? "upscaler pixel shuffle + base" : "upscaler pixel shuffle",
                 0.0, (double)n * h * w * (cl * 4 + (base ? 12 : 0)) + opx * 16, s);
  up_shuffle_base_kernel<<<up_grid(opx), 256, 0, s>>>(reinterpret_cast<const float*>(ws + pl.last), cl,
                                                      base ? img : nullptr, H, W, tiles, n, h, w, sc,
                                                      reinterpret_cast<float4*>(out4));
  HDRVAE_LAUNCHED();
  return 0;
}

}  // namespace hdrvae

// ------------------------------------------------------------------------------------------------ tiling plan
namespace hdrvae {

static const int kUpTile = 512, kUpOverlap = 64;                   // hdr_upscale_with_model.py:115-116
static const long long kUpMaxChunkPx = 8LL * 512 * 512;            // pixels of one forward batch (bounds the workspace: ~14 GB)

struct UpHostTile { int b, y0, x0, h, w; long long off, off2; };
struct UpGroup { int h, w; std::vector<int> tiles; };
// One forward batch: n tiles of a group, both passes at once ([n as-is inputs | n clamped inputs]: the two passes of
// hdr_upscale_with_model.py:181-186 share every launch, which halves the launch count and doubles the small grids)
struct UpChunk { int h, w, first, n; long long out_base; size_t origin0; };

static std::vector<int> up_positions(int size) {
  std::vector<int> p;
  if (size <= kUpTile) { p.push_back(0); return p; }
  for (int v = 0; v < size - kUpOverlap; v += kUpTile - kUpOverlap) p.push_back(v);
  return p;
}

struct UpTiling {
  bool single = false;
  std::vector<UpHostTile> tiles;      // reference accumulation order
  std::vector<UpGroup> groups;        // equal-shape tiles
  std::vector<UpChunk> chunks;        // forward batches
  std::vector<int> order;             // tile indices in chunk order
  long long out_px = 0;               // float4 elements of all tile outputs (both passes)
};

static UpTiling up_make_tiling(int B, int H, int W, int scale) {
  UpTiling t;
  t.single = H <= kUpTile && W <= kUpTile;
  const std::vector<int> py = up_positions(H), px = up_positions(W);
  for (int b = 0; b < B; ++b)
    for (int y : py)
      for (int x : px) {
        UpHostTile u;
        u.b = b;
        u.y0 = std::max(0, std::min(H - kUpOverlap, y)); u.h = std::min(kUpTile, H - u.y0);
        u.x0 = std::max(0, std::min(W - kUpOverlap, x)); u.w = std::min(kUpTile, W - u.x0);
        if (t.single) { u.y0 = u.x0 = 0; u.h = H; u.w = W; }
        u.off = u.off2 = 0;
        t.tiles.push_back(u);
      }
  for (size_t i = 0; i < t.tiles.size(); ++i) {
    const UpHostTile& u = t.tiles[i];
    size_t g = 0;
    for (; g < t.groups.size(); ++g)
      if (t.groups[g].h == u.h && t.groups[g].w == u.w) break;
    if (g == t.groups.size()) { UpGroup ng; ng.h = u.h; ng.w = u.w; t.groups.push_back(ng); }
    t.groups[g].tiles.push_back((int)i);
  }
  long long off = 0;
  for (UpGroup& g : t.groups) {
    const long long per = (long long)g.h * g.w, sz = (long long)scale * scale * per;
    const int cap = (int)std::max<long long>(1, std::min<long long>((long long)g.tiles.size(), kUpMaxChunkPx / (2 * per)));
    for (size_t i0 = 0; i0 < g.tiles.size(); i0 += cap) {
      UpChunk c;
      c.h = g.h; c.w = g.w; c.first = (int)t.order.size(); c.n = (int)std::min<size_t>(cap, g.tiles.size() - i0);
      c.out_base = off; c.origin0 = 2 * (size_t)t.order.size();
      for (int j = 0; j < c.n; ++j) {
        UpHostTile& u = t.tiles[g.tiles[i0 + j]];
        u.off = off + j * sz; u.off2 = off + (c.n + j) * sz;
        t.order.push_back(g.tiles[i0 + j]);
      }
      off += 2 * c.n * sz;
      t.chunks.push_back(c);
    }
  }
  t.out_px = off;
  return t;
}

struct UpWs { size_t descs, origins, out, ycc, tmp, fwd, total; };
static UpWs up_make_ws(const hdrvae_upscaler* up, const UpTiling& t, int B, int H, int W) {
  UpWs w;
  size_t off = 0;
  auto take = [&](size_t bytes) { const size_t o = off; off += (bytes + 1023) / 1024 * 1024; return o; };
  const size_t s2 = (size_t)up->scale * up->scale;
  w.descs = take(t.tiles.size() * sizeof(UpTile));
  w.origins = take(2 * t.tiles.size() * sizeof(int4));
  w.out = take((size_t)t.out_px * 16);
  w.ycc = take((size_t)B * s2 * H * W * 3 * 4);
  w.tmp = take((size_t)B * s2 * H * W * 3 * 4);
  size_t fwd = 0;
  for (const UpChunk& c : t.chunks) fwd = std::max(fwd, up_make_plan(up, 2 * c.n, c.h, c.w).total);
  w.fwd = take(fwd);
  w.total = off;
  return w;
}

// ------------------------------------------------------------------------------------------------ weight shapes
static std::string up_shape_str(const std::vector<int64_t>& sh) {
  std::string r = "[";
  for (size_t i = 0; i < sh.size(); ++i) r += (i ? "," : "") + std::to_string(sh[i]);
  return r + "]";
}

// shape of the staged tensor `key`
static std::string up_shape_str(const hdrvae_ctx* st, const std::string& key) {
  auto it = st->shapes.find(key);
  return it == st->shapes.end() ? std::string("(missing)") : up_shape_str(it->second);
}

// the staged tensor `key` with shape `want`, else an error naming both shapes
static int up_need(const hdrvae_ctx* st, const char* arch, const std::string& key, const std::vector<int64_t>& want) {
  auto it = st->shapes.find(key);
  HDRVAE_REQUIRE(it != st->shapes.end(), "%s upscaler state dict lacks %s (want shape %s)", arch, key.c_str(),
                 up_shape_str(want).c_str());
  HDRVAE_REQUIRE(it->second == want, "%s upscaler: %s has shape %s; want %s", arch, key.c_str(),
                 up_shape_str(it->second).c_str(), up_shape_str(want).c_str());
  return 0;
}

// <key>.weight [cout,cin,ks,ks] and <key>.bias [cout] packed for the conv kernel, the weights scaled by wscale
static int up_pack(hdrvae_ctx* st, const char* arch, const std::string& key, int cout, int cin, int ks, bool upsample,
                   float wscale, PackedConv* pc, cudaStream_t s) {
  HDRVAE_TRY(up_need(st, arch, key + ".weight", {cout, cin, ks, ks}));
  HDRVAE_TRY(up_need(st, arch, key + ".bias", {cout}));
  return pack_conv(st, st->raw[key + ".weight"], st->raw[key + ".bias"], cout, cin, ks, upsample, wscale, DT_F16, pc, s);
}

// nf of the first conv `key` [nf,3,ks,ks]: a multiple of 8 in 8..64
static int up_first_nf(const hdrvae_ctx* st, const char* arch, const std::string& key, int ks, int* nf) {
  auto it = st->shapes.find(key);
  HDRVAE_REQUIRE(it != st->shapes.end() && it->second.size() == 4 && it->second[1] == 3 && it->second[2] == ks &&
                 it->second[3] == ks, "%s upscaler: %s has shape %s; want [nf,3,%d,%d] (3 input channels)", arch,
                 key.c_str(), up_shape_str(st, key).c_str(), ks, ks);
  *nf = (int)it->second[0];
  HDRVAE_REQUIRE(*nf >= 8 && *nf <= 64 && *nf % 8 == 0, "%s upscaler: %s has shape %s; nf must be a multiple of 8 in 8..64",
                 arch, key.c_str(), up_shape_str(it->second).c_str());
  return 0;
}

// scale s of the output conv `key` [3 s^2,nf,3,3] (the pixel shuffle's input): 1, 2 or 4
static int up_out_scale(const hdrvae_ctx* st, const char* arch, const std::string& key, int nf, int* scale) {
  auto it = st->shapes.find(key);
  const int64_t c = it != st->shapes.end() && it->second.size() == 4 && it->second[1] == nf && it->second[2] == 3 &&
                    it->second[3] == 3 ? it->second[0] : 0;
  HDRVAE_REQUIRE(c == 3 || c == 12 || c == 48, "%s upscaler: %s has shape %s; want [3*scale^2,%d,3,3] with scale 1, 2 or 4",
                 arch, key.c_str(), up_shape_str(st, key).c_str(), nf);
  *scale = c == 3 ? 1 : c == 12 ? 2 : 4;
  return 0;
}

}  // namespace hdrvae

// ------------------------------------------------------------------------------------------------ C ABI
extern "C" {

int hdrvae_upscaler_create(hdrvae_ctx* ctx, hdrvae_upscaler** out) {
  HDRVAE_REQUIRE(ctx != nullptr && out != nullptr, "hdrvae_upscaler_create: null argument");
  hdrvae_upscaler* up = new hdrvae_upscaler();
  up->ctx = ctx;
  up->store.device = ctx->device; up->store.num_sms = ctx->num_sms;
  *out = up;
  return 0;
}

int hdrvae_upscaler_destroy(hdrvae_upscaler* up) {
  if (up == nullptr) return 0;
  cudaSetDevice(up->store.device);
  for (void* p : up->store.owned) cudaFree(p);
  delete up;
  return 0;
}

// Top-level conv index K of an old-arch key "model.K.weight" / "model.K.bias" (K != 1, the trunk), else -1.
static int up_old_top_index(const std::string& k) {
  int K = -1, len = 0;
  if (sscanf(k.c_str(), "model.%d.%n", &K, &len) != 1 || len == 0 || K == 1) return -1;
  const std::string leaf = k.substr(len);
  return leaf == "weight" || leaf == "bias" ? K : -1;
}

// Canonical (Real-ESRGAN) name of a state-dict key given in either layout; "" if it is not an RRDBNet tensor.
// BasicSR's sequential() flattens each upsampling stage into (Upsample, conv, LeakyReLU) and conv_hr into (conv,
// LeakyReLU), so with u upsampling convs the old-arch top-level convs sit at 0 (conv_first), 3 + 3k (conv_up{k+1}),
// 3u + 2 (conv_hr) and 3u + 4 (conv_last).
static std::string up_canonical(const std::string& k, int n_up) {
  if (k.compare(0, 6, "model.") != 0) return k;
  auto leaf = k.substr(k.rfind('.') + 1);
  const std::string head = k.substr(0, k.rfind('.'));
  const int K = up_old_top_index(k);
  if (K >= 0) {
    if (K == 0) return "conv_first." + leaf;
    if (K >= 3 && K < 3 + 3 * n_up && K % 3 == 0) return "conv_up" + std::to_string(K / 3) + "." + leaf;
    if (K == 3 * n_up + 2) return "conv_hr." + leaf;
    if (K == 3 * n_up + 4) return "conv_last." + leaf;
    return "";
  }
  int i = -1, r = -1, c = -1;
  if (sscanf(head.c_str(), "model.1.sub.%d.RDB%d.conv%d.0", &i, &r, &c) == 3)
    return "body." + std::to_string(i) + ".rdb" + std::to_string(r) + ".conv" + std::to_string(c) + "." + leaf;
  if (sscanf(head.c_str(), "model.1.sub.%d", &i) == 1 && head == "model.1.sub." + std::to_string(i)) return "conv_body." + leaf;
  return "";
}

// Upsampling convs of an RRDBNet state dict, found before any key is mapped: from the highest old-arch top-level conv
// index (conv_last sits at 3u + 4; its weight's key and shape in *top_key / *top_shape), else from the Real-ESRGAN
// conv_up1 / conv_up2 / conv_up3 names.  -1: an old-arch layout whose conv_last index fits no u.
static int up_count_upconvs(const hdrvae_weight_desc* descs, int n, std::string* top_key, std::string* top_shape) {
  int top = -1, named = 0;
  for (int i = 0; i < n; ++i) {
    const hdrvae_weight_desc& d = descs[i];
    if (d.name == nullptr || d.ndim < 1 || d.ndim > 4) continue;      // refused by the load loop
    const std::string k = d.name;
    const int K = up_old_top_index(k);
    if (K > top) { top = K; *top_key = "model." + std::to_string(K) + ".weight"; *top_shape = "(missing)"; }
    if (k == *top_key) *top_shape = up_shape_str(std::vector<int64_t>(d.shape, d.shape + d.ndim));
    for (int j = 1; j <= 3; ++j)
      if (k == "conv_up" + std::to_string(j) + ".weight") named = std::max(named, j);
  }
  if (top < 0) return named;
  return top >= 4 && (top - 4) % 3 == 0 ? (top - 4) / 3 : -1;
}

// Real-ESRGAN SRVGGNetCompact as spandrel loads it with act_type "prelu": body.0 = conv 3 -> nf, body.{2k+1} = PReLU
// slopes [nf] (k = 0..nc), body.{2+2m} = conv nf -> nf (m < nc), body.{2nc+2} = conv nf -> 3 s^2.  The scale s is
// limited to powers of two (1, 2, 4): only there do the local fix's resampling coordinates (dst + 0.5) / s equal torch's.
static int up_pack_compact(hdrvae_upscaler* up, cudaStream_t s) {
  hdrvae_ctx* st = &up->store;
  int last = -1;
  for (const auto& kv : st->shapes) {
    int bi = -1;
    if (sscanf(kv.first.c_str(), "body.%d.", &bi) == 1) last = std::max(last, bi);
  }
  HDRVAE_REQUIRE(last >= 2 && last % 2 == 0,
                 "Compact upscaler: the highest body index is %d; the last conv must sit at an even index >= 2", last);
  const int nc = (last - 2) / 2;
  int nf = 0;
  HDRVAE_TRY(up_first_nf(st, "Compact", "body.0.weight", 3, &nf));
  HDRVAE_TRY(up_out_scale(st, "Compact", "body." + std::to_string(last) + ".weight", nf, &up->scale));
  up->nb = nc;
  up->convs.resize((size_t)nc + 2);
  HDRVAE_TRY(up_pack(st, "Compact", "body.0", nf, 3, 3, false, 1.f, &up->convs[0], s));
  for (int m = 0; m < nc; ++m)
    HDRVAE_TRY(up_pack(st, "Compact", "body." + std::to_string(2 + 2 * m), nf, nf, 3, false, 1.f, &up->convs[1 + m], s));
  HDRVAE_TRY(up_pack(st, "Compact", "body." + std::to_string(last), 3 * up->scale * up->scale, nf, 3, false, 1.f,
                     &up->convs[nc + 1], s));
  const int cp = up->convs[0].cout_pad;
  for (int k = 0; k <= nc; ++k) {
    const std::string key = "body." + std::to_string(2 * k + 1) + ".weight";
    auto it = st->shapes.find(key);
    HDRVAE_REQUIRE(it != st->shapes.end(), "Compact upscaler state dict lacks the PReLU slopes %s (only act_type \"prelu\" is "
                   "supported)", key.c_str());
    HDRVAE_REQUIRE(it->second.size() == 1 && it->second[0] == nf, "Compact upscaler: %s has shape %s; want [%d] (one PReLU "
                   "slope per channel)", key.c_str(), up_shape_str(it->second).c_str(), nf);
    float* slope = nullptr;
    HDRVAE_TRY(dev_alloc(st, cp * sizeof(float), (void**)&slope));
    HDRVAE_CUDA_OK(cudaMemsetAsync(slope, 0, cp * sizeof(float), s));
    HDRVAE_CUDA_OK(cudaMemcpyAsync(slope, st->raw[key], nf * sizeof(float), cudaMemcpyDeviceToDevice, s));
    up->slopes.push_back(slope);
  }
  return 0;
}

// SPAN (spandrel's "SPAN"; hongyuanyu/SPAN) as spandrel loads it: conv_1, block_1 .. block_6 (c1_r, c2_r, c3_r), conv_2 —
// each a Conv3XC — then conv_cat (1x1, 4 nf -> nf) and upsampler.0 (3x3, nf -> 3 s^2, then the pixel shuffle); the
// buffer no_norm switches the input normalisation (x - mean) 255 off.  A Conv3XC in eval mode rebuilds eval_conv from
// sk (1x1, cin -> cout), conv.0 (1x1, cin -> m1), conv.1 (3x3, m1 -> m2) and conv.2 (1x1, m2 -> cout) on every forward
// and runs eval_conv with zero padding 1; the stored eval_conv.* may be stale, so the same fusion happens here, in fp64:
//   W = w3 . w2 . w1 (+ sk at the centre tap),  b = w3 (sum_{m1,taps} w2 b1 + b2) + b3 + b_sk.
static int up_pack_span(hdrvae_upscaler* up, cudaStream_t s) {
  hdrvae_ctx* st = &up->store;
  auto host = [&](const std::string& k, std::vector<double>* out) -> int {
    size_t cnt = 1;
    for (int64_t d : st->shapes[k]) cnt *= (size_t)d;
    std::vector<float> f(cnt);
    HDRVAE_CUDA_OK(cudaMemcpy(f.data(), st->raw[k], cnt * sizeof(float), cudaMemcpyDeviceToHost));
    out->assign(f.begin(), f.end());
    return 0;
  };
  int nf = 0;
  HDRVAE_TRY(up_first_nf(st, "SPAN", "conv_1.sk.weight", 1, &nf));
  for (const auto& kv : st->shapes) {
    int bi = -1;
    HDRVAE_REQUIRE(sscanf(kv.first.c_str(), "block_%d.", &bi) != 1 || (bi >= 1 && bi <= 6),
                   "SPAN upscaler: %s has shape %s; SPAN has exactly the blocks block_1 .. block_6", kv.first.c_str(),
                   up_shape_str(kv.second).c_str());
  }
  HDRVAE_TRY(up_out_scale(st, "SPAN", "upsampler.0.weight", nf, &up->scale));
  const bool norm = st->shapes.count("no_norm") == 0;
  // Conv3XC `pre` (cin -> cout) fused into one 3x3 conv, packed with its weights scaled by wscale
  auto conv3xc = [&](const std::string& pre, int cin, int cout, float wscale, PackedConv* pc) -> int {
    auto it = st->shapes.find(pre + ".conv.0.weight");
    const int m1 = it != st->shapes.end() && it->second.size() == 4 ? (int)it->second[0] : 0;
    it = st->shapes.find(pre + ".conv.1.weight");
    const int m2 = it != st->shapes.end() && it->second.size() == 4 ? (int)it->second[0] : 0;
    HDRVAE_REQUIRE(m1 >= 1 && m2 >= 1, "SPAN upscaler: %s.conv.0.weight has shape %s and %s.conv.1.weight %s; want [m1,%d,1,1] "
                   "and [m2,m1,3,3]", pre.c_str(), up_shape_str(st, pre + ".conv.0.weight").c_str(), pre.c_str(),
                   up_shape_str(st, pre + ".conv.1.weight").c_str(), cin);
    HDRVAE_TRY(up_need(st, "SPAN", pre + ".sk.weight", {cout, cin, 1, 1}));
    HDRVAE_TRY(up_need(st, "SPAN", pre + ".sk.bias", {cout}));
    HDRVAE_TRY(up_need(st, "SPAN", pre + ".conv.0.weight", {m1, cin, 1, 1}));
    HDRVAE_TRY(up_need(st, "SPAN", pre + ".conv.0.bias", {m1}));
    HDRVAE_TRY(up_need(st, "SPAN", pre + ".conv.1.weight", {m2, m1, 3, 3}));
    HDRVAE_TRY(up_need(st, "SPAN", pre + ".conv.1.bias", {m2}));
    HDRVAE_TRY(up_need(st, "SPAN", pre + ".conv.2.weight", {cout, m2, 1, 1}));
    HDRVAE_TRY(up_need(st, "SPAN", pre + ".conv.2.bias", {cout}));
    std::vector<double> sk, skb, w1, b1, w2, b2, w3, b3;
    HDRVAE_TRY(host(pre + ".sk.weight", &sk)); HDRVAE_TRY(host(pre + ".sk.bias", &skb));
    HDRVAE_TRY(host(pre + ".conv.0.weight", &w1)); HDRVAE_TRY(host(pre + ".conv.0.bias", &b1));
    HDRVAE_TRY(host(pre + ".conv.1.weight", &w2)); HDRVAE_TRY(host(pre + ".conv.1.bias", &b2));
    HDRVAE_TRY(host(pre + ".conv.2.weight", &w3)); HDRVAE_TRY(host(pre + ".conv.2.bias", &b3));
    // a[m2][i][tap] = sum_m1 w2[m2][m1][tap] w1[m1][i];  bm[m2] = sum_{m1,tap} w2[m2][m1][tap] b1[m1] + b2[m2]
    std::vector<double> a((size_t)m2 * cin * 9, 0.0), bm(m2);
    for (int o = 0; o < m2; ++o) {
      double acc = b2[o];
      for (int j = 0; j < m1; ++j)
        for (int k = 0; k < 9; ++k) {
          const double v = w2[((size_t)o * m1 + j) * 9 + k];
          acc += v * b1[j];
          for (int i = 0; i < cin; ++i) a[((size_t)o * cin + i) * 9 + k] += v * w1[(size_t)j * cin + i];
        }
      bm[o] = acc;
    }
    std::vector<float> wf((size_t)cout * cin * 9), bf(cout);
    for (int o = 0; o < cout; ++o) {
      double acc = b3[o] + skb[o];
      for (int m = 0; m < m2; ++m) acc += w3[(size_t)o * m2 + m] * bm[m];
      bf[o] = (float)acc;
      for (int i = 0; i < cin; ++i)
        for (int k = 0; k < 9; ++k) {
          double v = k == 4 ? sk[(size_t)o * cin + i] : 0.0;
          for (int m = 0; m < m2; ++m) v += w3[(size_t)o * m2 + m] * a[((size_t)m * cin + i) * 9 + k];
          wf[((size_t)o * cin + i) * 9 + k] = (float)v;
        }
    }
    // device copies under the fp32 state-dict map, so that up_finish_load frees them with the rest
    float *dw = nullptr, *db = nullptr;
    HDRVAE_TRY(dev_alloc(st, wf.size() * sizeof(float), (void**)&dw));
    HDRVAE_TRY(dev_alloc(st, bf.size() * sizeof(float), (void**)&db));
    st->raw[pre + ".fused.weight"] = dw;
    st->raw[pre + ".fused.bias"] = db;
    HDRVAE_CUDA_OK(cudaMemcpy(dw, wf.data(), wf.size() * sizeof(float), cudaMemcpyHostToDevice));
    HDRVAE_CUDA_OK(cudaMemcpy(db, bf.data(), bf.size() * sizeof(float), cudaMemcpyHostToDevice));
    return pack_conv(st, dw, db, cout, cin, 3, false, wscale, DT_F16, pc, s);
  };
  up->convs.resize(22);
  // (x - mean) 255: the input stage subtracts the mean, conv_1's weights carry the 255 (its bias is not scaled)
  HDRVAE_TRY(conv3xc("conv_1", 3, nf, norm ? 255.f : 1.f, &up->convs[0]));
  for (int b = 0; b < 6; ++b)
    for (int c = 0; c < 3; ++c)
      HDRVAE_TRY(conv3xc("block_" + std::to_string(b + 1) + ".c" + std::to_string(c + 1) + "_r", nf, nf, 1.f,
                         &up->convs[1 + 3 * b + c]));
  HDRVAE_TRY(conv3xc("conv_2", nf, nf, 1.f, &up->convs[19]));
  HDRVAE_TRY(up_pack(st, "SPAN", "conv_cat", nf, 4 * nf, 1, false, 1.f, &up->convs[20], s));
  HDRVAE_TRY(up_pack(st, "SPAN", "upsampler.0", 3 * up->scale * up->scale, nf, 3, false, 1.f, &up->convs[21], s));
  if (norm) up->mean = make_float3(0.4488f, 0.4371f, 0.4040f);
  up->nb = 6;
  return 0;
}

// SwinIR (spandrel's "SwinIR": JingyunLiang/SwinIR network_swinir.py) with 3 input channels, embed_dim C <= 256, head dim
// C / heads <= 32, window 8, any RSTB count and depths, any MLP width, resi_connection "1conv" / "3conv", with or without
// patch_embed.norm, no absolute_pos_embed, and the upsamplers "pixelshuffle" (2x, 4x), "pixelshuffledirect" (2x, 4x),
// "nearest+conv" (2x, 4x) and "" (1x).  The stored relative_position_index and attn_mask buffers are not read: the index is
// a function of the window, and the mask is computed for each tile's padded size (window_attention_kernel).  HAT shares
// SwinIR's key prefix and is refused by its own keys.
static const char* kSwinKey = "layers.0.residual_group.blocks.0.attn.relative_position_bias_table";
static int up_pack_swinir(hdrvae_upscaler* up, cudaStream_t s) {
  hdrvae_ctx* st = &up->store;
  UpSwin& sw = up->sw;
  const char* A = "SwinIR";
  for (const auto& kv : st->shapes) {
    const std::string& k = kv.first;
    HDRVAE_REQUIRE(k.find("conv_block") == std::string::npos && k.find("overlap_attn") == std::string::npos &&
                   k.find("relative_position_index_SA") == std::string::npos,
                   "SwinIR upscaler: %s has shape %s: a HAT model (conv_block / overlap_attn / relative_position_index_SA "
                   "keys); HAT is not supported", k.c_str(), up_shape_str(kv.second).c_str());
    HDRVAE_REQUIRE(k != "absolute_pos_embed", "SwinIR upscaler: absolute_pos_embed has shape %s; models with ape (an "
                   "absolute position embedding) are not supported", up_shape_str(kv.second).c_str());
  }
  auto shape = [&](const std::string& k) -> const std::vector<int64_t>* {
    auto it = st->shapes.find(k);
    return it == st->shapes.end() ? nullptr : &it->second;
  };
  auto host = [&](const std::string& k, std::vector<float>* out) -> int {
    size_t cnt = 1;
    for (int64_t d : st->shapes[k]) cnt *= (size_t)d;
    out->resize(cnt);
    HDRVAE_CUDA_OK(cudaMemcpy(out->data(), st->raw[k], cnt * sizeof(float), cudaMemcpyDeviceToHost));
    return 0;
  };
  // a device copy of the staged tensor `k` that outlives the staging (LayerNorm parameters, bias tables)
  auto keep = [&](const std::string& k, size_t cnt, float** out) -> int {
    HDRVAE_TRY(dev_alloc(st, cnt * sizeof(float), (void**)out));
    HDRVAE_CUDA_OK(cudaMemcpyAsync(*out, st->raw[k], cnt * sizeof(float), cudaMemcpyDeviceToDevice, s));
    return 0;
  };
  // host fp32 weights [cout][cin][ks][ks] and bias [cout] packed for the conv kernel (kept under the fp32 state-dict map, so
  // that up_finish_load frees them with the rest)
  auto pack_host = [&](const std::string& k, const std::vector<float>& wf, const std::vector<float>& bf, int cout, int cin,
                       int ks, PackedConv* pc) -> int {
    float *dw = nullptr, *db = nullptr;
    HDRVAE_TRY(dev_alloc(st, wf.size() * sizeof(float), (void**)&dw));
    HDRVAE_TRY(dev_alloc(st, bf.size() * sizeof(float), (void**)&db));
    st->raw[k + ".packed.weight"] = dw;
    st->raw[k + ".packed.bias"] = db;
    HDRVAE_CUDA_OK(cudaMemcpy(dw, wf.data(), wf.size() * sizeof(float), cudaMemcpyHostToDevice));
    HDRVAE_CUDA_OK(cudaMemcpy(db, bf.data(), bf.size() * sizeof(float), cudaMemcpyHostToDevice));
    return pack_conv(st, dw, db, cout, cin, ks, false, 1.f, DT_F16, pc, s);
  };
  // nn.Linear `k` [out][in] + bias [out], packed as a 1x1 conv
  auto linear = [&](const std::string& k, int out, int in, PackedConv* pc) -> int {
    HDRVAE_TRY(up_need(st, A, k + ".weight", {out, in}));
    HDRVAE_TRY(up_need(st, A, k + ".bias", {out}));
    return pack_conv(st, st->raw[k + ".weight"], st->raw[k + ".bias"], out, in, 1, false, 1.f, DT_F16, pc, s);
  };
  // + mean in the bias of the conv that produces the output colours (channel o belongs to colour o / per)
  auto add_mean = [&](PackedConv* pc, int cout, int per) -> int {
    std::vector<float> b(cout);
    HDRVAE_CUDA_OK(cudaMemcpy(b.data(), pc->bias, cout * sizeof(float), cudaMemcpyDeviceToHost));
    const float m[3] = {up->mean.x, up->mean.y, up->mean.z};
    for (int o = 0; o < cout; ++o) b[o] += m[o / per];
    HDRVAE_CUDA_OK(cudaMemcpy(pc->bias, b.data(), cout * sizeof(float), cudaMemcpyHostToDevice));
    return 0;
  };
  const std::vector<int64_t>* cf = shape("conv_first.weight");
  HDRVAE_REQUIRE(cf != nullptr && cf->size() == 4 && (*cf)[0] >= 1 && (*cf)[0] <= 256 && (*cf)[1] == 3 && (*cf)[2] == 3 &&
                 (*cf)[3] == 3, "SwinIR upscaler: conv_first.weight has shape %s; want [embed_dim,3,3,3] with embed_dim "
                 "<= 256 (3 input channels)", up_shape_str(st, "conv_first.weight").c_str());
  const int C = (int)(*cf)[0];
  sw.C = C;
  sw.CP = (C + 7) / 8 * 8;
  const std::vector<int64_t>* tb = shape(kSwinKey);
  HDRVAE_REQUIRE(tb->size() == 2 && (*tb)[0] == 225 && (*tb)[1] >= 1, "SwinIR upscaler: %s has shape %s; want [225,heads] "
                 "(window size 8: (2 ws - 1)^2 rows)", kSwinKey, up_shape_str(*tb).c_str());
  sw.heads = (int)(*tb)[1];
  HDRVAE_REQUIRE(C % sw.heads == 0 && C / sw.heads <= 32, "SwinIR upscaler: %s has shape %s: embed_dim %d over %d heads; "
                 "the head dimension must divide embed_dim and be at most 32", kSwinKey, up_shape_str(*tb).c_str(), C, sw.heads);
  const int hd = C / sw.heads;
  const std::string b00 = "layers.0.residual_group.blocks.0.";
  const std::vector<int64_t>* f1 = shape(b00 + "mlp.fc1.weight");
  HDRVAE_REQUIRE(f1 != nullptr && f1->size() == 2 && (*f1)[0] >= 1 && (*f1)[1] == C, "SwinIR upscaler: %smlp.fc1.weight has "
                 "shape %s; want [hidden,%d]", b00.c_str(), up_shape_str(st, b00 + "mlp.fc1.weight").c_str(), C);
  sw.hidden = (int)(*f1)[0];
  sw.HP = (sw.hidden + 7) / 8 * 8;
  sw.conv3 = shape("layers.0.conv.weight") == nullptr && shape("layers.0.conv.0.weight") != nullptr;
  sw.c4 = C / 4;
  sw.c4p = (sw.c4 + 7) / 8 * 8;
  HDRVAE_REQUIRE(!sw.conv3 || sw.c4 >= 1, "SwinIR upscaler: embed_dim %d is too small for resi_connection \"3conv\"", C);
  sw.patch_norm = shape("patch_embed.norm.weight") != nullptr;
  // RSTBs layers.i and their blocks layers.i.residual_group.blocks.j
  int nl = 0;
  for (const auto& kv : st->shapes) {
    int i = -1;
    if (sscanf(kv.first.c_str(), "layers.%d.", &i) == 1) nl = std::max(nl, i + 1);
  }
  sw.depths.assign(nl, 0);
  for (const auto& kv : st->shapes) {
    int i = -1, j = -1;
    if (sscanf(kv.first.c_str(), "layers.%d.residual_group.blocks.%d.", &i, &j) == 2 && i >= 0 && j >= 0)
      sw.depths[i] = std::max(sw.depths[i], j + 1);
  }
  for (int i = 0; i < nl; ++i)
    HDRVAE_REQUIRE(sw.depths[i] >= 1, "SwinIR upscaler state dict lacks layers.%d.residual_group.blocks.0.* (every RSTB "
                   "needs at least one Swin transformer layer)", i);
  // upsampler and scale
  int scale = 1;
  if (shape("conv_up1.weight") != nullptr) {
    sw.tail = SW_NEAREST;
    sw.n_up = shape("conv_up2.weight") != nullptr ? 2 : 1;
  } else if (shape("conv_before_upsample.0.weight") != nullptr) {
    sw.tail = SW_PIXELSHUFFLE;
    HDRVAE_TRY(up_need(st, A, "upsample.0.weight", {256, 64, 3, 3}));
    HDRVAE_REQUIRE(shape("upsample.4.weight") == nullptr, "SwinIR upscaler: upsample.4.weight has shape %s: a third 2x stage "
                   "(an 8x SwinIR) is not supported; SwinIR runs at 1x, 2x and 4x", up_shape_str(st, "upsample.4.weight").c_str());
    sw.n_up = shape("upsample.2.weight") != nullptr ? 2 : 1;
  } else if (shape("upsample.0.weight") != nullptr) {
    sw.tail = SW_DIRECT;
    const std::vector<int64_t>* u = shape("upsample.0.weight");
    const int64_t c = u->size() == 4 && (*u)[1] == C && (*u)[2] == 3 && (*u)[3] == 3 ? (*u)[0] : 0;
    HDRVAE_REQUIRE(c == 12 || c == 48, "SwinIR upscaler: upsample.0.weight has shape %s; want [3*scale^2,%d,3,3] with "
                   "scale 2 or 4", up_shape_str(*u).c_str(), C);
    scale = c == 12 ? 2 : 4;
  } else {
    sw.tail = SW_NONE;
  }
  if (sw.tail == SW_NEAREST || sw.tail == SW_PIXELSHUFFLE) scale = 1 << sw.n_up;
  up->scale = scale;
  up->mean = make_float3(0.4488f, 0.4371f, 0.4040f);       // in_chans 3: the RGB mean; img_range 1
  // packing, in launch order
  auto res_convs = [&](const std::string& k) -> int {     // RSTB conv / conv_after_body: 1conv or 3conv
    if (!sw.conv3) {
      up->convs.emplace_back();
      return up_pack(st, A, k, C, C, 3, false, 1.f, &up->convs.back(), s);
    }
    up->convs.emplace_back();
    HDRVAE_TRY(up_pack(st, A, k + ".0", sw.c4, C, 3, false, 1.f, &up->convs.back(), s));
    up->convs.emplace_back();
    HDRVAE_TRY(up_pack(st, A, k + ".2", sw.c4, sw.c4, 1, false, 1.f, &up->convs.back(), s));
    up->convs.emplace_back();
    return up_pack(st, A, k + ".4", C, sw.c4, 3, false, 1.f, &up->convs.back(), s);
  };
  up->convs.reserve(2 + 3 * (size_t)nl + 3 + 6);
  up->convs.emplace_back();
  HDRVAE_TRY(up_pack(st, A, "conv_first", C, 3, 3, false, 1.f, &up->convs.back(), s));
  if (sw.patch_norm) {
    HDRVAE_TRY(up_need(st, A, "patch_embed.norm.weight", {C}));
    HDRVAE_TRY(up_need(st, A, "patch_embed.norm.bias", {C}));
    HDRVAE_TRY(keep("patch_embed.norm.weight", C, &sw.pn_g));
    HDRVAE_TRY(keep("patch_embed.norm.bias", C, &sw.pn_b));
  }
  const float qscale = (float)(1.0 / sqrt((double)hd));
  const int QK = sw.heads * 32;                            // columns of q (and of k, v, and the attention output)
  for (int i = 0; i < nl; ++i) {
    for (int j = 0; j < sw.depths[i]; ++j) {
      const std::string b = "layers." + std::to_string(i) + ".residual_group.blocks." + std::to_string(j) + ".";
      UpSwinBlock blk;
      for (const char* nm : {"norm1.weight", "norm1.bias", "norm2.weight", "norm2.bias"}) HDRVAE_TRY(up_need(st, A, b + nm, {C}));
      HDRVAE_TRY(up_need(st, A, b + "attn.relative_position_bias_table", {225, sw.heads}));
      HDRVAE_TRY(keep(b + "norm1.weight", C, &blk.ln1_g)); HDRVAE_TRY(keep(b + "norm1.bias", C, &blk.ln1_b));
      HDRVAE_TRY(keep(b + "norm2.weight", C, &blk.ln2_g)); HDRVAE_TRY(keep(b + "norm2.bias", C, &blk.ln2_b));
      HDRVAE_TRY(keep(b + "attn.relative_position_bias_table", 225 * (size_t)sw.heads, &blk.table));
      // qkv [3C][C] -> [3][heads][32][C], q rows and bias x hd^-0.5, rows d >= hd of a head zero
      HDRVAE_TRY(up_need(st, A, b + "attn.qkv.weight", {3 * C, C}));
      HDRVAE_TRY(up_need(st, A, b + "attn.qkv.bias", {3 * C}));
      std::vector<float> w, bias;
      HDRVAE_TRY(host(b + "attn.qkv.weight", &w));
      HDRVAE_TRY(host(b + "attn.qkv.bias", &bias));
      std::vector<float> wq((size_t)3 * QK * C, 0.f), bq((size_t)3 * QK, 0.f);
      for (int q = 0; q < 3; ++q)
        for (int hh = 0; hh < sw.heads; ++hh)
          for (int d = 0; d < hd; ++d) {
            const int src = q * C + hh * hd + d, dst = (q * sw.heads + hh) * 32 + d;
            const float f = q == 0 ? qscale : 1.f;
            for (int c = 0; c < C; ++c) wq[(size_t)dst * C + c] = w[(size_t)src * C + c] * f;
            bq[dst] = bias[src] * f;
          }
      HDRVAE_TRY(pack_host(b + "attn.qkv", wq, bq, 3 * QK, C, 1, &blk.qkv));
      // proj [C][C] -> [C][heads * 32]: input channel h hd + d moves to h 32 + d
      HDRVAE_TRY(up_need(st, A, b + "attn.proj.weight", {C, C}));
      HDRVAE_TRY(up_need(st, A, b + "attn.proj.bias", {C}));
      HDRVAE_TRY(host(b + "attn.proj.weight", &w));
      HDRVAE_TRY(host(b + "attn.proj.bias", &bias));
      std::vector<float> wp((size_t)C * QK, 0.f);
      for (int o = 0; o < C; ++o)
        for (int hh = 0; hh < sw.heads; ++hh)
          for (int d = 0; d < hd; ++d) wp[(size_t)o * QK + hh * 32 + d] = w[(size_t)o * C + hh * hd + d];
      HDRVAE_TRY(pack_host(b + "attn.proj", wp, bias, C, QK, 1, &blk.proj));
      HDRVAE_TRY(linear(b + "mlp.fc1", sw.hidden, C, &blk.fc1));
      HDRVAE_TRY(linear(b + "mlp.fc2", C, sw.hidden, &blk.fc2));
      sw.blocks.push_back(blk);
    }
    HDRVAE_TRY(res_convs("layers." + std::to_string(i) + ".conv"));
  }
  HDRVAE_TRY(up_need(st, A, "norm.weight", {C}));
  HDRVAE_TRY(up_need(st, A, "norm.bias", {C}));
  HDRVAE_TRY(keep("norm.weight", C, &sw.norm_g));
  HDRVAE_TRY(keep("norm.bias", C, &sw.norm_b));
  HDRVAE_TRY(res_convs("conv_after_body"));
  auto add = [&](const std::string& k, int cout, int cin, bool upsample) -> int {
    up->convs.emplace_back();
    return up_pack(st, A, k, cout, cin, 3, upsample, 1.f, &up->convs.back(), s);
  };
  switch (sw.tail) {
    case SW_PIXELSHUFFLE:
      HDRVAE_TRY(add("conv_before_upsample.0", 64, C, false));
      for (int k = 0; k < sw.n_up; ++k) HDRVAE_TRY(add("upsample." + std::to_string(2 * k), 256, 64, false));
      HDRVAE_TRY(add("conv_last", 3, 64, false));
      HDRVAE_TRY(add_mean(&up->convs.back(), 3, 1));
      break;
    case SW_NEAREST:
      HDRVAE_TRY(add("conv_before_upsample.0", 64, C, false));
      for (int k = 1; k <= sw.n_up; ++k) HDRVAE_TRY(add("conv_up" + std::to_string(k), 64, 64, true));
      HDRVAE_TRY(add("conv_hr", 64, 64, false));
      HDRVAE_TRY(add("conv_last", 3, 64, false));
      HDRVAE_TRY(add_mean(&up->convs.back(), 3, 1));
      break;
    case SW_DIRECT:
      HDRVAE_TRY(add("upsample.0", 3 * scale * scale, C, false));
      HDRVAE_TRY(add_mean(&up->convs.back(), 3 * scale * scale, scale * scale));
      break;
    case SW_NONE:
      HDRVAE_TRY(add("conv_last", 3, C, false));          // the mean comes back with the input in the base add
      break;
  }
  up->nb = nl;
  return 0;
}

// ESRGAN / RRDBNet (nf 64, gc 32) in Real-ESRGAN names (staging mapped the old-arch keys): conv_first, nb RRDBs of three
// dense blocks (conv1 .. conv5), conv_body, n_up upsampling convs, conv_hr, conv_last.  n_up, top_*: up_count_upconvs.
static int up_pack_rrdb(hdrvae_upscaler* up, int n_up, const std::string& top_key, const std::string& top_shape,
                        cudaStream_t s) {
  hdrvae_ctx* st = &up->store;
  int nb = 0;
  for (const auto& kv : st->shapes) {
    int bi = -1;
    if (sscanf(kv.first.c_str(), "body.%d.", &bi) == 1) nb = std::max(nb, bi + 1);
  }
  HDRVAE_REQUIRE(nb >= 1, "upscaler state dict holds no RRDB blocks (body.N.rdbK.convJ / model.1.sub.N.RDBK.convJ.0) and is "
                 "no Real-ESRGAN Compact model (body.0.weight without conv_first) or SPAN model (conv_1.sk.weight), nor a "
                 "SwinIR model (%s)", kSwinKey);
  up->nb = nb;
  // the layout: u upsampling convs (counted on load) and the pixel-unshuffle factor f from conv_first's 3 f^2 input channels
  HDRVAE_REQUIRE(n_up >= 0, "RRDBNet: %s has shape %s; an old-arch RRDBNet's last top-level conv sits at index 3u + 4 "
                 "(4, 7 or 10 for u = 0, 1 or 2 upsampling convs)", top_key.c_str(), top_shape.c_str());
  HDRVAE_REQUIRE(n_up <= 2, "RRDBNet: %s has shape %s: a third upsampling conv (an 8x RRDBNet) is not supported; RRDBNet "
                 "runs with 0, 1 or 2 upsampling convs", top_key.empty() ? "conv_up3.weight" : "model.9.weight",
                 up_shape_str(st, "conv_up3.weight").c_str());
  auto it = st->shapes.find("conv_first.weight");
  HDRVAE_REQUIRE(it != st->shapes.end(), "upscaler state dict lacks conv_first.{weight,bias}");
  const std::vector<int64_t>& w0 = it->second;
  const int64_t cin = w0.size() == 4 ? w0[1] : 0;
  HDRVAE_REQUIRE(cin == 3 || cin == 12 || cin == 48, "RRDBNet: conv_first.weight has shape %s; want [64,3 f^2,3,3] with "
                 "pixel-unshuffle factor f = 1, 2 or 4 (3, 12 or 48 input channels)", up_shape_str(w0).c_str());
  const int f = cin == 3 ? 1 : cin == 12 ? 2 : 4;
  HDRVAE_REQUIRE((1 << n_up) >= f, "RRDBNet: conv_first.weight has shape %s (pixel-unshuffle factor %d) and the model has "
                 "%d upsampling conv(s): its scale 2^%d / %d would be below 1", up_shape_str(w0).c_str(), f, n_up, n_up, f);
  up->n_up = n_up;
  up->shuffle = f;
  up->scale = (1 << n_up) / f;
  up->convs.resize(1 + 15 * (size_t)nb + n_up + 3);
  PackedConv* pc = up->convs.data();                  // filled in launch order
  HDRVAE_TRY(up_pack(st, "RRDBNet", "conv_first", 64, 3 * f * f, 3, false, 1.f, pc++, s));
  for (int i = 0; i < nb; ++i)
    for (int r = 0; r < 3; ++r) {
      const std::string base = "body." + std::to_string(i) + ".rdb" + std::to_string(r + 1) + ".conv";
      for (int j = 0; j < 4; ++j)
        HDRVAE_TRY(up_pack(st, "RRDBNet", base + std::to_string(j + 1), 32, 64 + 32 * j, 3, false, 1.f, pc++, s));
      // residual scaling folded into conv5's weights and bias: 0.2, and 0.2 * 0.2 for the block that ends an RRDB
      const float rs = r == 2 ? 0.2f * 0.2f : 0.2f;
      HDRVAE_TRY(up_pack(st, "RRDBNet", base + "5", 64, 192, 3, false, rs, pc, s));
      up_scale_f32_kernel<<<1, 64, 0, s>>>(pc->bias, 64, rs);
      HDRVAE_CUDA_OK(cudaGetLastError());
      ++pc;
    }
  HDRVAE_TRY(up_pack(st, "RRDBNet", "conv_body", 64, 64, 3, false, 1.f, pc++, s));
  for (int k = 1; k <= n_up; ++k)
    HDRVAE_TRY(up_pack(st, "RRDBNet", "conv_up" + std::to_string(k), 64, 64, 3, true, 1.f, pc++, s));
  HDRVAE_TRY(up_pack(st, "RRDBNet", "conv_hr", 64, 64, 3, false, 1.f, pc++, s));
  return up_pack(st, "RRDBNet", "conv_last", 3, 64, 3, false, 1.f, pc, s);
}

// After packing: waits for the copies, frees the staging buffers and the fp32 copies of the state dict.
static int up_finish_load(hdrvae_upscaler* up, std::vector<void*>& staging, cudaStream_t s) {
  hdrvae_ctx* st = &up->store;
  HDRVAE_CUDA_OK(cudaStreamSynchronize(s));
  for (void* p : staging) cudaFree(p);
  for (auto& kv : st->raw) cudaFree(kv.second);        // fp32 copies are no longer needed
  {
    std::vector<void*> keep;
    for (void* p : st->owned) {
      bool raw = false;
      for (auto& kv : st->raw) if (kv.second == p) { raw = true; break; }
      if (!raw) keep.push_back(p);
    }
    st->owned.swap(keep);
    st->raw.clear();
  }
  up->loaded = true;
  return 0;
}

int hdrvae_upscaler_load_weights(hdrvae_upscaler* up, const hdrvae_weight_desc* descs, int n) {
  HDRVAE_REQUIRE(up != nullptr && descs != nullptr && n > 0, "hdrvae_upscaler_load_weights: null argument");
  HDRVAE_REQUIRE(!up->loaded, "hdrvae_upscaler_load_weights: model already loaded (create a new one)");
  hdrvae_ctx* st = &up->store;
  HDRVAE_CUDA_OK(cudaSetDevice(st->device));
  cudaStream_t s = nullptr;
  std::vector<void*> staging;
  std::string top_key, top_shape;
  const int n_up = up_count_upconvs(descs, n, &top_key, &top_shape);
  for (int i = 0; i < n; ++i) {
    const hdrvae_weight_desc& d = descs[i];
    HDRVAE_REQUIRE(d.name && d.data && d.ndim >= 1 && d.ndim <= 4, "hdrvae_upscaler_load_weights: bad descriptor %d", i);
    const std::string name = up_canonical(d.name, n_up);
    if (name.empty()) continue;
    long long cnt = 1;
    std::vector<int64_t> shp;
    for (int k = 0; k < d.ndim; ++k) { cnt *= d.shape[k]; shp.push_back(d.shape[k]); }
    const size_t esz = d.dtype == HDRVAE_F32 ? 4 : 2;
    void* stage = nullptr;
    HDRVAE_CUDA_OK(cudaMalloc(&stage, cnt * esz));
    staging.push_back(stage);
    HDRVAE_CUDA_OK(cudaMemcpyAsync(stage, d.data, cnt * esz, cudaMemcpyDefault, s));
    float* f = nullptr;
    HDRVAE_TRY(dev_alloc(st, cnt * sizeof(float), (void**)&f));
    HDRVAE_TRY(launch_to_f32(stage, d.dtype, f, cnt, s));
    st->raw[name] = f;
    st->shapes[name] = shp;
  }
  // Compact: body.0.weight and no conv_first (in either layout); SPAN: conv_1.sk.weight; SwinIR (and HAT, which its loader
  // refuses): the first block's relative-position bias table; anything else is an RRDBNet
  bool has_conv_first = false;
  for (const auto& kv : st->shapes) has_conv_first = has_conv_first || kv.first.compare(0, 11, "conv_first.") == 0;
  UpArch arch = UP_RRDB;
  if (st->shapes.count("body.0.weight") && !has_conv_first) arch = UP_COMPACT;
  else if (st->shapes.count("conv_1.sk.weight")) arch = UP_SPAN;
  else if (st->shapes.count(kSwinKey)) arch = UP_SWINIR;
  switch (arch) {
    case UP_RRDB: HDRVAE_TRY(up_pack_rrdb(up, n_up, top_key, top_shape, s)); break;
    case UP_COMPACT: HDRVAE_TRY(up_pack_compact(up, s)); break;
    case UP_SPAN: HDRVAE_TRY(up_pack_span(up, s)); break;
    case UP_SWINIR: HDRVAE_TRY(up_pack_swinir(up, s)); break;
  }
  up->arch = arch;
  return up_finish_load(up, staging, s);
}

int hdrvae_upscaler_blocks(hdrvae_upscaler* up) { return up ? up->nb : -1; }

int hdrvae_upscaler_scale(hdrvae_upscaler* up) {
  HDRVAE_REQUIRE(up != nullptr && up->loaded, "hdrvae_upscaler_scale: weights not loaded");
  return up->scale;
}

int hdrvae_upscaler_forward_bytes(hdrvae_upscaler* up, int n, int h, int w, size_t* bytes) {
  HDRVAE_REQUIRE(up && bytes && n >= 1 && h >= 1 && w >= 1, "hdrvae_upscaler_forward_bytes: bad argument");
  HDRVAE_TRY(up_check_sides(up, h, w));
  const UpPlan pl = up_make_plan(up, n, h, w);
  *bytes = pl.total + (size_t)n * up->scale * up->scale * h * w * 16 + (size_t)n * sizeof(int4) + 4096;
  return 0;
}

int hdrvae_upscaler_forward(hdrvae_upscaler* up, const float* x_bhwc, int n, int h, int w, int reversal, float* y_bhwc,
                            void* workspace, size_t workspace_bytes, void* stream) {
  HDRVAE_REQUIRE(up && up->loaded && x_bhwc && y_bhwc && workspace, "hdrvae_upscaler_forward: null argument / no weights");
  HDRVAE_REQUIRE(reversal >= 0 && reversal <= 2, "hdrvae_upscaler_forward: reversal must be 0 (none), 1 (atanh) or 2 (logit)");
  size_t need = 0;
  HDRVAE_TRY(hdrvae_upscaler_forward_bytes(up, n, h, w, &need));
  HDRVAE_REQUIRE(workspace_bytes >= need, "hdrvae_upscaler_forward: workspace too small (%zu < %zu)", workspace_bytes, need);
  HDRVAE_CUDA_OK(cudaSetDevice(up->store.device));
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
  const UpPlan pl = up_make_plan(up, n, h, w);
  const long long npx = (long long)n * up->scale * up->scale * h * w;
  float* out4 = reinterpret_cast<float*>(ws + pl.total);
  int4* origins = reinterpret_cast<int4*>(ws + pl.total + (size_t)npx * 16);
  std::vector<int4> host(n);
  for (int i = 0; i < n; ++i) host[i] = make_int4(i, 0, 0, 0);
  HDRVAE_CUDA_OK(cudaMemcpyAsync(origins, host.data(), n * sizeof(int4), cudaMemcpyHostToDevice, s));
  HDRVAE_TRY(up_run_model(up, x_bhwc, h, w, origins, n, h, w, ws, pl, out4, s));
  up_finish_tiles_kernel<<<up_grid(npx), 256, 0, s>>>(reinterpret_cast<const float4*>(out4), npx, reversal, y_bhwc);
  HDRVAE_LAUNCHED();
  HDRVAE_CUDA_OK(cudaGetLastError());
  return 0;
}

int hdrvae_upscale_workspace_bytes(hdrvae_upscaler* up, int B, int H, int W, size_t* bytes) {
  HDRVAE_REQUIRE(up && bytes && B >= 1 && H >= 1 && W >= 1, "hdrvae_upscale_workspace_bytes: bad argument");
  const UpTiling t = up_make_tiling(B, H, W, up->scale);
  for (const UpGroup& g : t.groups) HDRVAE_TRY(up_check_sides(up, g.h, g.w));
  *bytes = up_make_ws(up, t, B, H, W).total;
  return 0;
}

int hdrvae_upscale(hdrvae_upscaler* up, const float* image_bhwc, int B, int H, int W, int reversal, int small_blur,
                   int local_fix, int upscale_method, float* out_bhwc, void* workspace, size_t workspace_bytes,
                   void* stream) {
  HDRVAE_REQUIRE(up && up->loaded && image_bhwc && out_bhwc && workspace, "hdrvae_upscale: null argument / no weights");
  HDRVAE_REQUIRE(reversal == 1 || reversal == 2, "hdrvae_upscale: reversal must be 1 (atanh) or 2 (logit)");
  HDRVAE_REQUIRE(!local_fix || (upscale_method >= HDRVAE_UPSCALE_NEAREST_EXACT && upscale_method <= HDRVAE_UPSCALE_BISLERP),
                 "hdrvae_upscale: local_fix supports upscale_method nearest-exact, bilinear, area, bicubic and bislerp (got %d)", upscale_method);
  HDRVAE_CUDA_OK(cudaSetDevice(up->store.device));
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const int sc = up->scale;
  const UpTiling t = up_make_tiling(B, H, W, sc);
  for (const UpGroup& g : t.groups) HDRVAE_TRY(up_check_sides(up, g.h, g.w));
  const UpWs wsl = up_make_ws(up, t, B, H, W);
  HDRVAE_REQUIRE(workspace_bytes >= wsl.total, "hdrvae_upscale: workspace too small (%zu < %zu)", workspace_bytes, wsl.total);
  uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
  const int OH = H * sc, OW = W * sc;
  // tile descriptors (output coordinates) in the reference's accumulation order
  std::vector<UpTile> descs(t.tiles.size());
  for (size_t i = 0; i < t.tiles.size(); ++i) {
    const UpHostTile& u = t.tiles[i];
    descs[i].b = u.b; descs[i].oy = u.y0 * sc; descs[i].ox = u.x0 * sc;
    descs[i].oh = u.h * sc; descs[i].ow = u.w * sc; descs[i].off = u.off; descs[i].off2 = u.off2;
  }
  HDRVAE_CUDA_OK(cudaMemcpyAsync(ws + wsl.descs, descs.data(), descs.size() * sizeof(UpTile), cudaMemcpyHostToDevice, s));
  // small_blur's input filter (:176-178) is torchvision gaussian_blur(kernel 3, sigma 0.1): taps exp(-50) = 1.9e-22
  // around a centre tap that rounds to 1.0f, i.e. the identity on fp32 images; nothing to launch.
  int4* origins = reinterpret_cast<int4*>(ws + wsl.origins);
  std::vector<int4> host_or(2 * t.tiles.size());
  for (const UpChunk& c : t.chunks)
    for (int pass = 0; pass < 2; ++pass)
      for (int j = 0; j < c.n; ++j) {
        const UpHostTile& u = t.tiles[t.order[c.first + j]];
        host_or[c.origin0 + pass * c.n + j] = make_int4(u.b, u.y0, u.x0, pass);     // .w: clamp the input to [-1, 1]
      }
  HDRVAE_CUDA_OK(cudaMemcpyAsync(origins, host_or.data(), host_or.size() * sizeof(int4), cudaMemcpyHostToDevice, s));
  float* out_all = reinterpret_cast<float*>(ws + wsl.out);
  for (const UpChunk& c : t.chunks) {
    const UpPlan pl = up_make_plan(up, 2 * c.n, c.h, c.w);
    HDRVAE_TRY(up_run_model(up, image_bhwc, H, W, origins + c.origin0, 2 * c.n, c.h, c.w, ws + wsl.fwd, pl,
                            out_all + c.out_base * 4, s));
  }
  const long long opx = (long long)B * OH * OW;
  float* ycc = reinterpret_cast<float*>(ws + wsl.ycc);
  float* tmp = reinterpret_cast<float*>(ws + wsl.tmp);
  {
    ProfScope prof("upscaler blend + YCbCr", 0.0, (double)t.out_px * 16 + opx * 12, s);
    up_blend_ycc_kernel<<<up_grid(opx), 256, 0, s>>>(reinterpret_cast<const float4*>(ws + wsl.out),
                                                      reinterpret_cast<const UpTile*>(ws + wsl.descs), (int)t.tiles.size(),
                                                      t.single ? 1 : 0, B, OH, OW, kUpOverlap * sc, reversal, ycc);
    HDRVAE_LAUNCHED();
  }
  {
    ProfScope prof("upscaler median Y + recombine", 0.0, opx * 24.0, s);
    up_recombine_kernel<<<up_grid(opx), 256, 0, s>>>(ycc, B, OH, OW, small_blur ? tmp : out_bhwc);
    HDRVAE_LAUNCHED();
  }
  if (small_blur) {
    ProfScope prof("upscaler median RGB (small_blur)", 0.0, opx * 24.0, s);
    up_median_rgb_kernel<<<up_grid(opx * 3), 256, 0, s>>>(tmp, B, OH, OW, out_bhwc);
    HDRVAE_LAUNCHED();
  }
  if (local_fix) {
    ProfScope prof("upscaler local fix", 0.0, opx * 24.0 + (double)B * H * W * 12, s);
    up_local_fix_kernel<<<up_grid(opx), 256, 0, s>>>(image_bhwc, B, H, W, sc, upscale_method, out_bhwc);
    HDRVAE_LAUNCHED();
  }
  HDRVAE_CUDA_OK(cudaGetLastError());
  return 0;
}

}  // extern "C"
