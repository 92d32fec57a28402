// Kernels of the SwinIR upscaler (upscaler.cu up_forward_swinir) that are not convs: LayerNorm over the channels of each
// token, the (shifted) window attention, and the fp16 pixel shuffle of the "pixelshuffle" tail.  The linears (qkv, proj,
// fc1 with GELU, fc2) and the convs run on the tcgen05 conv kernel of gemm_tc.cu.
#include <math.h>

#include "engine.cuh"

namespace hdrvae {

// ------------------------------------------------------------------------------------------------ LayerNorm
// One warp per token, C <= 256: 8 values per lane in registers, mean and variance in fp32 with a second pass over the
// registers (torch's biased variance), eps 1e-5.  y fp32 [P][C], or fp16 [P][y_ld] with channels C .. y_ld - 1 zero.
constexpr int kLnMaxC = 256;
__global__ void __launch_bounds__(256) layernorm_kernel(const float* __restrict__ x, long long P, int C,
                                                        const float* __restrict__ gamma, const float* __restrict__ beta,
                                                        void* __restrict__ y, int y_f16, int y_ld) {
  const int lane = threadIdx.x & 31;
  const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
  for (long long t = blockIdx.x * (long long)(blockDim.x >> 5) + (threadIdx.x >> 5); t < P; t += warps) {
    const float* xr = x + t * C;
    float v[kLnMaxC / 32];
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < kLnMaxC / 32; ++k) {
      const int c = lane + 32 * k;
      v[k] = c < C ? xr[c] : 0.f;
      s += v[k];
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const float mean = s / (float)C;
    float q = 0.f;
#pragma unroll
    for (int k = 0; k < kLnMaxC / 32; ++k) {
      const float d = lane + 32 * k < C ? v[k] - mean : 0.f;
      q = fmaf(d, d, q);
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
    const float rstd = rsqrtf(q / (float)C + 1e-5f);
#pragma unroll
    for (int k = 0; k < kLnMaxC / 32; ++k) {
      const int c = lane + 32 * k;
      if (y_f16) {
        if (c < y_ld)
          reinterpret_cast<__half*>(y)[t * y_ld + c] =
              __float2half_rn(c < C ? fmaf((v[k] - mean) * rstd, __ldg(gamma + c), __ldg(beta + c)) : 0.f);
      } else if (c < C) {
        reinterpret_cast<float*>(y)[t * C + c] = fmaf((v[k] - mean) * rstd, __ldg(gamma + c), __ldg(beta + c));
      }
    }
  }
}

int launch_layernorm(const float* x, long long P, int C, const float* gamma, const float* beta, void* y, int y_dtype,
                     int y_ld, cudaStream_t s) {
  HDRVAE_REQUIRE(C >= 1 && C <= kLnMaxC, "layernorm: C (%d) must be in 1..%d", C, kLnMaxC);
  HDRVAE_REQUIRE(y_dtype == DT_F32 || (y_dtype == DT_F16 && y_ld >= C && y_ld <= kLnMaxC && y_ld % 8 == 0),
                 "layernorm: y must be fp32, or fp16 with a pixel stride >= C, <= %d and a multiple of 8", kLnMaxC);
  if (P <= 0) return 0;
  const int grid = (int)std::min<long long>((P + 7) / 8, 148 * 32);
  ProfScope prof("swinir layernorm", 0.0, (double)P * (C * 4 + (y_dtype == DT_F32 ? C * 4 : y_ld * 2)), s);
  layernorm_kernel<<<grid, 256, 0, s>>>(x, P, C, gamma, beta, y, y_dtype == DT_F16 ? 1 : 0, y_ld);
  HDRVAE_LAUNCHED();
  HDRVAE_CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------ window attention
// One CTA of 128 threads per (8 x 8 window, head).  K and V of the window's 64 tokens (head dim padded to 32) are gathered
// into shared memory as fp32; the roll by -shift and the window partition are the gather's index arithmetic, and the
// output goes back to the same pixels (the roll by +shift and the window reverse).  Thread 2i + e owns query i and the 32
// keys 2j + e: its q row and its 32 scores stay in registers, S = q k^T + the relative-position bias (and the -100 region
// mask) in fp32, softmax over the pair of threads (one shuffle for the max, one for the sum), then P V in fp32 and the two
// partial outputs summed by shuffles.  FFMA on the CUDA cores: the library's SASS carries no mma.sync (HMMA) code.
constexpr int kWin = 8, kTok = 64, kHd = 32;
constexpr int kKvPitch = kHd + 4;       // floats per K / V row: the pair of rows 2j, 2j + 1 a warp reads sit 4 banks apart

__global__ void __launch_bounds__(128) window_attention_kernel(const __half* __restrict__ qkv, int heads, int H, int W,
                                                               const float* __restrict__ table, int shift,
                                                               __half* __restrict__ o) {
  __shared__ __align__(16) float sk[kTok][kKvPitch];
  __shared__ __align__(16) float sv[kTok][kKvPitch];
  __shared__ float sbias[(2 * kWin - 1) * (2 * kWin - 1)];
  __shared__ long long spix[kTok];
  __shared__ int sreg[kTok];
  const int qkv_ld = 3 * heads * kHd, o_ld = heads * kHd;
  const int h = blockIdx.x % heads;
  const int win = blockIdx.x / heads;
  const int wpr = W / kWin, wpc = H / kWin;
  const int wx = win % wpr, wy = (win / wpr) % wpc, img = win / (wpr * wpc);
  const int tid = threadIdx.x;
  if (tid < kTok) {
    const int r = tid >> 3, c = tid & 7;
    const int ys = wy * kWin + r, xs = wx * kWin + c;        // position in the rolled image
    const int yy = (ys + shift) % H, xx = (xs + shift) % W;  // the pixel it came from
    spix[tid] = ((long long)img * H + yy) * W + xx;
    // calculate_mask: slices (0, -ws), (-ws, -shift), (-shift, None) of each axis of the rolled image
    const int rh = shift == 0 ? 0 : ys < H - kWin ? 0 : ys < H - shift ? 1 : 2;
    const int rw = shift == 0 ? 0 : xs < W - kWin ? 0 : xs < W - shift ? 1 : 2;
    sreg[tid] = rh * 3 + rw;
  }
  for (int i = tid; i < (2 * kWin - 1) * (2 * kWin - 1); i += blockDim.x) sbias[i] = __ldg(table + (long long)i * heads + h);
  __syncthreads();
  for (int e = tid; e < kTok * 4; e += blockDim.x) {
    const int tok = e >> 2, part = e & 3;
    const __half* base = qkv + spix[tok] * qkv_ld + (heads + h) * kHd + part * 8;
    const uint4 kr = __ldg(reinterpret_cast<const uint4*>(base));
    const uint4 vr = __ldg(reinterpret_cast<const uint4*>(base + heads * kHd));
    const __half2* k2 = reinterpret_cast<const __half2*>(&kr);
    const __half2* v2 = reinterpret_cast<const __half2*>(&vr);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      *reinterpret_cast<float2*>(&sk[tok][part * 8 + 2 * j]) = __half22float2(k2[j]);
      *reinterpret_cast<float2*>(&sv[tok][part * 8 + 2 * j]) = __half22float2(v2[j]);
    }
  }
  const int qi = tid >> 1, half = tid & 1;
  float q[kHd];
  {
    const __half* base = qkv + spix[qi] * qkv_ld + h * kHd;
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      const uint4 r = __ldg(reinterpret_cast<const uint4*>(base + p * 8));
      const __half2* r2 = reinterpret_cast<const __half2*>(&r);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 f = __half22float2(r2[j]);
        q[p * 8 + 2 * j] = f.x;
        q[p * 8 + 2 * j + 1] = f.y;
      }
    }
  }
  __syncthreads();
  // bias: index (ri - rj + 7) * 15 + (ci - cj + 7) of the relative-position table
  const int bq = ((qi >> 3) + 7) * 15 + (qi & 7) + 7, rq = sreg[qi];
  float sc[kTok / 2];
  float m = -INFINITY;
#pragma unroll
  for (int j = 0; j < kTok / 2; ++j) {
    const int key = 2 * j + half;
    float acc = 0.f;
#pragma unroll
    for (int d = 0; d < kHd; d += 4) {
      const float4 k = *reinterpret_cast<const float4*>(&sk[key][d]);
      acc = fmaf(q[d], k.x, acc); acc = fmaf(q[d + 1], k.y, acc); acc = fmaf(q[d + 2], k.z, acc); acc = fmaf(q[d + 3], k.w, acc);
    }
    acc += sbias[bq - ((key >> 3) * 15 + (key & 7))];
    if (shift && sreg[key] != rq) acc += -100.f;
    sc[j] = acc;
    m = fmaxf(m, acc);
  }
  m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 1));
  float l = 0.f, oa[kHd];
#pragma unroll
  for (int d = 0; d < kHd; ++d) oa[d] = 0.f;
#pragma unroll
  for (int j = 0; j < kTok / 2; ++j) {
    const float p = __expf(sc[j] - m);
    l += p;
    const int key = 2 * j + half;
#pragma unroll
    for (int d = 0; d < kHd; d += 4) {
      const float4 v = *reinterpret_cast<const float4*>(&sv[key][d]);
      oa[d] = fmaf(p, v.x, oa[d]); oa[d + 1] = fmaf(p, v.y, oa[d + 1]);
      oa[d + 2] = fmaf(p, v.z, oa[d + 2]); oa[d + 3] = fmaf(p, v.w, oa[d + 3]);
    }
  }
  l += __shfl_xor_sync(0xffffffffu, l, 1);
#pragma unroll
  for (int d = 0; d < kHd; ++d) oa[d] += __shfl_xor_sync(0xffffffffu, oa[d], 1);
  const float inv = 1.f / l;
  // thread e of the pair stores channels 16 e .. 16 e + 15
  __align__(16) __half out[kHd / 2];
#pragma unroll
  for (int d = 0; d < kHd / 2; ++d) out[d] = __float2half_rn((half ? oa[kHd / 2 + d] : oa[d]) * inv);
  uint4* dst = reinterpret_cast<uint4*>(o + spix[qi] * o_ld + h * kHd + half * (kHd / 2));
  dst[0] = reinterpret_cast<const uint4*>(out)[0];
  dst[1] = reinterpret_cast<const uint4*>(out)[1];
}

int launch_window_attention(const void* qkv, int B, int H, int W, int heads, const float* table, int shift, void* o,
                            cudaStream_t s) {
  HDRVAE_REQUIRE(B >= 1 && H >= kWin && W >= kWin && H % kWin == 0 && W % kWin == 0,
                 "window attention: H and W (%d x %d) must be multiples of %d", H, W, kWin);
  HDRVAE_REQUIRE(heads >= 1 && heads <= 256, "window attention: heads (%d) must be in 1..256", heads);
  HDRVAE_REQUIRE(shift == 0 || shift == kWin / 2, "window attention: shift (%d) must be 0 or %d", shift, kWin / 2);
  const long long units = (long long)B * (H / kWin) * (W / kWin) * heads;
  HDRVAE_REQUIRE(units < (1LL << 31), "window attention: too many windows");
  const double tok = (double)B * H * W;
  ProfScope prof("swinir window attention", tok * heads * 4.0 * kTok * kHd, tok * heads * kHd * 2.0 * 4.0, s);
  window_attention_kernel<<<(unsigned)units, 128, 0, s>>>(reinterpret_cast<const __half*>(qkv), heads, H, W, table, shift,
                                                          reinterpret_cast<__half*>(o));
  HDRVAE_LAUNCHED();
  HDRVAE_CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------ pixel shuffle (fp16)
// nn.PixelShuffle(2) on NHWC fp16: in [n][h][w][4 c] -> out [n][2h][2w][c]; channel 4 k + 2 i + j of input pixel (y, x)
// is channel k of output pixel (2 y + i, 2 x + j).  One thread per (output pixel, 8 channels).
__global__ void pixel_shuffle2_f16_kernel(const __half* __restrict__ in, int n, int h, int w, int c, __half* __restrict__ out) {
  const int OW = 2 * w, OH = 2 * h, c8 = c / 8;
  const long long total = (long long)n * OH * OW * c8;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int k8 = (int)(i % c8);
    const long long px = i / c8;
    const int X = (int)(px % OW);
    const int Y = (int)((px / OW) % OH);
    const int t = (int)(px / ((long long)OW * OH));
    const int y = Y >> 1, x = X >> 1, sub = (Y & 1) * 2 + (X & 1);
    const __half* src = in + (((long long)t * h + y) * w + x) * 4 * c + k8 * 32 + sub;
    __align__(16) __half v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = src[4 * j];
    reinterpret_cast<uint4*>(out)[i] = *reinterpret_cast<const uint4*>(v);
  }
}

int launch_pixel_shuffle2_f16(const void* in, int n, int h, int w, int c, void* out, cudaStream_t s) {
  HDRVAE_REQUIRE(c % 8 == 0, "pixel shuffle: channels (%d) must be a multiple of 8", c);
  const long long total = (long long)n * 4 * h * w * (c / 8);
  ProfScope prof("swinir pixel shuffle", 0.0, (double)n * h * w * c * 4 * 2 * 2, s);
  pixel_shuffle2_f16_kernel<<<(int)std::min<long long>((total + 255) / 256, 148 * 32), 256, 0, s>>>(
      reinterpret_cast<const __half*>(in), n, h, w, c, reinterpret_cast<__half*>(out));
  HDRVAE_LAUNCHED();
  HDRVAE_CUDA_OK(cudaGetLastError());
  return 0;
}

}  // namespace hdrvae

// ------------------------------------------------------------------------------------------------ C ABI
extern "C" {

int hdrvae_layernorm(hdrvae_ctx* ctx, const float* x, long long n_tokens, int C, const float* gamma, const float* beta,
                     void* y, int y_dtype, int y_channels, void* stream) {
  HDRVAE_REQUIRE(ctx && x && gamma && beta && y && n_tokens >= 0, "hdrvae_layernorm: bad argument");
  HDRVAE_REQUIRE(y_dtype == HDRVAE_F32 || y_dtype == HDRVAE_F16, "hdrvae_layernorm: y must be float32 or fp16");
  HDRVAE_CUDA_OK(cudaSetDevice(ctx->device));
  return launch_layernorm(x, n_tokens, C, gamma, beta, y, y_dtype == HDRVAE_F32 ? DT_F32 : DT_F16,
                          y_dtype == HDRVAE_F32 ? C : y_channels, reinterpret_cast<cudaStream_t>(stream));
}

int hdrvae_window_attention(hdrvae_ctx* ctx, const void* qkv, int B, int H, int W, int heads, const float* bias_table,
                            int shift, void* o, void* stream) {
  HDRVAE_REQUIRE(ctx && qkv && bias_table && o, "hdrvae_window_attention: null argument");
  HDRVAE_REQUIRE((reinterpret_cast<uintptr_t>(qkv) & 15) == 0 && (reinterpret_cast<uintptr_t>(o) & 15) == 0,
                 "hdrvae_window_attention: qkv and o must be 16-byte aligned");
  HDRVAE_CUDA_OK(cudaSetDevice(ctx->device));
  return launch_window_attention(qkv, B, H, W, heads, bias_table, shift, o, reinterpret_cast<cudaStream_t>(stream));
}

}  // extern "C"
