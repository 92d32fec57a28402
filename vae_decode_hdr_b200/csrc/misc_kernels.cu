// Small kernels around the GEMM core: weight repack, latent layout change, CUDA-core
// validation conv, attention row softmax, fp16 pack for the EXR exporter.
#include "common.cuh"

namespace hdrvae {

// ------------------------------------------------------------------ dtype -> fp32 copy
__global__ void to_f32_kernel(const void* __restrict__ src, int dtype, float* __restrict__ dst, long long n) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    float v;
    if (dtype == 0) v = reinterpret_cast<const float*>(src)[i];
    else if (dtype == 1) v = __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(src)[i]);
    else v = __half2float(reinterpret_cast<const __half*>(src)[i]);
    dst[i] = v;
  }
}
int launch_to_f32(const void* src, int dtype, float* dst, long long n, cudaStream_t s) {
  if (n == 0) return 0;
  to_f32_kernel<<<ceil_div(n, 256) > 1184 ? 1184 : ceil_div(n, 256), 256, 0, s>>>(src, dtype, dst, n);
  HDRVAE_LAUNCHED();
  HDRVAE_CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------ c = a + b (bias vectors)
__global__ void add_vectors_kernel(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ c, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) c[i] = a[i] + b[i];
}
int launch_add_vectors(const float* a, const float* b, float* c, int n, cudaStream_t s) {
  add_vectors_kernel<<<ceil_div(n, 256), 256, 0, s>>>(a, b, c, n);
  HDRVAE_LAUNCHED();
  HDRVAE_CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------ weight repack
// OIHW fp32 [Cout][Cin][ks][ks] -> K-major bf16 [Cout][ntaps][cin_pad]; output tap t is the SUM of
// the source kernel positions set in tap_mask[t] (bit ky*ks+kx).  Plain 3x3: mask = 1<<t.
// Upsample phase matrices: 2x2 taps, each the sum of the 3x3 positions that land on the same
// source pixel after nearest-2x upsampling.  `scale` multiplies every weight (attention 1/sqrt(d)).
struct PackArgs {
  int cout, cin, ks, ntaps, cin_pad, out_dtype;
  int tap_mask[9];
  float scale;
  int split3;   // fp16 only: every tap's K range is [hi | hi | lo] (3 * cin_pad) with hi = fp16(w), lo = fp16(w - hi)
};
__device__ __forceinline__ void store_as(void* out, long long i, int dtype, float v) {
  if (dtype == DT_F32) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));      // fp32 operands feed kind::tf32 MMAs: pre-round (RN)
    reinterpret_cast<float*>(out)[i] = __uint_as_float(r);
  } else if (dtype == DT_BF16) {
    reinterpret_cast<__nv_bfloat16*>(out)[i] = __float2bfloat16_rn(v);
  } else {
    reinterpret_cast<__half*>(out)[i] = __float2half_rn(v);
  }
}
__global__ void pack_weight_kernel(const float* __restrict__ w, void* __restrict__ out, PackArgs a) {
  const long long total = (long long)a.cout * a.ntaps * a.cin_pad;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int ci = (int)(i % a.cin_pad);
    const int t = (int)((i / a.cin_pad) % a.ntaps);
    const int co = (int)(i / ((long long)a.cin_pad * a.ntaps));
    float acc = 0.f;
    if (ci < a.cin) {
      const int kk = a.ks * a.ks;
      for (int s = 0; s < kk; ++s)
        if (a.tap_mask[t] & (1 << s)) acc += w[((long long)co * a.cin + ci) * kk + s];
    }
    const float v = acc * a.scale;
    if (a.split3) {
      // "precision high": w = hi + lo to ~2^-22; the activations come as [hi | lo | hi], so the K-concatenated product
      // is hi*hi + lo*hi + hi*lo (the lo*lo term, ~2^-22 relative, is dropped)
      __half* o = reinterpret_cast<__half*>(out) + ((long long)co * a.ntaps + t) * 3 * a.cin_pad + ci;
      const __half hi = __float2half_rn(v);
      o[0] = hi;
      o[a.cin_pad] = hi;
      o[2 * a.cin_pad] = __float2half_rn(v - __half2float(hi));
    } else {
      store_as(out, i, a.out_dtype, v);
    }
  }
}
int launch_pack_weight(const float* w, void* out, int out_dtype, int cout, int cin, int ks, int ntaps, int cin_pad,
                       const int* tap_mask, float scale, cudaStream_t s, int split3) {
  PackArgs a;
  a.split3 = split3;
  a.out_dtype = out_dtype;
  a.cout = cout; a.cin = cin; a.ks = ks; a.ntaps = ntaps; a.cin_pad = cin_pad; a.scale = scale;
  for (int t = 0; t < 9; ++t) a.tap_mask[t] = t < ntaps ? tap_mask[t] : 0;
  const long long total = (long long)cout * ntaps * cin_pad;
  int grid = ceil_div(total, 256);
  if (grid > 2368) grid = 2368;
  pack_weight_kernel<<<grid, 256, 0, s>>>(w, out, a);
  HDRVAE_LAUNCHED();
  HDRVAE_CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------ latent NCHW fp32 -> NHWC bf16 (channels zero-padded)
// Channel c of one latent pixel as conv_in sees it.  zp points at the pixel's channel 0, channels `cstride` apart.  With
// post_quant_conv (SD1.x / SDXL first-stage models): y[c] = b[c] + sum_c' W[c][c'] z[c'] in fp32, fmaf in the fixed order
// c' = 0 .. C_lat-1; without it the latent itself.
__device__ __forceinline__ float staged_latent(const float* __restrict__ zp, long long cstride, int c, int C_lat,
                                               const float* __restrict__ pq_w, const float* __restrict__ pq_b) {
  if (pq_w == nullptr) return zp[c * cstride];
  float v = pq_b[c];
  for (int k = 0; k < C_lat; ++k) v = fmaf(pq_w[c * C_lat + k], zp[k * cstride], v);
  return v;
}

__global__ void latent_to_nhwc_kernel(const float* __restrict__ z, void* __restrict__ out, int out_dtype, int B, int C,
                                      int C_lat, const float* __restrict__ pq_w, const float* __restrict__ pq_b, int HW,
                                      int cpad) {
  const long long total = (long long)B * HW * cpad;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % cpad);
    const long long p = i / cpad;
    const int hw = (int)(p % HW);
    const int b = (int)(p / HW);
    const float v = c < C ? staged_latent(z + (long long)b * C_lat * HW + hw, HW, c, C_lat, pq_w, pq_b) : 0.f;
    if (out_dtype == DT_F32) reinterpret_cast<float*>(out)[i] = v;
    else if (out_dtype == DT_BF16) reinterpret_cast<__nv_bfloat16*>(out)[i] = __float2bfloat16_rn(v);
    else reinterpret_cast<__half*>(out)[i] = __float2half_rn(v);
  }
}
int launch_latent_to_nhwc(const float* z, void* out, int out_dtype, int B, int C, int C_lat, const float* pq_w,
                          const float* pq_b, int HW, int cpad, cudaStream_t s) {
  const long long total = (long long)B * HW * cpad;
  int grid = ceil_div(total, 256);
  if (grid > 2368) grid = 2368;
  latent_to_nhwc_kernel<<<grid, 256, 0, s>>>(z, out, out_dtype, B, C, C_lat, pq_w, pq_b, HW, cpad);
  HDRVAE_LAUNCHED();
  HDRVAE_CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------ latent row slab (row tiling)
// full latent NCHW fp32 [C_lat][h][w] -> NHWC 16-bit slab [rows][w][cpad] holding latent rows y0 .. y0+rows-1 (after
// post_quant_conv, if any); rows outside the image and the padding channels are zero — conv_in's zero padding applies
// to post_quant_conv's output, so its bias must not reach those rows.
__global__ void latent_rows_to_nhwc_kernel(const float* __restrict__ z, void* __restrict__ out, int out_dtype, int C,
                                           int C_lat, const float* __restrict__ pq_w, const float* __restrict__ pq_b,
                                           int h, int w, int y0, int rows, int cpad) {
  const long long total = (long long)rows * w * cpad;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % cpad);
    const long long p = i / cpad;
    const int x = (int)(p % w);
    const int y = y0 + (int)(p / w);
    const float v = (c < C && y >= 0 && y < h) ? staged_latent(z + (long long)y * w + x, (long long)h * w, c, C_lat, pq_w, pq_b)
                                               : 0.f;
    if (out_dtype == DT_BF16) reinterpret_cast<__nv_bfloat16*>(out)[i] = __float2bfloat16_rn(v);
    else reinterpret_cast<__half*>(out)[i] = __float2half_rn(v);
  }
}
int launch_latent_rows_to_nhwc(const float* z, void* out, int out_dtype, int C, int C_lat, const float* pq_w,
                               const float* pq_b, int h, int w, int y0, int rows, int cpad, cudaStream_t s) {
  const long long total = (long long)rows * w * cpad;
  int grid = ceil_div(total, 256);
  if (grid > 2368) grid = 2368;
  latent_rows_to_nhwc_kernel<<<grid, 256, 0, s>>>(z, out, out_dtype, C, C_lat, pq_w, pq_b, h, w, y0, rows, cpad);
  HDRVAE_LAUNCHED();
  HDRVAE_CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------ CUDA-core validation conv (same GemmParams)
// One thread per output element; used only to validate the tcgen05 kernel on the GPU
// (HDRVAE_CONV_DIRECT), never on the product path.
__device__ __forceinline__ float load_as(const void* base, long long i, int dtype) {
  if (dtype == DT_F32) return reinterpret_cast<const float*>(base)[i];
  if (dtype == DT_BF16) return __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(base)[i]);
  return __half2float(reinterpret_cast<const __half*>(base)[i]);
}
__device__ __forceinline__ float trunc_tf32(float v) { return __uint_as_float(__float_as_uint(v) & 0xffffe000u); }

__global__ void gemm_direct_kernel(const GemmParams p) {
  const long long total = (long long)p.n_img * p.H * p.W * p.n_cols;
  const bool tf32 = p.ab_dtype == DT_F32;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int col = (int)(i % p.n_cols);
    if (p.n_store > 0 && col >= p.n_store) continue;   // a column that is not stored reads no residual / slope either
    long long r = i / p.n_cols;
    const int x = (int)(r % p.W); r /= p.W;
    const int y = (int)(r % p.H);
    const int img = (int)(r / p.H);
    float acc = 0.f;
    if (!(p.b_rows > 0 && col >= p.b_rows)) {
      for (int t = 0; t < p.ntaps; ++t) {
        const int ys = y + p.tap_dy[t] + p.y_pad, xs = x + p.tap_dx[t];
        if (ys < 0 || ys >= p.H + 2 * p.y_pad || xs < 0 || xs >= p.W) continue;
        const long long ao = img * p.a_img_stride + ys * p.a_row_stride + xs * p.a_px_stride;
        const long long bo = col * p.b_row_stride + (long long)t * p.k_per_tap;
        const int kv = p.a_k_valid > 0 ? p.a_k_valid : p.k_per_tap;
        for (int c = 0; c < kv; ++c) {
          float av = load_as(p.a, ao + c, p.ab_dtype), bv = load_as(p.b, bo + c, p.ab_dtype);
          if (tf32) { av = trunc_tf32(av); bv = trunc_tf32(bv); }     // the tensor core ignores the low 13 bits
          acc = fmaf(av, bv, acc);
        }
      }
    }
    float v = acc * p.alpha * (p.row_scale != nullptr ? p.row_scale[x] : 1.f);
    if (p.bias != nullptr) v += p.bias_per_row ? p.bias[x] : p.bias[col];
    const float gate = p.act == ACT_GATE ? 1.f / (1.f + expf(-v)) - 0.5f : 0.f;    // from t before the residual
    const long long off = (long long)img * p.out_img_stride + (long long)(y * p.sy + p.py) * p.out_row_stride +
                          (long long)(x * p.sx + p.px) * p.out_px_stride + col;
    if (p.residual != nullptr) v += (p.res_scale != 0.f ? p.res_scale : 1.f) * load_as(p.residual, off, p.res_dtype);
    if (p.residual2 != nullptr) v += p.residual2[off];
    if (p.lrelu != 0.f && v < 0.f) v *= p.lrelu;
    if (p.act_slope != nullptr && v < 0.f) v *= p.act_slope[col];
    if (p.act == ACT_SILU) v *= 1.f / (1.f + expf(-v));
    if (p.act == ACT_GATE) v *= gate;
    if (p.out2 != nullptr) {
      const long long off2 = p.out2_px_stride == 0 ? off
          : (long long)img * p.out2_img_stride + (long long)(y * p.sy + p.py) * p.out2_row_stride +
            (long long)(x * p.sx + p.px) * p.out2_px_stride + col;
      if (p.out2_dtype == DT_BF16) reinterpret_cast<__nv_bfloat16*>(p.out2)[off2] = __float2bfloat16_rn(v * p.out2_scale);
      else reinterpret_cast<__half*>(p.out2)[off2] = __float2half_rn(v * p.out2_scale);
    }
    if (p.out_dtype == DT_F32) {
      if (p.round_tf32) { uint32_t rr; asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(rr) : "f"(v)); v = __uint_as_float(rr); }
      reinterpret_cast<float*>(p.out)[off] = v;
    } else if (p.out_dtype == DT_BF16) reinterpret_cast<__nv_bfloat16*>(p.out)[off] = __float2bfloat16_rn(v);
    else reinterpret_cast<__half*>(p.out)[off] = __float2half_rn(v);
  }
}
int launch_gemm_direct(const GemmParams& p, cudaStream_t s) {
  const long long total = (long long)p.n_img * p.H * p.W * p.n_cols;
  int grid = ceil_div(total, 256);
  if (grid > 148 * 16) grid = 148 * 16;
  gemm_direct_kernel<<<grid, 256, 0, s>>>(p);
  HDRVAE_LAUNCHED();
  HDRVAE_CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------ fp32 tensor -> K-concatenated fp16 hi / lo operand
// x [n][C] fp32 (row stride x_ld) -> out [n][3 C] fp16 (row stride out_ld): activation order [hi | lo | hi] (order 0) or
// weight-side order [hi | hi | lo] (order 1) of scale * x, hi = fp16(v), lo = fp16(v - hi).  "precision high" feeds every
// GEMM-shaped op with such operands: sum_k a_k b_k over the 3 C columns = hi*hi + lo*hi + hi*lo.
__global__ void split3_kernel(const float* __restrict__ x, long long x_ld, __half* __restrict__ out, long long out_ld,
                              long long n, int C, float scale, int order) {
  const int c4 = C >> 2;
  const long long total = n * c4;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / c4;
    const int c = (int)(i - r * c4) * 4;
    const float4 v = *reinterpret_cast<const float4*>(x + r * x_ld + c);
    const float f[4] = {v.x * scale, v.y * scale, v.z * scale, v.w * scale};
    __half hi[4], lo[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) { hi[j] = __float2half_rn(f[j]); lo[j] = __float2half_rn(f[j] - __half2float(hi[j])); }
    __half* o = out + r * out_ld + c;
    const uint2 h2 = *reinterpret_cast<const uint2*>(hi), l2 = *reinterpret_cast<const uint2*>(lo);
    *reinterpret_cast<uint2*>(o) = h2;
    *reinterpret_cast<uint2*>(o + C) = order == 0 ? l2 : h2;
    *reinterpret_cast<uint2*>(o + 2 * C) = order == 0 ? h2 : l2;
  }
}
int launch_split3(const float* x, long long x_ld, void* out, long long out_ld, long long n, int C, float scale, int order,
                  cudaStream_t s) {
  HDRVAE_REQUIRE(C % 4 == 0 && x_ld % 4 == 0 && out_ld % 4 == 0, "split3: channel count / strides must be multiples of 4");
  if (n == 0) return 0;
  const long long total = n * (C >> 2);
  int grid = ceil_div(total, 256);
  if (grid > 148 * 16) grid = 148 * 16;
  split3_kernel<<<grid, 256, 0, s>>>(x, x_ld, reinterpret_cast<__half*>(out), out_ld, n, C, scale, order);
  HDRVAE_LAUNCHED();
  HDRVAE_CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------ fp32 weights -> fp16 hi / lo rows
// w [rows][k] fp32 -> w8 [8][k] fp32: rows 0..2 = w (packs to hi = fp16(w)), rows 4..6 = w - float(fp16(w)) (packs to
// lo), rows 3 and 7 zero; rows must be 3 (conv_out).  hi + lo carries ~21 mantissa bits of w.
__global__ void split_hi_lo_kernel(const float* __restrict__ w, float* __restrict__ w8, int k) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 8 * k) return;
  const int r = i / k, c = i - r * k;
  float v = 0.f;
  if ((r & 3) < 3) {
    const float x = w[(r & 3) * k + c];
    v = r < 4 ? x : x - __half2float(__float2half_rn(x));
  }
  w8[i] = v;
}
int launch_split_hi_lo(const float* w, float* w8, int k, cudaStream_t s) {
  split_hi_lo_kernel<<<ceil_div(8 * k, 256), 256, 0, s>>>(w, w8, k);
  HDRVAE_LAUNCHED();
  HDRVAE_CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------ attention row softmax, split form
// fp32 scores -> e = exp(s - rowmax) as 16-bit operand (max element is exactly 1: no fp16 range problem
// for long rows) + inv_sum[row] = 1 / sum(exp), applied later as the PV GEMM's per-row scale.
// One CTA per query row; two passes over the row (max, exp+sum+write); the row (<= 1 MB) stays in L2.
// Columns [n_valid, n_pad) are padding keys: excluded from the softmax and written as 0.
__device__ __forceinline__ uint32_t pack2(float a, float b, int dtype) {
  if (dtype == DT_BF16) { __nv_bfloat162 v = __floats2bfloat162_rn(a, b); return *reinterpret_cast<uint32_t*>(&v); }
  __half2 v = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}
__global__ void __launch_bounds__(256) softmax_rows_kernel(const float* __restrict__ s, void* __restrict__ p, int p_dtype,
                                                           float* __restrict__ inv_sum, int n_valid, int n_pad,
                                                           long long s_ld, long long p_ld) {
  const float* row = s + (long long)blockIdx.x * s_ld;
  uint16_t* out = reinterpret_cast<uint16_t*>(p) + (long long)blockIdx.x * p_ld;
  __shared__ float red[8];
  __shared__ float bcast;
  const int nv = n_valid >> 2;                      // full float4 groups
  const float4* row4 = reinterpret_cast<const float4*>(row);
  float m = -INFINITY;
  for (int i = threadIdx.x; i < nv; i += 256) {
    const float4 v = row4[i];
    m = fmaxf(fmaxf(m, fmaxf(v.x, v.y)), fmaxf(v.z, v.w));
  }
  for (int i = nv * 4 + threadIdx.x; i < n_valid; i += 256) m = fmaxf(m, row[i]);
  for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = red[0];
    for (int i = 1; i < 8; ++i) t = fmaxf(t, red[i]);
    bcast = t;
  }
  __syncthreads();
  m = bcast;
  float sum = 0.f;
  uint2* out4 = reinterpret_cast<uint2*>(out);
  for (int i = threadIdx.x; i < nv; i += 256) {
    const float4 v = row4[i];
    const float e0 = __expf(v.x - m), e1 = __expf(v.y - m), e2 = __expf(v.z - m), e3 = __expf(v.w - m);
    sum += (e0 + e1) + (e2 + e3);
    uint2 o2;
    o2.x = pack2(e0, e1, p_dtype);
    o2.y = pack2(e2, e3, p_dtype);
    out4[i] = o2;
    if (p_dtype == DT_F16X3) {
      // "precision high": the row is [hi | lo | hi] over the keys (3 * n_pad columns); pack2 wrote hi = fp16(e)
      const __half2 h01 = *reinterpret_cast<const __half2*>(&o2.x), h23 = *reinterpret_cast<const __half2*>(&o2.y);
      const float2 f01 = __half22float2(h01), f23 = __half22float2(h23);
      uint2 l2;
      l2.x = pack2(e0 - f01.x, e1 - f01.y, DT_F16);
      l2.y = pack2(e2 - f23.x, e3 - f23.y, DT_F16);
      reinterpret_cast<uint2*>(out + n_pad)[i] = l2;
      reinterpret_cast<uint2*>(out + 2 * (long long)n_pad)[i] = o2;
    }
  }
  for (int i = nv * 4 + threadIdx.x; i < n_pad; i += 256) {
    const float e = i < n_valid ? __expf(row[i] - m) : 0.f;
    sum += e;
    const uint16_t hi = (uint16_t)(pack2(e, 0.f, p_dtype) & 0xffffu);
    out[i] = hi;
    if (p_dtype == DT_F16X3) {
      const float fh = __half2float(*reinterpret_cast<const __half*>(&hi));
      out[n_pad + i] = (uint16_t)(pack2(e - fh, 0.f, DT_F16) & 0xffffu);
      out[2 * (long long)n_pad + i] = hi;
    }
  }
  for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = sum;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int i = 0; i < 8; ++i) t += red[i];
    inv_sum[blockIdx.x] = 1.f / t;
  }
}
int launch_softmax_rows(const float* s, void* p, int p_dtype, float* inv_sum, int n_rows, int n_valid, int n_pad,
                        long long s_ld, long long p_ld, cudaStream_t st) {
  HDRVAE_REQUIRE(s_ld % 4 == 0 && p_ld % 4 == 0 && n_pad >= n_valid, "softmax: bad leading dimensions");
  softmax_rows_kernel<<<n_rows, 256, 0, st>>>(s, p, p_dtype, inv_sum, n_valid, n_pad, s_ld, p_ld);
  HDRVAE_LAUNCHED();
  HDRVAE_CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------ [rows][cols] -> [cols][out_ld] transpose (test entry only)
__global__ void transpose_pad_kernel(const uint16_t* __restrict__ in, uint16_t* __restrict__ out, int rows,
                                     int cols, int out_ld) {
  __shared__ uint16_t tile[32][33];
  const int r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
  for (int j = threadIdx.y; j < 32; j += 8) {
    const int r = r0 + j, c = c0 + threadIdx.x;
    tile[j][threadIdx.x] = (r < rows && c < cols) ? in[(long long)r * cols + c] : (uint16_t)0;
  }
  __syncthreads();
  for (int j = threadIdx.y; j < 32; j += 8) {
    const int c = c0 + j, r = r0 + threadIdx.x;
    if (c < cols && r < rows) out[(long long)c * out_ld + r] = tile[threadIdx.x][j];
  }
}
int launch_transpose_pad(const void* in, void* out, int rows, int cols, int out_ld, cudaStream_t s) {
  transpose_pad_kernel<<<dim3(ceil_div(cols, 32), ceil_div(rows, 32)), dim3(32, 8), 0, s>>>(reinterpret_cast<const uint16_t*>(in), reinterpret_cast<uint16_t*>(out), rows, cols, out_ld);
  HDRVAE_LAUNCHED();
  HDRVAE_CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------ fp32 -> fp16 pack (LinearEXRExport, linear_exr_export.py:155,165)
// layout 0: same element order as the input (numpy astype(np.float16)); layout 1: EXR scanline order,
// per image row the B plane, then G, then R (OpenEXR stores channels alphabetically).
__global__ void pack_half_kernel(const float* __restrict__ img, __half* __restrict__ out, int B, int H, int W, int layout) {
  const long long total = (long long)B * H * W * 3;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    if (layout == 0) {
      out[i] = __float2half_rn(img[i]);
    } else {
      const int x = (int)(i % W);
      long long r = i / W;
      const int plane = (int)(r % 3); r /= 3;         // 0 = B, 1 = G, 2 = R
      const long long row = r;                        // b*H + y
      out[i] = __float2half_rn(img[(row * W + x) * 3 + (2 - plane)]);
    }
  }
}
int launch_pack_half(const float* img, uint16_t* out, int B, int H, int W, int layout, cudaStream_t s) {
  const long long total = (long long)B * H * W * 3;
  if (total == 0) return 0;
  int grid = ceil_div(total, 256);
  if (grid > 148 * 16) grid = 148 * 16;
  pack_half_kernel<<<grid, 256, 0, s>>>(img, reinterpret_cast<__half*>(out), B, H, W, layout);
  HDRVAE_LAUNCHED();
  HDRVAE_CUDA_OK(cudaGetLastError());
  return 0;
}

}  // namespace hdrvae
