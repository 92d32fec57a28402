// GroupNorm(32 groups, eps 1e-6, affine) + SiLU on NHWC activations — HBM-streaming kernels.
// Replaces norm1/norm2/norm_out + swish of ComfyUI's Decoder (driven through vae.decode,
// reference hdr_vae_decode.py:859,:1022).
//
//   statistics  : per (image, chunk) partial (sum, sum of squares) of every group in fp32.  In the decoder
//                 they are emitted by the epilogue of the conv that produced the tensor (gemm_tc.cu), so the
//                 tensor is not re-read; gn_stats_kernel is the standalone producer (test entry).  Partials are
//                 written, never atomically added: the reduction order is fixed -> deterministic, and under
//                 row tiling independent of the GPU count once the partials are all-reduced;
//   gn_finalize : fixed-order double reduction of the partials -> per (image, channel) scale/shift;
//   gn_apply    : y = silu(x * a[c] + b[c]); x fp32 (residual / conv stream) or 16-bit, y fp16/bf16 (the next
//                 conv's tensor-core operand), 16-byte accesses.
// Algorithmic traffic in the decoder: 4 B read + 2 B written per element.
#include <type_traits>

#include "common.cuh"

namespace hdrvae {

constexpr int kGroups = 32;
constexpr int kGnThreads = 256;

// 8 consecutive channels of one pixel as floats
template <typename T> struct Ld8;
template <> struct Ld8<float> {
  static __device__ __forceinline__ void ld(const float* p, float (&v)[8]) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(p)), b = __ldg(reinterpret_cast<const float4*>(p) + 1);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  }
};
template <> struct Ld8<__nv_bfloat16> {
  static __device__ __forceinline__ void ld(const __nv_bfloat16* p, float (&v)[8]) {
    const uint4 r = __ldg(reinterpret_cast<const uint4*>(p));
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&r);
#pragma unroll
    for (int e = 0; e < 4; ++e) { const float2 f = __bfloat1622float2(h[e]); v[2 * e] = f.x; v[2 * e + 1] = f.y; }
  }
};
template <> struct Ld8<__half> {
  static __device__ __forceinline__ void ld(const __half* p, float (&v)[8]) {
    const uint4 r = __ldg(reinterpret_cast<const uint4*>(p));
    const __half2* h = reinterpret_cast<const __half2*>(&r);
#pragma unroll
    for (int e = 0; e < 4; ++e) { const float2 f = __half22float2(h[e]); v[2 * e] = f.x; v[2 * e + 1] = f.y; }
  }
};
template <typename T> struct St8;
template <> struct St8<__nv_bfloat16> {
  static __device__ __forceinline__ void st(__nv_bfloat16* p, const float (&v)[8]) {
    uint4 o; uint32_t* w = reinterpret_cast<uint32_t*>(&o);
#pragma unroll
    for (int e = 0; e < 4; ++e) { __nv_bfloat162 t = __floats2bfloat162_rn(v[2 * e], v[2 * e + 1]); w[e] = *reinterpret_cast<uint32_t*>(&t); }
    *reinterpret_cast<uint4*>(p) = o;
  }
};
template <> struct St8<__half> {
  static __device__ __forceinline__ void st(__half* p, const float (&v)[8]) {
    uint4 o; uint32_t* w = reinterpret_cast<uint32_t*>(&o);
#pragma unroll
    for (int e = 0; e < 4; ++e) { __half2 t = __floats2half2_rn(v[2 * e], v[2 * e + 1]); w[e] = *reinterpret_cast<uint32_t*>(&t); }
    *reinterpret_cast<uint4*>(p) = o;
  }
};

template <> struct St8<float> {
  static __device__ __forceinline__ void st(float* p, const float (&v)[8]) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4*>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
  }
};
// "precision high" operand: [hi | lo | hi] fp16 per pixel (3 C channels), hi = fp16(v), lo = fp16(v - hi)
struct HalfSplit3 { __half h; };
// 8 channels of pixel p -> y; vpp = C / 8 vectors per pixel
template <typename TOut>
__device__ __forceinline__ void store8(TOut* y, long long p, int vpp, int vi, const float (&v)[8]) {
  St8<TOut>::st(y + (p * vpp + vi) * 8, v);
}
template <>
__device__ __forceinline__ void store8<HalfSplit3>(HalfSplit3* y, long long p, int vpp, int vi, const float (&v)[8]) {
  const int C = vpp * 8;
  __half* o = reinterpret_cast<__half*>(y) + p * 3 * C + vi * 8;
  float lo[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) lo[j] = v[j] - __half2float(__float2half_rn(v[j]));
  St8<__half>::st(o, v);
  St8<__half>::st(o + C, lo);
  St8<__half>::st(o + 2 * C, v);
}

template <typename TIn>
__global__ void __launch_bounds__(kGnThreads)
gn_stats_kernel(const TIn* __restrict__ x, float* __restrict__ partial, int HW, int C, int px_per_block) {
  const int img = blockIdx.y;
  const int chunk = blockIdx.x;
  const int vpp = C >> 3;                       // 8-channel vectors per pixel
  const int cpg = C / kGroups;
  const int vi = threadIdx.x % vpp;
  const int p_off = threadIdx.x / vpp;
  const int p_step = kGnThreads / vpp;
  const int p0 = chunk * px_per_block;
  const int p1 = min(HW, p0 + px_per_block);
  const TIn* base = x + (long long)img * HW * C;
  float s0 = 0.f, q0 = 0.f, s1 = 0.f, q1 = 0.f;
  for (int p = p0 + p_off; p < p1; p += p_step) {
    float v[8];
    Ld8<TIn>::ld(base + ((long long)p * vpp + vi) * 8, v);
    s0 += (v[0] + v[1]) + (v[2] + v[3]);
    q0 += (v[0] * v[0] + v[1] * v[1]) + (v[2] * v[2] + v[3] * v[3]);
    s1 += (v[4] + v[5]) + (v[6] + v[7]);
    q1 += (v[4] * v[4] + v[5] * v[5]) + (v[6] * v[6] + v[7] * v[7]);
  }
  // Fixed-order block reduction (no float atomics): every thread parks its 4 partials, then 64
  // threads (group, stat) each add the 16 entries that belong to their group in a fixed order.
  __shared__ float parked[kGnThreads][4];
  parked[threadIdx.x][0] = s0;
  parked[threadIdx.x][1] = q0;
  parked[threadIdx.x][2] = s1;
  parked[threadIdx.x][3] = q1;
  __syncthreads();
  if (threadIdx.x < kGroups * 2) {
    const int g = threadIdx.x >> 1, stat = threadIdx.x & 1;
    const int halves_per_group = cpg >> 2;              // 4-channel halves of an 8-channel vector
    float t = 0.f;
    for (int hh = g * halves_per_group; hh < (g + 1) * halves_per_group; ++hh) {
      const int v = hh >> 1, half = hh & 1;
      for (int po = 0; po < p_step; ++po) t += parked[po * vpp + v][half * 2 + stat];
    }
    partial[((long long)img * gridDim.x + chunk) * (kGroups * 2) + threadIdx.x] = t;
  }
}

// Partial records are reduced by up to kGnSlices blocks per image; the last block to finish (a ticket per image)
// folds the slices in slice order, so the result does not depend on which block that is.
constexpr int kGnSlices = 128;
// Reduction of the partial records [B][n_chunks][32 groups][2] (conv epilogue: one record per 32 pixels; standalone
// statistics pass: one per block).  Grid (slices, B): every warp reads whole 256-byte records (coalesced), the block
// folds its 8 warps in warp order into slice sums (double), and the last block of an image folds the slices in slice
// order -> sums[B][32][2] (row tiling: all-reduced by the caller) and / or the per-(image, channel) scale / shift.
// (Round 2: the conv epilogue stopped combining its four TMEM lane quarters through shared memory, so there are 4x
// more records; one block per (group, image) reading 8 bytes at a 256-byte stride no longer hides that.)
__global__ void __launch_bounds__(256)
gn_reduce_kernel(const float* __restrict__ partial, int n_chunks, double* __restrict__ slice_sums,
                 unsigned int* __restrict__ tickets, double* __restrict__ sums, const float* __restrict__ gamma,
                 const float* __restrict__ beta, float* __restrict__ scale, float* __restrict__ shift, int C,
                 double count, float eps) {
  const int img = blockIdx.y, S = gridDim.x, sl = blockIdx.x;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int per = (n_chunks + S - 1) / S;
  const int c0 = sl * per, c1 = min(n_chunks, c0 + per);
  __shared__ double rs[8][kGroups], rq[8][kGroups];
  __shared__ int s_last;
  double s = 0.0, q = 0.0;
  const float2* rec = reinterpret_cast<const float2*>(partial) + (long long)img * n_chunks * kGroups + lane;
#pragma unroll 4
  for (int c = c0 + w; c < c1; c += 8) {
    const float2 pp = rec[(long long)c * kGroups];
    s += (double)pp.x;
    q += (double)pp.y;
  }
  rs[w][lane] = s;
  rq[w][lane] = q;
  __syncthreads();
  if (w == 0) {
    for (int k = 1; k < 8; ++k) { s += rs[k][lane]; q += rq[k][lane]; }
    double* o = slice_sums + (((long long)img * S + sl) * kGroups + lane) * 2;
    o[0] = s; o[1] = q;
    __threadfence();
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int t = atomicAdd(&tickets[img], 1u);
    s_last = (t == (unsigned int)S - 1u) ? 1 : 0;
    if (s_last) tickets[img] = 0;                       // ready for the next layer
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  if (w == 0) {
    double ts = 0.0, tq = 0.0;
    for (int k = 0; k < S; ++k) {
      const double* o = slice_sums + (((long long)img * S + k) * kGroups + lane) * 2;
      ts += __ldcg(o); tq += __ldcg(o + 1);
    }
    if (sums != nullptr) { sums[((long long)img * kGroups + lane) * 2] = ts; sums[((long long)img * kGroups + lane) * 2 + 1] = tq; }
    rs[0][lane] = ts; rq[0][lane] = tq;
  }
  __syncthreads();
  if (scale == nullptr) return;
  const int cpg = C / kGroups;
  for (int c = threadIdx.x; c < C; c += 256) {
    const int g = c / cpg;
    const double mean = rs[0][g] / count;
    double var = rq[0][g] / count - mean * mean;
    if (var < 0.0) var = 0.0;
    const float rstd = (float)(1.0 / sqrt(var + (double)eps));
    const float a = gamma[c] * rstd;
    scale[(long long)img * C + c] = a;
    shift[(long long)img * C + c] = beta[c] - (float)mean * a;
  }
}
static int gn_slices(int n_chunks) {
  int sl = n_chunks / 32;
  return sl < 1 ? 1 : (sl > kGnSlices ? kGnSlices : sl);
}


// v[j] = [silu](v[j] * a[j] + b[j]) for 8 channels of one pixel, in packed fp32 pairs (FFMA2 / FMUL2 / FADD2): the same
// operations in the same order as the scalar form, bit for bit, and the SAME helper (silu_nr2) the conv kernel's in-place
// slab transform uses, which is what keeps the two roads identical.  A third fewer instructions; measured neutral on the
// kernel's time (0.484 vs 0.488 ms for the 128-channel layers at 4 x 1024^2): it waits on its latency chain, not on issue.
// kNewton: how the SiLU's exp / reciprocal are evaluated — ex2 + Newton reciprocal (one XU op, 16-bit outputs) or ex2 +
// rcp (two XU ops, fp32 / hi|lo|hi outputs)
template <bool kSilu, bool kNewton>
__device__ __forceinline__ void norm_act8(float (&v)[8], const float (&a)[8], const float (&b)[8]) {
#pragma unroll
  for (int j = 0; j < 8; j += 2) {
    float2 t = f2_fma(make_float2(v[j], v[j + 1]), make_float2(a[j], a[j + 1]), make_float2(b[j], b[j + 1]));
    if (kSilu) {
      if (kNewton) t = silu_nr2(t);
      else t = make_float2(silu_mufu(t.x), silu_mufu(t.y));
    }
    v[j] = t.x; v[j + 1] = t.y;
  }
}

template <typename TIn, typename TOut, bool kSilu, bool kNewton>
__global__ void __launch_bounds__(kGnThreads)
gn_apply_kernel(const TIn* __restrict__ x, TOut* __restrict__ y, const float* __restrict__ scale,
                const float* __restrict__ shift, int HW, int C, int px_per_block, long long x_img_stride,
                long long y_img_stride, float in_scale) {
  extern __shared__ float tab[];   // [2][C]
  const int img = blockIdx.y;
  for (int c = threadIdx.x; c < C; c += kGnThreads) {
    tab[c] = scale[(long long)img * C + c];
    tab[C + c] = shift[(long long)img * C + c];
  }
  __syncthreads();
  const int vpp = C >> 3;
  const int vi = threadIdx.x % vpp;
  const int p_off = threadIdx.x / vpp;
  const int p_step = kGnThreads / vpp;
  const int p0 = blockIdx.x * px_per_block;
  const int p1 = min(HW, p0 + px_per_block);
  float a[8], b[8];
#pragma unroll
  // in_scale: x is stored scaled by 1 / in_scale (a power of two: exact) — folded into the per-channel scale
  for (int j = 0; j < 8; ++j) { a[j] = tab[vi * 8 + j] * in_scale; b[j] = tab[C + vi * 8 + j]; }
  const TIn* xin = x + (long long)img * x_img_stride;
  TOut* yout = y + (long long)img * y_img_stride;
  // U pixels per iteration: all loads are issued before the first use (memory-level parallelism).  (8 in flight for
  // the 16-bit-input layers measured no faster than 4: those layers are bound by the XU latency chain, not by loads.)
  constexpr int U = 4;
  int p = p0 + p_off;
  for (; p + (U - 1) * p_step < p1; p += U * p_step) {
    float v[U][8];
#pragma unroll
    for (int u = 0; u < U; ++u) Ld8<TIn>::ld(xin + ((long long)(p + u * p_step) * vpp + vi) * 8, v[u]);
#pragma unroll
    for (int u = 0; u < U; ++u) {
      norm_act8<kSilu, kNewton>(v[u], a, b);
      store8<TOut>(yout, (long long)(p + u * p_step), vpp, vi, v[u]);
    }
  }
  for (; p < p1; p += p_step) {
    float v[8];
    Ld8<TIn>::ld(xin + ((long long)p * vpp + vi) * 8, v);
    norm_act8<kSilu, kNewton>(v, a, b);
    store8<TOut>(yout, (long long)p, vpp, vi, v);
  }
}

size_t gn_scratch_bytes(int B, int C, int max_chunks) {
  return ((size_t)B * max_chunks * kGroups * 2 + (size_t)2 * B * C + 2) * sizeof(float) + (size_t)B * kGroups * 2 * sizeof(double) +
         (size_t)B * kGnSlices * kGroups * 2 * sizeof(double) + ((size_t)B + 1) * sizeof(unsigned int);
}

static void gn_chunking(int B, int HW, int C, int max_chunks, int* chunks, int* px_per_block) {
  const int px_per_iter = kGnThreads / (C >> 3);
  int want = (148 * 8 + B - 1) / B;                 // ~8 CTAs per SM over the whole batch
  int maxc = (HW + px_per_iter * 4 - 1) / (px_per_iter * 4);   // at least 4 iterations per thread
  if (maxc < 1) maxc = 1;
  int c = want < maxc ? want : maxc;
  if (c > max_chunks) c = max_chunks;
  int ppb = (HW + c - 1) / c;
  ppb = (ppb + px_per_iter - 1) / px_per_iter * px_per_iter;
  *px_per_block = ppb;
  *chunks = (HW + ppb - 1) / ppb;
}

static void gn_chunking(int B, int HW, int C, int max_chunks, int* chunks, int* px_per_block);

// Grid of the apply kernel: ONE full wave over the whole batch — blocks = SMs x (blocks that are actually resident per SM
// for this instantiation), split evenly over the images.  (Round 1 launched 148 x 8 blocks while 5 or 6 fit per SM: a
// second wave one third full, i.e. the last ~25 % of the time with two thirds of the chip idle.)
template <typename Kernel>
static void apply_chunking(Kernel kernel, int* cached_per_sm, size_t smem, int B, int HW, int C, int* chunks, int* px_per_block) {
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) sms = 148;
  }
  if (*cached_per_sm == 0) {
    int n = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, kGnThreads, smem) != cudaSuccess || n < 1) n = 4;
    *cached_per_sm = n;
  }
  const int px_per_iter = kGnThreads / (C >> 3);
  int c = sms * *cached_per_sm / B;
  int maxc = (HW + px_per_iter * 4 - 1) / (px_per_iter * 4);   // at least 4 iterations per thread
  if (c > maxc) c = maxc;
  if (c < 1) c = 1;
  int ppb = (HW + c - 1) / c;
  ppb = (ppb + px_per_iter - 1) / px_per_iter * px_per_iter;
  *px_per_block = ppb;
  *chunks = (HW + ppb - 1) / ppb;
}

template <typename TIn, typename TOut>
static void launch_apply(const void* x, void* y, const float* scale, const float* shift, int B, int HW, int C, int /*chunks*/,
                         int /*ppb*/, bool silu, long long xs, long long ys, cudaStream_t s, float in_scale = 1.f) {
  const size_t sm = 2 * C * sizeof(float);
  // This kernel is not purely HBM bound: same-box A/B of the C2 step 44.3 ms (polynomial exp) vs 43.4 ms (ex2 + rcp).
  // 16-bit outputs take ex2 + Newton reciprocal (silu_nr2); fp32 / hi|lo|hi outputs (high-precision mode) ex2 + rcp.
  constexpr bool kNewton = sizeof(TOut) == 2 && !std::is_same<TOut, HalfSplit3>::value;
  static int occ[2] = {0, 0};
  int chunks = 1, ppb = HW;
  const TIn* xi = reinterpret_cast<const TIn*>(x);
  TOut* yo = reinterpret_cast<TOut*>(y);
  if (silu) {
    apply_chunking(gn_apply_kernel<TIn, TOut, true, kNewton>, &occ[0], sm, B, HW, C, &chunks, &ppb);
    gn_apply_kernel<TIn, TOut, true, kNewton><<<dim3(chunks, B), kGnThreads, sm, s>>>(xi, yo, scale, shift, HW, C, ppb, xs, ys, in_scale);
  } else {
    apply_chunking(gn_apply_kernel<TIn, TOut, false, false>, &occ[1], sm, B, HW, C, &chunks, &ppb);
    gn_apply_kernel<TIn, TOut, false, false><<<dim3(chunks, B), kGnThreads, sm, s>>>(xi, yo, scale, shift, HW, C, ppb, xs, ys, in_scale);
  }
}

// Row tiling: the statistics of a (image, group) are sums over ALL ranks' rows.  gn_reduce_partials folds this
// rank's conv-emitted partials into sums[B][32][2] (double, fixed order); the host all-reduces that block (SUM);
// gn_finalize_sums turns the global sums into per-(image, channel) scale / shift.
__global__ void gn_finalize_sums_kernel(const double* __restrict__ sums, const float* __restrict__ gamma,
                                        const float* __restrict__ beta, float* __restrict__ scale, float* __restrict__ shift,
                                        int C, double count, float eps) {
  const int img = blockIdx.x;
  const int cpg = C / kGroups;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const int g = c / cpg;
    const double mean = sums[((long long)img * kGroups + g) * 2] / count;
    double var = sums[((long long)img * kGroups + g) * 2 + 1] / count - mean * mean;
    if (var < 0.0) var = 0.0;
    const float a = gamma[c] * (float)(1.0 / sqrt(var + (double)eps));
    scale[(long long)img * C + c] = a;
    shift[(long long)img * C + c] = beta[c] - (float)mean * a;
  }
}
// scratch layout (gn_scratch_bytes): [partials: B*max_chunks*64 floats][sums: B*64 doubles][scale: B*C][shift: B*C]
double* gn_sums_ptr(void* scratch, int B, int C, int max_chunks) {
  (void)C;
  return reinterpret_cast<double*>(reinterpret_cast<float*>(scratch) + (size_t)B * max_chunks * kGroups * 2);
}
// [partials][sums][slice sums: B*kGnSlices*64 doubles][tickets: B (+1)][scale: B*C][shift: B*C] — nothing in front of
// the tickets depends on C (a scratch buffer sized for 512 channels serves every layer)
static double* gn_slice_ptr(void* scratch, int B, int max_chunks) {
  return gn_sums_ptr(scratch, B, 0, max_chunks) + (size_t)B * kGroups * 2;
}
static unsigned int* gn_ticket_ptr(void* scratch, int B, int max_chunks) {
  return reinterpret_cast<unsigned int*>(gn_slice_ptr(scratch, B, max_chunks) + (size_t)B * kGnSlices * kGroups * 2);
}
static float* gn_scale_ptr(void* scratch, int B, int max_chunks) {
  return reinterpret_cast<float*>(gn_ticket_ptr(scratch, B, max_chunks) + B + 1);
}
// The tickets must be zero before the first GroupNorm that uses a scratch buffer (they reset themselves afterwards).
int gn_scratch_reset(void* scratch, int B, int max_chunks, cudaStream_t s) {
  HDRVAE_CUDA_OK(cudaMemsetAsync(gn_ticket_ptr(scratch, B, max_chunks), 0, (size_t)B * sizeof(unsigned int), s));
  return 0;
}
int launch_gn_reduce_partials(void* scratch, int B, int C, int max_chunks, int n_partials, cudaStream_t s) {
  gn_reduce_kernel<<<dim3(gn_slices(n_partials), B), 256, 0, s>>>(reinterpret_cast<const float*>(scratch), n_partials,
                                                                    gn_slice_ptr(scratch, B, max_chunks), gn_ticket_ptr(scratch, B, max_chunks),
                                                                    gn_sums_ptr(scratch, B, C, max_chunks), nullptr, nullptr, nullptr, nullptr, C, 1.0, 0.f);
  HDRVAE_LAUNCHED();
  HDRVAE_CUDA_OK(cudaGetLastError());
  return 0;
}
// Row tiling, normalisation applied inside the consuming conv: only the all-reduced sums -> scale / shift.
int launch_gn_scale_shift_from_sums(int B, int C, const float* gamma, const float* beta, void* scratch, int max_chunks,
                                    double count, cudaStream_t s, const float** scale_out, const float** shift_out) {
  float* scale = gn_scale_ptr(scratch, B, max_chunks);
  float* shift = scale + (size_t)B * C;
  gn_finalize_sums_kernel<<<B, 256, 0, s>>>(gn_sums_ptr(scratch, B, C, max_chunks), gamma, beta, scale, shift, C, count, 1e-6f);
  HDRVAE_LAUNCHED();
  HDRVAE_CUDA_OK(cudaGetLastError());
  *scale_out = scale; *shift_out = shift;
  return 0;
}
// x / y point at the first row to normalise; rows_px = pixels per image to process; count = elements per (image, group)
// over ALL ranks
int launch_gn_apply_from_sums(const void* x, int x_dtype, long long x_img_stride, void* y, int y_dtype, long long y_img_stride,
                              int B, int rows_px, int C, const float* gamma, const float* beta, bool silu, void* scratch,
                              int max_chunks, double count, cudaStream_t s, float in_scale) {
  HDRVAE_REQUIRE((y_dtype == DT_F16 || y_dtype == DT_BF16) && (x_dtype == DT_F32 || x_dtype == y_dtype),
                 "groupnorm (row tiling): fp32 or operand-typed in, 16-bit out");
  float* scale = gn_scale_ptr(scratch, B, max_chunks);
  float* shift = scale + (size_t)B * C;
  gn_finalize_sums_kernel<<<B, 256, 0, s>>>(gn_sums_ptr(scratch, B, C, max_chunks), gamma, beta, scale, shift, C, count, 1e-6f);
  HDRVAE_LAUNCHED();
  int chunks, ppb;
  gn_chunking(B, rows_px, C, max_chunks, &chunks, &ppb);
  if (x_dtype == DT_F32) {
    if (y_dtype == DT_F16) launch_apply<float, __half>(x, y, scale, shift, B, rows_px, C, chunks, ppb, silu, x_img_stride, y_img_stride, s, in_scale);
    else launch_apply<float, __nv_bfloat16>(x, y, scale, shift, B, rows_px, C, chunks, ppb, silu, x_img_stride, y_img_stride, s, in_scale);
  } else if (y_dtype == DT_F16) {
    launch_apply<__half, __half>(x, y, scale, shift, B, rows_px, C, chunks, ppb, silu, x_img_stride, y_img_stride, s, in_scale);
  } else {
    launch_apply<__nv_bfloat16, __nv_bfloat16>(x, y, scale, shift, B, rows_px, C, chunks, ppb, silu, x_img_stride, y_img_stride, s, in_scale);
  }
  HDRVAE_LAUNCHED();
  HDRVAE_CUDA_OK(cudaGetLastError());
  return 0;
}

// Only the reduction: the producer's partials -> per-(image, channel) scale / shift in the scratch buffer (returned), for a
// conv that applies the normalisation itself (gemm_tc.cu, GemmParams::xf_*).
int launch_gn_scale_shift(int B, int HW, int C, const float* gamma, const float* beta, void* scratch, int max_chunks,
                          int partial_chunks, cudaStream_t s, const float** scale_out, const float** shift_out) {
  HDRVAE_REQUIRE(partial_chunks > 0 && C % 32 == 0, "groupnorm (fused into the conv): needs the producer's statistics");
  float* scale = gn_scale_ptr(scratch, B, max_chunks);
  float* shift = scale + (size_t)B * C;
  gn_reduce_kernel<<<dim3(gn_slices(partial_chunks), B), 256, 0, s>>>(reinterpret_cast<const float*>(scratch), partial_chunks,
                                                                       gn_slice_ptr(scratch, B, max_chunks), gn_ticket_ptr(scratch, B, max_chunks),
                                                                       nullptr, gamma, beta, scale, shift, C, (double)HW * (double)(C / kGroups), 1e-6f);
  HDRVAE_LAUNCHED();
  HDRVAE_CUDA_OK(cudaGetLastError());
  *scale_out = scale; *shift_out = shift;
  return 0;
}

// partial_chunks > 0: the statistics partials [B][partial_chunks][32][2] are already in the scratch buffer
// (emitted by the producing conv); otherwise a standalone statistics pass over x runs first.
int launch_groupnorm(const void* x, int x_dtype, void* y, int y_dtype, int B, int HW, int C, const float* gamma,
                     const float* beta, bool silu, void* scratch, int max_chunks, int partial_chunks, cudaStream_t s,
                     float in_scale) {
  HDRVAE_REQUIRE(C % 32 == 0 && C >= 128 && C <= 2048 && (kGnThreads % (C >> 3)) == 0,
                 "groupnorm: unsupported channel count %d", C);
  HDRVAE_REQUIRE(in_scale == 1.f || partial_chunks > 0, "groupnorm: a scaled input needs the producer's statistics");
  HDRVAE_REQUIRE(y_dtype == DT_BF16 || y_dtype == DT_F16 || y_dtype == DT_F32 || y_dtype == DT_F16X3,
                 "groupnorm: output must be a 16-bit operand type, fp32 or the fp16 hi|lo|hi operand");
  HDRVAE_REQUIRE((y_dtype != DT_F32 && y_dtype != DT_F16X3) || x_dtype == DT_F32, "groupnorm: fp32 / split outputs need fp32 input");
  int chunks, ppb;
  gn_chunking(B, HW, C, max_chunks, &chunks, &ppb);
  float* partial = reinterpret_cast<float*>(scratch);
  float* scale = gn_scale_ptr(scratch, B, max_chunks);
  float* shift = scale + (size_t)B * C;
  int n_partials = partial_chunks;
  if (partial_chunks <= 0) {
    const dim3 grid(chunks, B);
    if (x_dtype == DT_F32) gn_stats_kernel<float><<<grid, kGnThreads, 0, s>>>(reinterpret_cast<const float*>(x), partial, HW, C, ppb);
    else if (x_dtype == DT_BF16) gn_stats_kernel<__nv_bfloat16><<<grid, kGnThreads, 0, s>>>(reinterpret_cast<const __nv_bfloat16*>(x), partial, HW, C, ppb);
    else gn_stats_kernel<__half><<<grid, kGnThreads, 0, s>>>(reinterpret_cast<const __half*>(x), partial, HW, C, ppb);
    HDRVAE_LAUNCHED();
    HDRVAE_CUDA_OK(cudaGetLastError());
    n_partials = chunks;
  }
  gn_reduce_kernel<<<dim3(gn_slices(n_partials), B), 256, 0, s>>>(partial, n_partials, gn_slice_ptr(scratch, B, max_chunks),
                                                                    gn_ticket_ptr(scratch, B, max_chunks), nullptr, gamma, beta, scale, shift, C,
                                                                    (double)HW * (double)(C / kGroups), 1e-6f);
  HDRVAE_LAUNCHED();
  HDRVAE_CUDA_OK(cudaGetLastError());
  if (y_dtype == DT_F32) {
    launch_apply<float, float>(x, y, scale, shift, B, HW, C, chunks, ppb, silu, (long long)HW * C, (long long)HW * C, s, in_scale);
  } else if (y_dtype == DT_F16X3) {
    // y_img_stride is counted in HalfSplit3 elements = 2-byte units
    launch_apply<float, HalfSplit3>(x, y, scale, shift, B, HW, C, chunks, ppb, silu, (long long)HW * C, (long long)HW * C * 3, s, in_scale);
  } else if (y_dtype == DT_F16) {
    if (x_dtype == DT_F32) launch_apply<float, __half>(x, y, scale, shift, B, HW, C, chunks, ppb, silu, (long long)HW * C, (long long)HW * C, s, in_scale);
    else if (x_dtype == DT_BF16) launch_apply<__nv_bfloat16, __half>(x, y, scale, shift, B, HW, C, chunks, ppb, silu, (long long)HW * C, (long long)HW * C, s, in_scale);
    else launch_apply<__half, __half>(x, y, scale, shift, B, HW, C, chunks, ppb, silu, (long long)HW * C, (long long)HW * C, s, in_scale);
  } else {
    if (x_dtype == DT_F32) launch_apply<float, __nv_bfloat16>(x, y, scale, shift, B, HW, C, chunks, ppb, silu, (long long)HW * C, (long long)HW * C, s, in_scale);
    else if (x_dtype == DT_BF16) launch_apply<__nv_bfloat16, __nv_bfloat16>(x, y, scale, shift, B, HW, C, chunks, ppb, silu, (long long)HW * C, (long long)HW * C, s, in_scale);
    else launch_apply<__half, __nv_bfloat16>(x, y, scale, shift, B, HW, C, chunks, ppb, silu, (long long)HW * C, (long long)HW * C, s, in_scale);
  }
  HDRVAE_LAUNCHED();
  HDRVAE_CUDA_OK(cudaGetLastError());
  return 0;
}

}  // namespace hdrvae
