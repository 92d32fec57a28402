// Shared host/device helpers for libhdrvae (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <string>

namespace hdrvae {

void set_error(const char* fmt, ...);
extern long long g_launch_count;   // kernels launched by this library (bench.py's gpu_launches)
#define HDRVAE_LAUNCHED() (++::hdrvae::g_launch_count)

#define HDRVAE_CUDA_OK(expr)                                                                  \
  do {                                                                                        \
    cudaError_t _e = (expr);                                                                  \
    if (_e != cudaSuccess) {                                                                  \
      ::hdrvae::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return -1;                                                                              \
    }                                                                                         \
  } while (0)

#define HDRVAE_REQUIRE(cond, ...)       \
  do {                                  \
    if (!(cond)) {                      \
      ::hdrvae::set_error(__VA_ARGS__); \
      return -2;                        \
    }                                   \
  } while (0)

#define HDRVAE_TRY(expr)      \
  do {                        \
    int _r = (expr);          \
    if (_r != 0) return _r;   \
  } while (0)

// The library's environment switches (DESIGN.md §6), read once per process by switches() (api.cu).  Defaults are the
// product path; each field says what setting the variable changes.
struct Switches {
  bool h16 = true;           // HDRVAE_H16=0: the block-internal tensor h in fp32
  bool x16 = true;           // HDRVAE_X16=0: the residual stream in fp32
  bool fuse_nin = true;      // HDRVAE_FUSE_NIN=0: nin_shortcut as its own launch
  bool fuse_gn = true;       // HDRVAE_FUSE_GN=0: GroupNorm + SiLU by the streaming kernel everywhere
  bool graphs = true;        // HDRVAE_NO_GRAPH=1: no CUDA-graph capture
  bool conv_direct = false;  // HDRVAE_CONV_IMPL=direct: new contexts start on the CUDA-core validation conv
  int gemm_dbg = 0;          // HDRVAE_GEMM_DBG: GemmParams::dbg of every tensor-core GEMM launch
};
const Switches& switches();

inline int ceil_div(long long a, long long b) { return static_cast<int>((a + b - 1) / b); }
inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// ----------------------------------------------------------------- GEMM / conv descriptor
// element type codes = the ABI codes of include/hdrvae.h
enum { DT_F32 = 0, DT_BF16 = 1, DT_F16 = 2,
       DT_F16X3 = 3 /* internal: fp16 [hi | lo | hi] K-concatenated operand of the "high" precision mode (groupnorm output) */ };
__host__ __device__ inline int dt_bytes(int dt) { return dt == DT_F32 ? 4 : 2; }

// out[n, y*sy+py, x*sx+px, col] = row_scale[x] * alpha * sum_{t<ntaps} sum_{c<K_per_tap}
//        A[n, y+dy[t], x+dx[t], c] * Bw[col][t*K_per_tap + c]  + bias[col]  (+ residual[...])
// A is addressed as a 4-D NHWC tensor (plain matrices use H = N = 1, W = rows).
// Operand type ab_dtype: DT_F16 / DT_BF16 -> tcgen05 kind::f16, DT_F32 -> kind::tf32 (the tensor core
// reads the top 19 bits of each fp32).
struct GemmParams {
  // A operand (activations): element strides, used by the direct kernel; the tcgen05 kernel
  // reads A through a TMA tensor map built from the same numbers.
  const void* a;
  long long a_img_stride, a_row_stride, a_px_stride;
  // B operand (weights / keys), [cols][ktot] K-major, same element type as A
  const void* b;
  long long b_row_stride;
  int b_rows;       // rows of B that exist in memory (0: same as n_cols); rows beyond are zero-filled by TMA
  int ab_dtype;
  int n_img, H, W;  // source grid of the M dimension
  int y_pad;        // halo rows stored above/below the H rows of A (row tiling): `a` points at the slab start, the
                    // A rows addressed are y + dy + y_pad of H + 2*y_pad stored rows (0: vertical padding by TMA zero fill)
  int k_per_tap;    // elements; multiple of one 128-byte row (64 for 16-bit operands, 32 for tf32)
  int a_k_valid;    // channels of A that exist per pixel (0: k_per_tap).  Smaller than k_per_tap when a conv reads a
                    // channel prefix that is not a multiple of the 128-byte row (dense-block concat buffers): TMA
                    // zero-fills the tail of the last K block, the packed weights hold zeros there
  int ntaps;
  int tap_dy[9], tap_dx[9];
  // Extra K blocks from a SECOND tensor (slab form only): after the 9 taps of A the kernel accumulates
  //   sum_{c < k2} A2[n, y, x, c] * B2[col][c]
  // into the same tile — a 1x1 conv of another tensor fused into this conv (the decoder's nin_shortcut, whose output is
  // the residual of conv2: no separate launch, no fp32 round trip).  A2 has A's spatial shape and halo rows (y_pad).
  const void* a2;
  long long a2_img_stride, a2_row_stride, a2_px_stride;
  int k2;                    // channels of A2 (multiple of 64 elements of 16 bits), 0: none
  const void* b2;            // [cols][k2] K-major, same element type
  long long b2_row_stride;
  int n_cols;       // valid output columns (Cout)
  // tiling of the M dimension: TW x TH = 128 pixels
  int tw_log2, TW, TH, tiles_x, tiles_y, n_tiles_n;
  // output
  void* out;
  int out_dtype;
  float out_scale;   // multiplier of a 16-bit main output (0 is read as 1): un-normalised tensors are stored scaled by a
                     // power of two so that fp16 cannot overflow (statistics are taken of the un-scaled values)
  long long out_img_stride, out_row_stride, out_px_stride;  // elements
  int sy, sx, py, px;
  const float* bias;
  int bias_per_row;  // bias indexed by the M row (x coordinate) instead of the column
  const void* residual;  // same addressing as out, or null
  int res_dtype;
  float res_scale;   // multiplier of `residual` (0 is read as 1)
  const float* residual2;  // second fp32 residual, same addressing as out, added unscaled; or null
  float lrelu;       // LeakyReLU negative slope applied last (0: none)
  int n_store;       // columns actually stored (multiple of 4; 0: n_cols) — a Cout padded up to 32 stores less
  const float* row_scale;  // per M row (x coordinate) multiplier of the accumulator, or null
  float alpha;       // accumulator scale applied before bias (1.0 for convs)
  void* out2;        // optional second output: out * out2_scale as a 16-bit tensor (same addressing), or null
  int out2_dtype;
  float out2_scale;
  long long out2_img_stride, out2_row_stride, out2_px_stride;  // elements; all 0: same addressing as out
  int round_tf32;    // round fp32 outputs to tf32 (RN) so a following kind::tf32 MMA reads them exactly
  // GroupNorm statistics of the output, emitted per (image, m-tile) as (sum, sum of squares) of each of the
  // 32 channel groups: stats[((img * tiles_per_img + m_tile) * 32 + group) * 2 + {0,1}], or null
  float* stats;
  int stats_chunks_per_img, stats_chunk0;
  int slab;          // 3x3 conv with narrow output (<= 64 columns): 8x16-pixel tiles whose 10x18 activation slab is loaded
                     // ONCE per K block and read by the 9 taps as shifted descriptors (gemm_tc.cu "slab" variant)
  // GroupNorm + SiLU applied to A inside the kernel (slab form, fp16 A): two otherwise idle warps rewrite every landed
  // slab in place as silu(a * xf_in_scale * xf_scale[img][c] + xf_shift[img][c]) before the MMAs read it; pixels outside
  // the image (x outside [0, W), y outside [xf_y_lo, xf_y_hi)) become the conv's zero padding.  null: A is used as it is.
  const float* xf_scale;
  const float* xf_shift;
  float xf_in_scale;
  int xf_y_lo, xf_y_hi;
  int cta_group;     // 0 = library default (CTA pairs), 1 = single CTA, 2 = CTA pair (tcgen05 cta_group::2)
  int dbg;           // diagnostics (Switches::gemm_dbg): bit0 = producer skips the TMA loads, bit1 = issuer skips the MMAs,
                     // bit5 (32) = CTA 0 prints its wait cycles
};

#ifdef __CUDACC__
// SiLU with exp on the special-function unit (ex2 + rcp): two XU operations per element
__device__ __forceinline__ float silu_mufu(float v) { return __fdividef(v, 1.f + __expf(-v)); }
// Packed fp32 pairs (sm_100 FFMA2 / FADD2 / FMUL2): one issue slot per two lanes of arithmetic.
__device__ __forceinline__ float2 f2_fma(float2 a, float2 b, float2 c) {
  unsigned long long d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(*reinterpret_cast<unsigned long long*>(&a)),
      "l"(*reinterpret_cast<unsigned long long*>(&b)), "l"(*reinterpret_cast<unsigned long long*>(&c)));
  return *reinterpret_cast<float2*>(&d);
}
__device__ __forceinline__ float2 f2_add(float2 a, float2 b) {
  unsigned long long d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(*reinterpret_cast<unsigned long long*>(&a)),
      "l"(*reinterpret_cast<unsigned long long*>(&b)));
  return *reinterpret_cast<float2*>(&d);
}
__device__ __forceinline__ float2 f2_mul(float2 a, float2 b) {
  unsigned long long d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(*reinterpret_cast<unsigned long long*>(&a)),
      "l"(*reinterpret_cast<unsigned long long*>(&b)));
  return *reinterpret_cast<float2*>(&d);
}
// silu_nr on a pair: the same operations in the same order (so the results are bit-identical), FFMA2 / FMUL2 / FADD2 where
// a packed form exists.  Used by the GroupNorm + SiLU streaming kernel and by the conv kernel's in-place slab transform.
__device__ __forceinline__ float2 silu_nr2(float2 v) {
  const float2 m = f2_mul(v, make_float2(-1.4426950408889634f, -1.4426950408889634f));
  float2 e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e.x) : "f"(fminf(m.x, 80.f)));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e.y) : "f"(fminf(m.y, 80.f)));
  const float2 d = f2_add(make_float2(1.f, 1.f), e);
  const float2 nd = make_float2(-d.x, -d.y);
  const float2 two = make_float2(2.f, 2.f);
  float2 r = make_float2(__int_as_float(0x7EF311C7 - __float_as_int(d.x)), __int_as_float(0x7EF311C7 - __float_as_int(d.y)));
  r = f2_mul(r, f2_fma(nd, r, two));
  r = f2_mul(r, f2_fma(nd, r, two));
  return f2_mul(v, r);
}
// ONE XU operation per element: ex2 on the special-function unit, the reciprocal of d = 1 + e^-v (d >= 1) by two Newton
// steps on the FMA pipe from the integer-subtraction first guess (relative error 7.6e-6: far below the 16-bit output
// rounding).  ncu on the streaming GroupNorm kernel: XU pipe 53 % busy, DRAM 57 %, issue 40 % with ex2 + rcp — neither
// memory nor any one pipe saturated, the XU latency chain is what the warps wait on.
__device__ __forceinline__ float silu_nr(float v) {
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(fminf(-v * 1.4426950408889634f, 80.f)));
  const float d = 1.f + e;
  float r = __int_as_float(0x7EF311C7 - __float_as_int(d));
  r = r * fmaf(-d, r, 2.f);
  r = r * fmaf(-d, r, 2.f);
  return v * r;
}
#endif

// cudaFuncSetAttribute is per device: remember per (call site, device) whether the opt-in shared-memory size has
// been set, so that a process driving several GPUs (not the one-process-per-GPU model, but legal) still works.
struct PerDeviceOnce {
  bool done[64] = {};
  bool first() {
    int d = 0;
    if (cudaGetDevice(&d) != cudaSuccess || d < 0 || d >= 64) return true;
    if (done[d]) return false;
    done[d] = true;
    return true;
  }
};

struct TensorMapPair {
  CUtensorMap a, b, a2, b2;
};

}  // namespace hdrvae
