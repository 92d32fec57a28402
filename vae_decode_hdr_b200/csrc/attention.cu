// Fused single-head attention (d = 512) for the decoder's mid.attn_1 on tcgen05 / TMEM (sm_100a): ONE launch computes
//   O = softmax(alpha * Q K^T) V
// for every query row, flash-style: no score or probability matrix ever exists in HBM.  The reference reaches this op only
// through vae.decode (hdr_vae_decode.py:859,:1022 -> ComfyUI Decoder.mid.attn_1; graph in SURVEY.md §8 a3, K5).
//
// Budget that shapes the design (one SM: 512 TMEM columns, 227 KB of shared memory):
//   * the O accumulator of a 128-query tile is 128 x 512 fp32 = ALL 512 TMEM columns, so d_v is split in two halves that
//     are computed by different CTA pairs (each recomputes S = Q K^T: 1.5x the MMA work of an un-split kernel — the same
//     MMA count as the two-pass GEMM form this kernel replaces, without its P round trip through HBM);
//   * per CTA: O half = 256 columns, S double-buffered = 2 x 128 columns; P = exp(S - m) is written back over S as packed
//     16-bit pairs (64 columns) and the PV MMA reads its A operand straight from TMEM — P never touches shared memory;
//   * the Q tile (128 rows x 512) stays resident in shared memory (128 KB), K and V^T stream through a 6 x 16 KB TMA ring;
//   * a CTA PAIR (tcgen05 cta_group::2, M = 256) works on 256 query rows: each CTA stages only half of every K / V^T
//     tile, which halves the L2 -> SM operand traffic (the bound of the two-pass form's GEMMs at M = 128).
//
// Roles (192 threads): warp 0 TMA producer, warp 1 MMA issuer (leader CTA of the pair), warps 2..5 soft-max: one query row
// per thread (TMEM hands a thread its row), online soft-max with LAZY rescaling — the running reference maximum m is only
// raised (and O rescaled in TMEM) when a block's maximum exceeds it by more than 8 in the log2 domain, so P <= 2^8 fits
// fp16 and the O correction runs a handful of times per row instead of once per key block.
//
// Tensor-pipe order: S_0, S_1, PV_0, S_2, PV_1, ...: soft-max of block j overlaps S_{j+1} and PV_{j-1}.
#include <algorithm>

#include "engine.cuh"
#include "ptx.cuh"

namespace hdrvae {

namespace {

constexpr int kAThreads = 192;
constexpr int kASlots = 6;
constexpr int kASlotBytes = 16384;
constexpr int kAQBytes = 128 * 512 * 2;          // resident Q tile
constexpr int kABlockKeys = 128;
constexpr int kASmemBytes = kAQBytes + kASlots * kASlotBytes + 256 /*barriers*/ + 1024 /*align slack*/;
constexpr float kLazyThreshold = 8.0f;            // log2 units: P <= 2^8

struct AttnParams {
  int n_q;            // query rows per image (rows >= n_q are not stored)
  int n_keys;         // valid keys per image (columns >= n_keys are masked)
  int n_blocks;       // ceil(n_keys / 128)
  int q_pairs;        // ceil(n_q / 256): 256-row query groups per image
  int n_img;
  float alpha_log2;   // alpha * log2(e)
  uint16_t* o;        // [n_img][n_q][512] 16-bit
  long long o_img_stride;
  int bf16;
  // key splitting (few work units: small images, or one rank's share of a row-tiled image): the key blocks are divided
  // over `key_splits` units per (query group, d_v half); every unit writes its UN-normalised fp32 O rows and its
  // (reference maximum, row sum) and attn_merge_kernel combines them.  1: one unit sees all keys and stores O / l itself.
  int key_splits, blocks_per_split;
  float* o_part;      // [key_splits][n_img][n_q][512] fp32
  float* ml_part;     // [key_splits][n_img][n_q][2]   (m in the log2 domain, l)
};

__device__ __forceinline__ void tmem_st_32x32_x16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      :
      : "r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]),
        "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_32x32_x32(uint32_t taddr, const uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      :
      : "r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]),
        "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]),
        "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]),
        "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// D[tmem] (+)= A[tmem] * B[smem]^T: the A operand (P, packed 16-bit pairs: column c of a lane holds K elements 2c, 2c+1 of
// that row) is read from tensor memory.
__device__ __forceinline__ void umma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "}\n"
      :
      : "r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_f16_ts_pair(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "}\n"
      :
      : "r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__device__ __forceinline__ uint32_t pack16(float lo, float hi, bool bf16) {
  if (bf16) {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
  }
  __half2 v = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}

// CG = CTAs per MMA: 2 = CTA pair on 256 query rows (product path); 1 = every CTA on its own 128 rows (validation /
// bisecting build: N = 128 MMAs, same ring and soft-max code).
template <int CG>
__global__ void __launch_bounds__(kAThreads, 1)
attn_fused_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                  const __grid_constant__ CUtensorMap tmV, const AttnParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smem_q = smem;
  uint8_t* smem_ring = smem + kAQBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_ring + kASlots * kASlotBytes);
  uint64_t* full_bar = bars;                 // [6]
  uint64_t* empty_bar = bars + kASlots;      // [6]
  uint64_t* q_full = bars + 2 * kASlots;     // [1]
  uint64_t* s_full = q_full + 1;             // [2]
  uint64_t* p_full = s_full + 2;             // [2]
  uint64_t* o_full = p_full + 2;             // [1]
  uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(o_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = CG == 2 ? ptx::cluster_ctarank() : 0u;
  // work item: (image, 256-row (CG = 2) or 128-row (CG = 1) query group, d_v half); the two halves are neighbours in the
  // grid so that they stream the same K tiles through L2 at the same time
  const int unit0 = blockIdx.x / CG;
  const int split = unit0 % p.key_splits;
  const int unit = unit0 / p.key_splits;
  const int half = unit & 1;
  const int groups_per_img = CG == 2 ? p.q_pairs : p.q_pairs * 2;
  const int grp = (unit >> 1) % groups_per_img;
  const int img = (unit >> 1) / groups_per_img;
  const int row0 = grp * (128 * CG) + (int)rank * 128;
  const int kb0 = split * p.blocks_per_split;                  // first key block of this unit

  if (threadIdx.x == 0) {
    ptx::prefetch_tensormap(&tmQ); ptx::prefetch_tensormap(&tmK); ptx::prefetch_tensormap(&tmV);
    for (int i = 0; i < kASlots; ++i) { ptx::mbar_init(&full_bar[i], 1); ptx::mbar_init(&empty_bar[i], 1); }
    ptx::mbar_init(q_full, 1);
    for (int i = 0; i < 2; ++i) { ptx::mbar_init(&s_full[i], 1); ptx::mbar_init(&p_full[i], CG * 4); }
    ptx::mbar_init(o_full, 1);
    ptx::fence_barrier_init();
  }
  if (warp == 1) {
    if (CG == 2) ptx::tmem_alloc_pair<512>(tmem_ptr_s); else ptx::tmem_alloc<512>(tmem_ptr_s);
  }
  ptx::tc_fence_before_sync();
  if (CG == 2) ptx::cluster_sync_all(); else __syncthreads();
  ptx::tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_ptr_s;
  const uint32_t tmem_o = tmem_base + 256;
  const int nblk = min(p.blocks_per_split, p.n_blocks - kb0);

  // Ring slot contents (16 KB each).  K slot: 128 d of a key block — CG = 2: this CTA's 64 keys x (2 x 64 d), two 8 KB
  // boxes; CG = 1: 128 keys x 64 d, one box (then 8 K slots per block instead of 4).  V slot: 128 d_v rows x 64 keys —
  // CG = 2: this CTA's half of the pair's 256 d_v; CG = 1: one of the two 128-column quarters (4 V slots per block).
  constexpr int kKSlots = CG == 2 ? 4 : 8;
  constexpr int kVSlots = CG == 2 ? 2 : 4;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (ptx::elect_one()) {
      if (rank == 0) ptx::mbar_arrive_expect_tx(q_full, (uint32_t)(CG * kAQBytes));
      for (int c = 0; c < 8; ++c) {
        if (CG == 2) ptx::tma_load_3d_pair(smem_q + c * 16384, &tmQ, q_full, c * 64, row0, img);
        else ptx::tma_load_3d(smem_q + c * 16384, &tmQ, q_full, c * 64, row0, img);
      }
    }
    __syncwarp();
    int stage = 0;
    uint32_t phase = 0;
    for (int i = 0; i <= nblk; ++i) {
      if (i < nblk) {
        for (int s4 = 0; s4 < kKSlots; ++s4) {
          ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
          if (ptx::elect_one()) {
            if (rank == 0) ptx::mbar_arrive_expect_tx(&full_bar[stage], (uint32_t)(CG * kASlotBytes));
            uint8_t* dst = smem_ring + stage * kASlotBytes;
            if (CG == 2) {
              ptx::tma_load_3d_pair(dst, &tmK, &full_bar[stage], s4 * 128, (kb0 + i) * kABlockKeys + (int)rank * 64, img);
              ptx::tma_load_3d_pair(dst + 8192, &tmK, &full_bar[stage], s4 * 128 + 64, (kb0 + i) * kABlockKeys + (int)rank * 64, img);
            } else {
              ptx::tma_load_3d(dst, &tmK, &full_bar[stage], s4 * 64, (kb0 + i) * kABlockKeys, img);
            }
          }
          __syncwarp();
          if (++stage == kASlots) { stage = 0; phase ^= 1; }
        }
      }
      if (i >= 1) {
        for (int v = 0; v < kVSlots; ++v) {
          ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
          if (ptx::elect_one()) {
            if (rank == 0) ptx::mbar_arrive_expect_tx(&full_bar[stage], (uint32_t)(CG * kASlotBytes));
            uint8_t* dst = smem_ring + stage * kASlotBytes;
            // CG = 2: v = key chunk, rows = this CTA's 128 of the pair's 256 d_v; CG = 1: v = (key chunk, d_v quarter)
            const int kc = CG == 2 ? v : (v >> 1);
            const int vrow = half * 256 + (CG == 2 ? (int)rank * 128 : (v & 1) * 128);
            if (CG == 2) ptx::tma_load_3d_pair(dst, &tmV, &full_bar[stage], (kb0 + i - 1) * kABlockKeys + kc * 64, vrow, img);
            else ptx::tma_load_3d(dst, &tmV, &full_bar[stage], (kb0 + i - 1) * kABlockKeys + kc * 64, vrow, img);
          }
          __syncwarp();
          if (++stage == kASlots) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1 && rank == 0) {
    // ------------------------------------------------------------------ MMA issuer (leader CTA)
    const uint32_t fmt = p.bf16 ? 1u : 0u;
    const uint32_t idesc_s = ptx::make_idesc(fmt, 128 * CG, 128);
    const uint32_t idesc_o = ptx::make_idesc(fmt, 128 * CG, CG == 2 ? 256 : 128);
    ptx::mbar_wait(q_full, 0);
    ptx::tc_fence_after_sync();
    const uint32_t q_addr = ptx::smem_u32(smem_q);
    int stage = 0;
    uint32_t phase = 0;
    for (int i = 0; i <= nblk; ++i) {
      if (i < nblk) {
        // S_i = Q K_i^T into S buffer i & 1.  The buffer is free: PV_{i-2}, which read P_{i-2} from it, was issued before
        // (MMAs execute in order) and the soft-max warps finished with it before they released P_{i-2}.
        const uint32_t d_s = tmem_base + (i & 1) * 128;
        for (int s4 = 0; s4 < kKSlots; ++s4) {
          ptx::mbar_wait(&full_bar[stage], phase);
          ptx::tc_fence_after_sync();
          if (ptx::elect_one()) {
            const uint32_t sb = ptx::smem_u32(smem_ring + stage * kASlotBytes);
            constexpr int kSub = CG == 2 ? 2 : 1;
#pragma unroll
            for (int sub = 0; sub < kSub; ++sub) {
              const int chunk = s4 * kSub + sub;                                  // 64-wide d chunk of Q
              const uint64_t da = ptx::make_sw128_kmajor_desc(q_addr + chunk * 16384);
              const uint64_t db = ptx::make_sw128_kmajor_desc(sb + sub * 8192);
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                const uint32_t accum = (s4 | sub | k) != 0 ? 1u : 0u;
                if (CG == 2) ptx::umma_f16_pair(d_s, da + 2 * k, db + 2 * k, idesc_s, accum);
                else ptx::umma_f16(d_s, da + 2 * k, db + 2 * k, idesc_s, accum);
              }
            }
            if (CG == 2) ptx::umma_commit_pair(&empty_bar[stage]); else ptx::umma_commit(&empty_bar[stage]);
            if (s4 == kKSlots - 1) {
              if (CG == 2) ptx::umma_commit_pair(&s_full[i & 1]); else ptx::umma_commit(&s_full[i & 1]);
            }
          }
          __syncwarp();
          if (++stage == kASlots) { stage = 0; phase ^= 1; }
        }
      }
      if (i >= 1) {
        // O += P_j V_j, j = i - 1: A = P_j from TMEM (packed 16-bit, 8 columns per 16-key MMA step), B = V^T tile
        const int j = i - 1;
        ptx::mbar_wait(&p_full[j & 1], (uint32_t)((j >> 1) & 1));
        ptx::tc_fence_after_sync();
        const uint32_t a_p = tmem_base + (j & 1) * 128;
        for (int v = 0; v < kVSlots; ++v) {
          ptx::mbar_wait(&full_bar[stage], phase);
          ptx::tc_fence_after_sync();
          if (ptx::elect_one()) {
            const uint64_t db = ptx::make_sw128_kmajor_desc(ptx::smem_u32(smem_ring + stage * kASlotBytes));
            const int kc = CG == 2 ? v : (v >> 1);
            const uint32_t d_o = tmem_o + (CG == 2 ? 0 : (v & 1) * 128);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const uint32_t accum = (j | kc | k) != 0 ? 1u : 0u;
              const uint32_t a = a_p + (uint32_t)((kc * 4 + k) * 8);
              if (CG == 2) umma_f16_ts_pair(d_o, a, db + 2 * k, idesc_o, accum);
              else umma_f16_ts(d_o, a, db + 2 * k, idesc_o, accum);
            }
            if (CG == 2) ptx::umma_commit_pair(&empty_bar[stage]); else ptx::umma_commit(&empty_bar[stage]);
            if (v == kVSlots - 1) {
              if (CG == 2) ptx::umma_commit_pair(o_full); else ptx::umma_commit(o_full);
            }
          }
          __syncwarp();
          if (++stage == kASlots) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp >= 2) {
    // ------------------------------------------------------------------ soft-max + correction + output (4 warps)
    const int q = warp & 3;                                   // TMEM lane quarter this warp may access
    const int row = q * 32 + lane;
    const int grow = row0 + row;
    const uint32_t lane_addr = static_cast<uint32_t>(q * 32) << 16;
    const bool bf16 = p.bf16 != 0;
    const float a2 = p.alpha_log2;
    float m_ref = -INFINITY, l = 0.f;
    uint32_t v[32];
    for (int j = 0; j < nblk; ++j) {
      ptx::mbar_wait(&s_full[j & 1], (uint32_t)((j >> 1) & 1));
      ptx::tc_fence_after_sync();
      const uint32_t t_s = tmem_base + lane_addr + (j & 1) * 128;
      const int nvalid = p.n_keys - (kb0 + j) * kABlockKeys;   // >= 128 except in the last block of the image
      // pass 1: block maximum of this row
      float bm = -INFINITY;
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        ptx::tmem_ld_32x32(t_s + c * 32, v);
        ptx::tmem_ld_wait(v);
#pragma unroll
        for (int e = 0; e < 32; ++e) {
          const float sv = __uint_as_float(v[e]);
          bm = fmaxf(bm, (c * 32 + e) < nvalid ? sv : -INFINITY);
        }
      }
      bm *= a2;
      bool waited = false;
      if (j == 0) {
        m_ref = bm;
      } else if (__any_sync(0xffffffffu, bm > m_ref + kLazyThreshold)) {
        // raise the reference maximum: O (and l) of this warp's rows are rescaled in TMEM once PV_{j-1} has landed
        ptx::mbar_wait(o_full, (uint32_t)((j - 1) & 1));
        ptx::tc_fence_after_sync();
        waited = true;
        const float m_new = fmaxf(m_ref, bm);
        const float f = exp2f(m_ref - m_new);
        m_ref = m_new;
        l *= f;
#pragma unroll 1
        for (int c = 0; c < 8; ++c) {
          ptx::tmem_ld_32x32(tmem_o + lane_addr + c * 32, v);
          ptx::tmem_ld_wait(v);
#pragma unroll
          for (int e = 0; e < 32; ++e) v[e] = __float_as_uint(__uint_as_float(v[e]) * f);
          tmem_st_32x32_x32(tmem_o + lane_addr + c * 32, v);
        }
        tmem_st_wait();
      }
      // pass 2: P = exp2(alpha_log2 * s - m_ref), packed to 16-bit pairs over the S columns already consumed
      const float nm = -m_ref;
#pragma unroll 1
      for (int c = 0; c < 4; ++c) {
        ptx::tmem_ld_32x32(t_s + c * 32, v);
        ptx::tmem_ld_wait(v);
        uint32_t pk[16];
#pragma unroll
        for (int e = 0; e < 16; ++e) {
          float p0 = ex2_approx(fmaf(__uint_as_float(v[2 * e]), a2, nm));
          float p1 = ex2_approx(fmaf(__uint_as_float(v[2 * e + 1]), a2, nm));
          if ((c * 32 + 2 * e) >= nvalid) p0 = 0.f;
          if ((c * 32 + 2 * e + 1) >= nvalid) p1 = 0.f;
          l += p0 + p1;
          pk[e] = pack16(p0, p1, bf16);
        }
        tmem_st_32x32_x16(t_s + c * 16, pk);
      }
      tmem_st_wait();
      // keep o_full's phase in step (one wait per block) BEFORE releasing P_j: the barrier can then never run two phases
      // ahead of this warp.  PV_{j-1} was issued right after S_j, so it has normally landed by now.
      if (j >= 1 && !waited) ptx::mbar_wait(o_full, (uint32_t)((j - 1) & 1));
      ptx::tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) {
        if (CG == 2) ptx::mbar_arrive_cluster(&p_full[j & 1], 0); else ptx::mbar_arrive(&p_full[j & 1]);
      }
    }
    // output: O / l — or, with key splitting, the un-normalised fp32 rows plus (m, l) for the merge kernel
    ptx::mbar_wait(o_full, (uint32_t)((nblk - 1) & 1));
    ptx::tc_fence_after_sync();
    if (p.key_splits > 1) {
      const long long prow = ((long long)split * p.n_img + img) * p.n_q + grow;
      float* orow = p.o_part + prow * 512 + half * 256;
      if (half == 0 && grow < p.n_q) *reinterpret_cast<float2*>(p.ml_part + prow * 2) = make_float2(m_ref, l);
#pragma unroll 1
      for (int c = 0; c < 8; ++c) {
        ptx::tmem_ld_32x32(tmem_o + lane_addr + c * 32, v);
        ptx::tmem_ld_wait(v);
        if (grow < p.n_q) {
#pragma unroll
          for (int e = 0; e < 8; ++e)
            *reinterpret_cast<uint4*>(orow + c * 32 + e * 4) = make_uint4(v[4 * e], v[4 * e + 1], v[4 * e + 2], v[4 * e + 3]);
        }
      }
    } else {
      const float inv = 1.0f / l;
      uint16_t* orow = p.o + (long long)img * p.o_img_stride + (long long)grow * 512 + half * 256;
#pragma unroll 1
      for (int c = 0; c < 8; ++c) {
        ptx::tmem_ld_32x32(tmem_o + lane_addr + c * 32, v);
        ptx::tmem_ld_wait(v);
        if (grow < p.n_q) {
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            uint4 o4;
            o4.x = pack16(__uint_as_float(v[8 * e + 0]) * inv, __uint_as_float(v[8 * e + 1]) * inv, bf16);
            o4.y = pack16(__uint_as_float(v[8 * e + 2]) * inv, __uint_as_float(v[8 * e + 3]) * inv, bf16);
            o4.z = pack16(__uint_as_float(v[8 * e + 4]) * inv, __uint_as_float(v[8 * e + 5]) * inv, bf16);
            o4.w = pack16(__uint_as_float(v[8 * e + 6]) * inv, __uint_as_float(v[8 * e + 7]) * inv, bf16);
            *reinterpret_cast<uint4*>(orow + c * 32 + e * 8) = o4;
          }
        }
      }
    }
  }

  ptx::tc_fence_before_sync();
  if (CG == 2) ptx::cluster_sync_all(); else __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after_sync();
    if (CG == 2) ptx::tmem_dealloc_pair<512>(tmem_base); else ptx::tmem_dealloc<512>(tmem_base);
  }
}

// Key splitting, second step: o[row] = sum_s 2^(m_s - M) O_s[row] / sum_s 2^(m_s - M) l_s with M = max_s m_s.
// One block of 128 threads per query row, 4 columns per thread; splits in ascending order (deterministic).
__global__ void __launch_bounds__(128) attn_merge_kernel(const float* __restrict__ o_part, const float* __restrict__ ml_part,
                                                         int splits, long long rows, uint16_t* __restrict__ o, int bf16) {
  const long long row = blockIdx.x;
  float M = -INFINITY;
  for (int s = 0; s < splits; ++s) M = fmaxf(M, ml_part[(s * rows + row) * 2]);
  float L = 0.f;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int s = 0; s < splits; ++s) {
    const float2 ml = *reinterpret_cast<const float2*>(ml_part + (s * rows + row) * 2);
    const float w = exp2f(ml.x - M);
    L = fmaf(w, ml.y, L);
    const float4 v = *reinterpret_cast<const float4*>(o_part + (s * rows + row) * 512 + threadIdx.x * 4);
    acc.x = fmaf(w, v.x, acc.x); acc.y = fmaf(w, v.y, acc.y); acc.z = fmaf(w, v.z, acc.z); acc.w = fmaf(w, v.w, acc.w);
  }
  const float inv = 1.0f / L;
  uint2 r;
  r.x = pack16(acc.x * inv, acc.y * inv, bf16 != 0);
  r.y = pack16(acc.z * inv, acc.w * inv, bf16 != 0);
  *reinterpret_cast<uint2*>(o + row * 512 + threadIdx.x * 4) = r;
}

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

PFN_encodeTiled attn_encode_fn() {
  static PFN_encodeTiled fn = nullptr;
  if (fn) return fn;
  void* ptr = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) != cudaSuccess ||
      qres != cudaDriverEntryPointSuccess || ptr == nullptr)
    return nullptr;
  fn = reinterpret_cast<PFN_encodeTiled>(ptr);
  return fn;
}

int map3d(CUtensorMap* m, const void* base, int dt, long long d0, long long d1, long long d2, long long s1_elems,
          long long s2_elems, int b0, int b1) {
  PFN_encodeTiled enc = attn_encode_fn();
  HDRVAE_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled entry point not available");
  HDRVAE_REQUIRE((reinterpret_cast<uintptr_t>(base) & 15) == 0 && s1_elems % 8 == 0 && s2_elems % 8 == 0,
                 "attention: operand pointers / strides must be 16-byte aligned");
  cuuint64_t dims[3] = {(cuuint64_t)d0, (cuuint64_t)d1, (cuuint64_t)d2};
  cuuint64_t strides[2] = {(cuuint64_t)s1_elems * 2, (cuuint64_t)(d2 > 1 ? s2_elems : s1_elems * d1) * 2};
  cuuint32_t box[3] = {(cuuint32_t)b0, (cuuint32_t)b1, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(m, dt == DT_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(base),
                   dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  HDRVAE_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(attention) failed: %d (dims %lld %lld %lld)", (int)r, d0, d1, d2);
  return 0;
}

}  // namespace

// Key splits of the fused kernel, a function of the key count ONLY (never of the query count, the batch or the GPU): a
// row-tiled decode (few query rows per rank, all keys) and the single-GPU decode of the same image then run the same
// arithmetic per query row and stay bit-identical.  One split per 1024 key blocks (131 072 keys), at most 8: 1 up to
// 2048^2, 2 at 4096^2.  It exists for wave quantisation: one rank's 32 768 query rows of a 4096^2 image row-tiled over 8
// GPUs are 256 pair units = 3.46 waves of the 74 concurrent pairs (86 %); with 2 splits 6.9 waves (99 %).  More splits
// than needed cost: every unit loads its Q tile and ramps its pipeline again (measured at T = 65 536: 4 splits 9.20 ms
// against 8.57 ms unsplit), so the rule is as coarse as the C4 case allows.
int attention_key_splits(int n_keys) {
  const int n_blocks = (n_keys + kABlockKeys - 1) / kABlockKeys;
  int splits = 1;
  while (splits < 8 && n_blocks / (splits * 2) >= 1024) splits *= 2;
  return splits;
}

// q: [n_img][>= n_q rows][q_ld] 16-bit (512 columns used), k: [n_img][k_rows][k_ld] (rows >= n_keys are ignored),
// vt: [n_img][512][vt_ld] (V transposed: keys contiguous), o: [n_img][n_q][512].  alpha scales q k^T before the soft-max.
int launch_attention_fused(const void* q, long long q_ld, long long q_img_stride, int n_q, const void* k, long long k_ld,
                           long long k_img_stride, int k_rows, const void* vt, long long vt_ld, long long vt_img_stride,
                           int n_keys, void* o, long long o_img_stride, int n_img, int dt, float alpha, int cta_group,
                           int num_sms, float* part, float* ml, long long part_rows, cudaStream_t s) {
  HDRVAE_REQUIRE(n_q >= 1 && n_keys >= 1 && n_img >= 1 && k_rows >= n_keys && vt_ld >= n_keys, "attention: bad shape");
  HDRVAE_REQUIRE(dt == DT_F16 || dt == DT_BF16, "attention: 16-bit operands only");
  const int CG = cta_group == 1 ? 1 : 2;
  CUtensorMap tmQ, tmK, tmV;
  HDRVAE_TRY(map3d(&tmQ, q, dt, 512, n_q, n_img, q_ld, q_img_stride, 64, 128));
  HDRVAE_TRY(map3d(&tmK, k, dt, 512, k_rows, n_img, k_ld, k_img_stride, 64, CG == 2 ? 64 : 128));
  HDRVAE_TRY(map3d(&tmV, vt, dt, vt_ld, 512, n_img, vt_ld, vt_img_stride, 64, 128));
  AttnParams p;
  p.n_q = n_q; p.n_keys = n_keys; p.n_blocks = (n_keys + kABlockKeys - 1) / kABlockKeys;
  p.q_pairs = (n_q + 255) / 256; p.n_img = n_img;
  p.alpha_log2 = alpha * 1.4426950408889634f;
  p.o = reinterpret_cast<uint16_t*>(o); p.o_img_stride = o_img_stride; p.bf16 = dt == DT_BF16 ? 1 : 0;
  // Key splitting: see attention_key_splits().  Needs the caller's scratch (`part`: splits x rows x 512 fp32, `ml`) and a
  // dense [n_img][n_q] output; without them one unit streams all the keys.
  const long long base_units = (long long)n_img * (CG == 2 ? p.q_pairs : p.q_pairs * 2) * 2;
  (void)num_sms;
  int splits = attention_key_splits(n_keys);
  if (part == nullptr || ml == nullptr || o_img_stride != (long long)n_q * 512 || (long long)n_img * n_q * splits > part_rows) splits = 1;
  p.key_splits = splits;
  p.blocks_per_split = (p.n_blocks + splits - 1) / splits;
  p.o_part = part; p.ml_part = ml;
  static PerDeviceOnce once1, once2;
  if (CG == 2) {
    if (once2.first())
      HDRVAE_CUDA_OK(cudaFuncSetAttribute(attn_fused_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, kASmemBytes));
  } else if (once1.first()) {
    HDRVAE_CUDA_OK(cudaFuncSetAttribute(attn_fused_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, kASmemBytes));
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof cfg);
  const long long units = base_units * splits;
  cfg.gridDim = dim3((unsigned)(units * CG));
  cfg.blockDim = dim3(kAThreads);
  cfg.dynamicSmemBytes = kASmemBytes;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CG; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  if (CG == 2) HDRVAE_CUDA_OK(cudaLaunchKernelEx(&cfg, attn_fused_kernel<2>, tmQ, tmK, tmV, p));
  else HDRVAE_CUDA_OK(cudaLaunchKernelEx(&cfg, attn_fused_kernel<1>, tmQ, tmK, tmV, p));
  HDRVAE_LAUNCHED();
  HDRVAE_CUDA_OK(cudaGetLastError());
  if (splits > 1) {
    const long long rows = (long long)n_img * n_q;
    attn_merge_kernel<<<(unsigned)rows, 128, 0, s>>>(part, ml, splits, rows, reinterpret_cast<uint16_t*>(o), p.bf16);
    HDRVAE_LAUNCHED();
    HDRVAE_CUDA_OK(cudaGetLastError());
  }
  return 0;
}

}  // namespace hdrvae
