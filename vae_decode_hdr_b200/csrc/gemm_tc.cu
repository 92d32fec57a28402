// Implicit-GEMM convolution / GEMM on tcgen05 tensor cores (sm_100a).
//
// One persistent, warp-specialised kernel serves every GEMM-shaped op of the Flux AE decoder
// (ComfyUI Decoder as driven by vae.decode, reference hdr_vae_decode.py:859,:1022):
//   * 3x3 convs       : 9 taps, each tap a TMA box load of the NHWC activation tile shifted by
//                       (dy,dx); out-of-bounds rows/cols are zero-filled by TMA = the conv padding;
//   * upsample convs  : nearest-2x folded into the load: 4 output phases, each a 2x2-tap conv on the
//                       SOURCE grid with pre-summed weights (launch per phase, strided output);
//   * 1x1 convs, QK^T, PV : 1 tap.
// Operands: fp16 or bf16 (kind::f16) for normalised activations x weights, or fp32 read as tf32
// (kind::tf32) where a conv consumes the raw fp32 residual stream.  Accumulation fp32 in TMEM.
//
// Roles (384 threads): warp 0 lane 0 = TMA producer, warp 1 lane 0 = tcgen05.mma issuer, warps 2..3 idle,
// warps 4..11 = epilogue (TMEM -> registers -> scale/bias/residual -> global, + GroupNorm partial
// statistics of the output).  Two TMEM accumulator stages let the epilogue of tile i overlap the
// MMAs of tile i+1.
//
// Tile: 128 pixels (TH x TW patch) x BLOCK_N output channels, K step = one 128-byte swizzle row.
#include "common.cuh"
#pragma nv_diag_suppress 128   // "loop is not reachable": the tap-reload loops after the slab branch of an if-constexpr
#include "ptx.cuh"

namespace hdrvae {

constexpr int kBlockM = 128;
constexpr int kRowBytes = 128;                    // K extent of one stage row (64 x 16-bit or 32 x tf32)
constexpr int kABytes = kBlockM * kRowBytes;      // 16 KB
constexpr int kEpilogueThreads = 256;             // 8 warps: 2 per TMEM lane quarter, each taking half of the columns
// Warpgroup 0 = warps 0..3: TMA producer, MMA issuer, two idle warps; warpgroups 1 and 2 = the epilogue.  The register
// file is allotted per 4 warps anyway (a 320-thread CTA got the 168 registers per thread of a 384-thread one), and whole
// warpgroups let setmaxnreg move registers from the two single-thread roles to the epilogue: 64 + 2 x 216 per thread.
constexpr int kNumThreads = 128 + kEpilogueThreads;
constexpr int kRegsControl = 64, kRegsEpilogue = 216;   // 128 * 64 + 256 * 216 <= 384 * 168

constexpr int kSmemLimit = 232448;                // 227 KB opt-in shared memory per CTA on sm_100
constexpr int kSmemFixed = 8 * 4096 /*epilogue transpose patches*/ + 256 /*barriers*/ +
                           1024 /*align slack*/;

// CG = CTAs cooperating on one MMA (tcgen05 cta_group): 1, or 2 = a CTA pair computing a 256-pixel x BLOCK_N
// tile with M = 256 instructions; each CTA then stages only half of the B (weight) tile, which cuts the
// L2->SM operand traffic by a third, deepens the pipeline and halves the per-MMA issue/barrier overhead.
// SLAB > 0 (3x3 convs): the tile is 8 x 16 pixels and its activation slab is staged ONCE per K block instead of once
// per tap: one TMA box of 18 rows x 16 pixels (the 10 x 18 halo slab at a 16-line pitch) goes into a ring of
// kSlabStages buffers, the weights go into their own ring in groups of SLAB taps (9, 3 or 1: one 3-D TMA box each),
// and the 9 taps are shifted UMMA descriptors into the slab.  L2 -> SM operand traffic drops 4x and the MMA time a
// byte of shared memory keeps in flight doubles, which is what bounds the layers with <= 128 output columns.
// Pitch: the 10 pixels a tile row needs (8 + halo), not a power of two: the 128-byte swizzle is a function of the shared
// memory address bits, which TMA (writing) and the UMMA descriptors (reading, 8-row groups 10 lines apart) both honour,
// so row groups need not start on 1024-byte boundaries — only the buffers do.
constexpr int kSlabRows = 18, kSlabPitch = 10;
constexpr int kSlabBytes = kSlabRows * kSlabPitch * kRowBytes;   // 22.5 KB of TMA traffic per slab
constexpr int kSlabBufBytes = (kSlabBytes + 1023) / 1024 * 1024;
template <int BLOCK_N, int CG, int KSUB, int SLAB = 0>
struct TcConfig {
  static constexpr int kATile = kABytes;
  static constexpr int kBBytes = (SLAB ? SLAB : 1) * (BLOCK_N / CG) * kRowBytes;   // one B stage staged by this CTA
  static constexpr int kSubBytes = kATile + kBBytes;               // bytes one CTA loads per k-sub-block (tap-reload form)
  static constexpr int kStageBytes = SLAB ? kBBytes : KSUB * kSubBytes;
  static constexpr int kSlabStages = SLAB ? 3 : 0;                   // three slabs in flight cover the TMA latency
  static constexpr int kSlabBuf = kSlabBufBytes;                     // bytes of one fp16 slab buffer
  static constexpr int kPitch = kSlabPitch;                          // 128-byte lines per slab row
  static constexpr int kStagesFit = (kSmemLimit - kSmemFixed - kSlabStages * kSlabBuf) / kStageBytes;
  static constexpr int kStages = kStagesFit > 8 ? 8 : kStagesFit;
  static constexpr int kTmemCols = 2 * BLOCK_N;   // two accumulator stages (power of two: 64 ... 512)
  static constexpr int kSmemBytes = kStages * kStageBytes + kSlabStages * kSlabBuf + kSmemFixed;
  static_assert(kStages >= (SLAB ? 2 : 3) && kSmemBytes <= kSmemLimit, "shared memory plan does not fit");
  static_assert(SLAB == 0 || ((SLAB == 9 || SLAB == 3 || SLAB == 1) && KSUB == 1), "the slab variant stages 9, 3 or 1 taps of B per pipeline slot");
  static constexpr bool kFusedTensorFits = kBBytes >= kABytes && kStages >= 4;   // a ring slot holds a 16 KB centre tile
};

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {
  __half2 v = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float round_tf32(float v) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
  return __uint_as_float(r);
}

// Per GroupNorm group (CPG consecutive channels of this thread's 32-column chunk): sum and sum of squares
// over the warp's 32 pixels; lane 0 parks them in shared memory for the cross-warp sum.
template <int CPG>
__device__ __forceinline__ void emit_group_stats(const float (&f)[32], bool live, int lane, float* dst) {
#pragma unroll
  for (int g = 0; g < 32 / CPG; ++g) {
    float s = 0.f, qq = 0.f;
#pragma unroll
    for (int j = 0; j < CPG; ++j) {
      const float t = live ? f[g * CPG + j] : 0.f;
      s += t;
      qq = fmaf(t, t, qq);
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      s += __shfl_xor_sync(0xffffffffu, s, o);
      qq += __shfl_xor_sync(0xffffffffu, qq, o);
    }
    if (lane == 0) { dst[g * 2 + 0] = s; dst[g * 2 + 1] = qq; }
  }
}

// Epilogue feature sets compiled in (EPI template parameter)
enum : int {
  EPI_GENERIC = 1,   // every switch decided at run time (test entry, tf32, single-CTA builds)
  EPI_OUT16 = 2,     // 16-bit output (else fp32)
  EPI_RES = 4,       // + fp32 residual
  EPI_OUT2 = 8,      // + scaled 16-bit second output
  EPI_STATS = 16,    // + GroupNorm partial statistics
  EPI_ROWOPS = 32,   // per-row bias / per-row scale (attention GEMMs)
  EPI_LRELU = 64,    // LeakyReLU applied last (upscaler convs)
  EPI_RES2 = 128,    // + second fp32 residual (end of an RRDB: 0.04 acc + 0.2 x2 + x0)
  EPI_RES16 = 1024,  // + residual stored as a (scaled) 16-bit tensor of type res_dtype: t += res_scale * r
};

// XF builds (GroupNorm + SiLU applied to the activation slabs in place) carry two more warpgroups: 8 transform warps per
// CTA, two per scheduler (warps 2 and 3 stay idle: with them as transform warps two schedulers carried twice the load).
constexpr int kXfWarps = 8;
constexpr int kXfThreads = kNumThreads + kXfWarps * 32;  // 640
constexpr int kRegsControlXf = 64, kRegsXf = 64, kRegsEpilogueXf = 144;   // 128 x 64 + 256 x 64 + 256 x 144 = 640 x 96 (the launch allocation)

template <int BLOCK_N, bool kTf32, int CG, int EPI, int KSUB, int SLAB = 0, bool XF = false>
__global__ void __launch_bounds__(XF ? kXfThreads : kNumThreads, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmA2, const __grid_constant__ CUtensorMap tmB2, const GemmParams p) {
  using Cfg = TcConfig<BLOCK_N, CG, KSUB, SLAB>;
  constexpr int kAT = Cfg::kATile;
  const uint32_t rank = CG == 2 ? ptx::cluster_ctarank() : 0u;     // position in the CTA pair (0 = leader)
  constexpr int kStages = Cfg::kStages;
  // 32-column tiles are drained by the 4 warps that cover the 4 TMEM lane quarters; the other 4 stay idle
  constexpr int kActiveEpiWarps = BLOCK_N >= 64 ? 8 : 4;
  constexpr int kElemsPerRow = kTf32 ? 32 : 64;   // K elements per stage
  extern __shared__ uint8_t smem_raw[];
  // SWIZZLE_128B needs 1024-byte aligned stage buffers.
  // (pointer arithmetic on the __shared__ array, not an integer round trip: the compiler then knows every derived
  // pointer is shared memory and emits LDS / STS for the epilogue patches instead of generic LD / ST)
  uint8_t* smem = smem_raw + ((1024u - (ptx::smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* smem_a = smem;
  // tap-reload form: [A stages][B stages]; slab form: [B stages][slab ring]
  uint8_t* smem_b = SLAB ? smem : smem + kStages * KSUB * kAT;
  uint8_t* smem_slab = smem + kStages * Cfg::kStageBytes;
  float* stage_s = reinterpret_cast<float*>(smem_slab + Cfg::kSlabStages * Cfg::kSlabBuf);   // [8 warps][32 rows][32 floats]
  uint64_t* bars = reinterpret_cast<uint64_t*>(stage_s + 8 * 1024);
  uint64_t* full_bar = bars;                      // [kStages]
  uint64_t* empty_bar = bars + kStages;           // [kStages]
  uint64_t* tmem_full_bar = bars + 2 * kStages;   // [2]
  uint64_t* tmem_empty_bar = bars + 2 * kStages + 2;  // [2]
  uint64_t* slab_full_bar = bars + 2 * kStages + 4;   // [3]
  uint64_t* slab_empty_bar = bars + 2 * kStages + 7;  // [3]
  uint64_t* slab_ready_bar = bars + 2 * kStages + 10; // [3] fused GroupNorm: the transform warps are done with a slab
  uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 13);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    ptx::prefetch_tensormap(&tmA);
    ptx::prefetch_tensormap(&tmB);
    if (SLAB && p.k2 > 0) { ptx::prefetch_tensormap(&tmA2); ptx::prefetch_tensormap(&tmB2); }
    for (int i = 0; i < kStages; ++i) {
      ptx::mbar_init(&full_bar[i], 1);
      ptx::mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 3; ++i) {
      ptx::mbar_init(&slab_full_bar[i], 1);
      ptx::mbar_init(&slab_empty_bar[i], 1);
      ptx::mbar_init(&slab_ready_bar[i], CG * kXfWarps);    // the transform warps of every CTA of the pair
    }
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&tmem_full_bar[i], 1);
      ptx::mbar_init(&tmem_empty_bar[i], CG * kActiveEpiWarps);   // draining epilogue warps of every CTA of the pair
    }
    ptx::fence_barrier_init();
  }
  if (warp == 1) {
    if (CG == 2) ptx::tmem_alloc_pair<Cfg::kTmemCols>(tmem_ptr_s);
    else ptx::tmem_alloc<Cfg::kTmemCols>(tmem_ptr_s);
  }
  ptx::tc_fence_before_sync();
  if (CG == 2) ptx::cluster_sync_all(); else __syncthreads();
  ptx::tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_ptr_s;

  // Work items: (group of CG consecutive m-tiles, n-tile), n fastest; CTA `rank` of the pair takes m-tile
  // group*CG + rank.  An m-tile past the end is processed as an empty tile (TMA zero-fills, nothing is stored).
  const int tiles_per_img = p.tiles_x * p.tiles_y;
  const int m_tiles = p.n_img * tiles_per_img;
  const int num_tiles = ((m_tiles + CG - 1) / CG) * p.n_tiles_n;
  const int w_first = blockIdx.x / CG, w_step = gridDim.x / CG;
  const int kb_per_tap = p.k_per_tap / kElemsPerRow;
  const int num_kb = p.ntaps * kb_per_tap;
  const int kb2_blocks = SLAB ? p.k2 / kElemsPerRow : 0;      // extra K blocks from the second tensor (fused 1x1 conv)
  const int ntg = SLAB ? p.ntaps / SLAB : 0;                  // slab form: B stages per K block (taps in groups of SLAB)
  constexpr bool xf = XF && SLAB > 0;                         // GroupNorm + SiLU applied to the slabs in place

  // Producer and MMA issuer run as whole (converged) warps with one elected lane issuing: loop state and
  // addresses are then warp-uniform and stay in the uniform datapath that UTMALDG / UTCHMMA read from (a
  // single-lane loop costs ~70 cycles of register->uniform moves per MMA: measured with HDRVAE_GEMM_DBG).
  // A pipeline stage holds KSUB k-sub-blocks (128 bytes of K each), so one full/empty handshake (~380 cycles
  // of latency in the issuing thread) is amortised over 4*KSUB MMAs.
  const int num_groups = (num_kb + KSUB - 1) / KSUB;
  // (each role's code sits INSIDE the branch that changed its register budget: ptxas applies the smaller budget to
  // everything after a join of the two)
  if (warp < 4 || warp >= 12) {
  if (!XF) ptx::reg_dec<kRegsControl>();
  else if (warp < 4) ptx::reg_dec<kRegsControlXf>();
  else ptx::reg_dec<kRegsXf>();
  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    int stage = 0, ss = 0;
    uint32_t phase = 0, sphase = 0;
    // slab cursor (slab form): (work item, K block) of the next activation slab to request
    int s_tile = w_first, s_kb = 0;
    auto issue_next_slab = [&]() {
      if (s_tile >= num_tiles) return;
      const int mt = (s_tile / p.n_tiles_n) * CG + (int)rank;
      const int img = mt / tiles_per_img;                  // == n_img for the empty tile: out of bounds -> zeros
      const int rem = mt - img * tiles_per_img;
      const int ty = rem / p.tiles_x;
      const int tx = rem - ty * p.tiles_x;
      const int x0 = tx * p.TW, y0 = ty * p.TH;
      ptx::mbar_wait(&slab_empty_bar[ss], sphase ^ 1);
      if (ptx::elect_one()) {
        uint8_t* sa = smem_slab + ss * Cfg::kSlabBuf;
        // slab: rows y0-1 .. y0+16, pixels x0-1 .. x0+8 (outside the image: zero fill = the conv padding)
        if (xf) {
          // fused GroupNorm: every CTA's own barrier sees its own slab land (its transform warps wait there)
          ptx::mbar_arrive_expect_tx(&slab_full_bar[ss], (uint32_t)kSlabBytes);
          ptx::tma_load_4d(sa, &tmA, &slab_full_bar[ss], s_kb * kElemsPerRow, x0 - 1, y0 - 1 + p.y_pad, img);
        } else {
          if (rank == 0) ptx::mbar_arrive_expect_tx(&slab_full_bar[ss], (uint32_t)(CG * kSlabBytes));
          if (CG == 2) ptx::tma_load_4d_pair(sa, &tmA, &slab_full_bar[ss], s_kb * kElemsPerRow, x0 - 1, y0 - 1 + p.y_pad, img);
          else ptx::tma_load_4d(sa, &tmA, &slab_full_bar[ss], s_kb * kElemsPerRow, x0 - 1, y0 - 1 + p.y_pad, img);
        }
      }
      __syncwarp();
      if (++ss == Cfg::kSlabStages) { ss = 0; sphase ^= 1; }
      if (++s_kb == kb_per_tap) { s_kb = 0; s_tile += w_step; }
    };
    for (int tile = w_first; tile < num_tiles; tile += w_step) {
      const int nt = tile % p.n_tiles_n;
      const int mt = (tile / p.n_tiles_n) * CG + (int)rank;
      const int img = mt / tiles_per_img;                  // == n_img for the empty tile: out of bounds -> zeros
      const int rem = mt - img * tiles_per_img;
      const int ty = rem / p.tiles_x;
      const int tx = rem - ty * p.tiles_x;
      const int x0 = tx * p.TW, y0 = ty * p.TH, n0 = nt * BLOCK_N + (int)rank * (BLOCK_N / CG);
      if constexpr (SLAB > 0) {
        if (tile == w_first) issue_next_slab();             // the very first slab; afterwards always one K block ahead
        for (int kb = 0; kb < kb_per_tap; ++kb) {
          // The slab AFTER this K block's is requested before this K block's weights: the weight ring is shorter than a K
          // block's taps (7 one-tap stages for 9 taps), so in program order a slab could only be requested once the MMAs
          // of the previous one were under way — no problem while a slab is usable as it lands, but with the GroupNorm
          // transform between landing and MMAs it made the period 7 150 instead of 4 608 cycles per slab.
          issue_next_slab();
          for (int tg = 0; tg < ntg; ++tg) {
            ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
            if (ptx::elect_one()) {
              if (rank == 0) ptx::mbar_arrive_expect_tx(&full_bar[stage], (uint32_t)(CG * Cfg::kBBytes));
              uint8_t* sb = smem_b + stage * Cfg::kBBytes;
              if (CG == 2) ptx::tma_load_3d_pair(sb, &tmB, &full_bar[stage], kb * kElemsPerRow, n0, tg * SLAB);
              else ptx::tma_load_3d(sb, &tmB, &full_bar[stage], kb * kElemsPerRow, n0, tg * SLAB);
            }
            __syncwarp();
            if (++stage == kStages) { stage = 0; phase ^= 1; }
          }
        }
        // fused 1x1 conv of the second tensor: per K block the 8 x 16 centre pixels (a dense 16 KB A tile, no halo) and
        // ONE tap of its weights, each in a slot of the B-stage ring — the ring is 5 to 7 slots deep, so these short K
        // blocks (4 MMAs each) stream; through the two-slot slab ring (round-2 first version: a whole 36 KB halo slab per
        // block) the issuer waited for them longer than it computed (nin-fused 128-column conv: 2.32 M cycles against
        // 1.25 M of MMA work).
        // (128-column tiles: centre tile + weights = 16 + 8 KB share ONE slot, so a tile's 2 to 4 fused blocks are all in
        // flight while the 3x3 part still computes; 256-column tiles: two consecutive slots)
        constexpr int kB2Bytes = (BLOCK_N / CG) * kRowBytes;
        constexpr bool kOneSlot = Cfg::kBBytes >= kABytes + kB2Bytes;
        for (int kb = 0; kb < kb2_blocks; ++kb) {
          ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
          if (ptx::elect_one()) {
            if (rank == 0) ptx::mbar_arrive_expect_tx(&full_bar[stage], (uint32_t)(CG * (kABytes + (kOneSlot ? kB2Bytes : 0))));
            uint8_t* sa = smem_b + stage * Cfg::kBBytes;
            if (CG == 2) ptx::tma_load_4d_pair(sa, &tmA2, &full_bar[stage], kb * kElemsPerRow, x0, y0 + p.y_pad, img);
            else ptx::tma_load_4d(sa, &tmA2, &full_bar[stage], kb * kElemsPerRow, x0, y0 + p.y_pad, img);
            if (kOneSlot) {
              if (CG == 2) ptx::tma_load_2d_pair(sa + kABytes, &tmB2, &full_bar[stage], kb * kElemsPerRow, n0);
              else ptx::tma_load_2d(sa + kABytes, &tmB2, &full_bar[stage], kb * kElemsPerRow, n0);
            }
          }
          __syncwarp();
          if (++stage == kStages) { stage = 0; phase ^= 1; }
          if (!kOneSlot) {
            ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
            if (ptx::elect_one()) {
              if (rank == 0) ptx::mbar_arrive_expect_tx(&full_bar[stage], (uint32_t)(CG * kB2Bytes));
              uint8_t* sb = smem_b + stage * Cfg::kBBytes;
              if (CG == 2) ptx::tma_load_2d_pair(sb, &tmB2, &full_bar[stage], kb * kElemsPerRow, n0);
              else ptx::tma_load_2d(sb, &tmB2, &full_bar[stage], kb * kElemsPerRow, n0);
            }
            __syncwarp();
            if (++stage == kStages) { stage = 0; phase ^= 1; }
          }
        }
        continue;
      }
      for (int g = 0; g < num_groups; ++g) {
        ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
        const int kb0 = g * KSUB;
        const int nsub = min(KSUB, num_kb - kb0);
        if (ptx::elect_one()) {
          if (p.dbg & 1) {                                 // diagnostics: no loads, just hand the slot over
            if (rank == 0) ptx::mbar_arrive(&full_bar[stage]);
          } else {
            // the leader's barrier collects the bytes of both CTAs' loads
            if (rank == 0) ptx::mbar_arrive_expect_tx(&full_bar[stage], (uint32_t)(CG * nsub * Cfg::kSubBytes));
            for (int j = 0; j < nsub; ++j) {
              const int kbl = kb0 + j;
              const int t = kbl / kb_per_tap;
              const int kb = kbl - t * kb_per_tap;
              uint8_t* sa = smem_a + (stage * KSUB + j) * kAT;
              uint8_t* sb = smem_b + (stage * KSUB + j) * Cfg::kBBytes;
              const int xs = x0 + p.tap_dx[t], ys = y0 + p.tap_dy[t] + p.y_pad;
              if (CG == 2) {
                ptx::tma_load_4d_pair(sa, &tmA, &full_bar[stage], kb * kElemsPerRow, xs, ys, img);
                ptx::tma_load_2d_pair(sb, &tmB, &full_bar[stage], kbl * kElemsPerRow, n0);
              } else {
                ptx::tma_load_4d(sa, &tmA, &full_bar[stage], kb * kElemsPerRow, xs, ys, img);
                ptx::tma_load_2d(sb, &tmB, &full_bar[stage], kbl * kElemsPerRow, n0);
              }
            }
          }
        }
        __syncwarp();
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1 && rank == 0) {
    // ------------------------------------------------------------ MMA issuer (one warp of the leader CTA)
    const uint32_t idesc = kTf32 ? ptx::make_idesc(2u, kBlockM * CG, BLOCK_N)
                                 : ptx::make_idesc(p.ab_dtype == DT_BF16 ? 1u : 0u, kBlockM * CG, BLOCK_N);
    int stage = 0, ss = 0;
    uint32_t phase = 0, sphase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    // HDRVAE_GEMM_DBG & 32: CTA 0 reports where its issuer warp waited (cycles) — accumulator hand-back, slab, B stage
    const bool tim = (p.dbg & 32) != 0;
    long long w_acc = 0, w_slab = 0, w_b = 0, tq = 0;
    const long long t_begin = clock64();
    for (int tile = w_first; tile < num_tiles; tile += w_step) {
      if (tim) tq = clock64();
      ptx::mbar_wait(&tmem_empty_bar[acc], acc_phase ^ 1);
      if (tim) w_acc += clock64() - tq;
      ptx::tc_fence_after_sync();
      const uint32_t d_tmem = tmem_base + acc * BLOCK_N;
      if constexpr (SLAB > 0) {
        for (int kb = 0; kb < kb_per_tap; ++kb) {
          if (tim) tq = clock64();
          ptx::mbar_wait(xf ? &slab_ready_bar[ss] : &slab_full_bar[ss], sphase);
          if (tim) w_slab += clock64() - tq;
          ptx::tc_fence_after_sync();
          // descriptors are built once per slab / stage; a tap only ADDS its line offset (>> 4) to the 14-bit address field
          // (all of shared memory fits in it, so no carry leaves the field): two 64-bit uniform adds per MMA instead of a
          // shift-mask-or chain — the 32- and 64-column builds (16- and 32-cycle MMAs) are issue-bound
          const uint64_t da_slab = ptx::make_sw128_kmajor_desc_sbo(ptx::smem_u32(smem_slab + ss * Cfg::kSlabBuf), Cfg::kPitch * kRowBytes);
          for (int tg = 0; tg < ntg; ++tg) {
            if (tim) tq = clock64();
            ptx::mbar_wait(&full_bar[stage], phase);
            if (tim) w_b += clock64() - tq;
            ptx::tc_fence_after_sync();
            if (ptx::elect_one()) {
              const uint64_t db_stage = ptx::make_sw128_kmajor_desc(ptx::smem_u32(smem_b + stage * Cfg::kBBytes));
#pragma unroll
              for (int tt = 0; tt < SLAB; ++tt) {
                // tap (dy,dx): MMA row m = pixel (m>>3, m&7) of the tile reads slab line (m>>3 + 1+dy)*16 + (m&7) + 1+dx
                // (9 taps of a 3x3 conv, or the 4 taps of one output phase of an upsample conv)
                const int t = tg * SLAB + tt;
                // (tap table only in the one-tap-per-stage build, whose 128-cycle MMAs hide the lookup; the 3- and 9-tap
                // groups are 3x3 convs by construction and keep compile-time offsets: the 32-column build is issue-bound)
                const uint32_t a_off = SLAB == 1 ? (uint32_t)(((p.tap_dy[t] + 1) * Cfg::kPitch + (p.tap_dx[t] + 1)) * kRowBytes)
                                                 : (uint32_t)(((t / 3) * Cfg::kPitch + (t % 3)) * kRowBytes);
                const uint64_t da = da_slab + (a_off >> 4);
                const uint64_t db = db_stage + (uint32_t)((tt * (BLOCK_N / CG) * kRowBytes) >> 4);
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  const uint32_t accum = (kb | t | k) != 0 ? 1u : 0u;
                  if (CG == 2) ptx::umma_f16_pair(d_tmem, da + 2 * k, db + 2 * k, idesc, accum);
                  else ptx::umma_f16(d_tmem, da + 2 * k, db + 2 * k, idesc, accum);
                }
              }
              if (CG == 2) ptx::umma_commit_pair(&empty_bar[stage]); else ptx::umma_commit(&empty_bar[stage]);
              if (tg == ntg - 1) {
                if (CG == 2) ptx::umma_commit_pair(&slab_empty_bar[ss]); else ptx::umma_commit(&slab_empty_bar[ss]);
                if (kb == kb_per_tap - 1 && kb2_blocks == 0) {
                  if (CG == 2) ptx::umma_commit_pair(&tmem_full_bar[acc]); else ptx::umma_commit(&tmem_full_bar[acc]);
                }
              }
            }
            __syncwarp();
            if (++stage == kStages) { stage = 0; phase ^= 1; }
          }
          if (++ss == Cfg::kSlabStages) { ss = 0; sphase ^= 1; }
        }
        for (int kb = 0; kb < kb2_blocks; ++kb) {
          // fused 1x1 conv: the second tensor's centre tile (ring slot `sa_stage`) against one tap of its weights (next slot)
          constexpr bool kOneSlot = Cfg::kBBytes >= kABytes + (BLOCK_N / CG) * kRowBytes;
          if (tim) tq = clock64();
          ptx::mbar_wait(&full_bar[stage], phase);
          const int sa_stage = stage;
          if (!kOneSlot) {
            if (++stage == kStages) { stage = 0; phase ^= 1; }
            ptx::mbar_wait(&full_bar[stage], phase);
          }
          if (tim) w_b += clock64() - tq;
          ptx::tc_fence_after_sync();
          if (ptx::elect_one()) {
            const uint64_t da = ptx::make_sw128_kmajor_desc(ptx::smem_u32(smem_b + sa_stage * Cfg::kBBytes));
            const uint64_t db = ptx::make_sw128_kmajor_desc(ptx::smem_u32(smem_b + stage * Cfg::kBBytes + (kOneSlot ? kABytes : 0)));
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              if (CG == 2) ptx::umma_f16_pair(d_tmem, da + 2 * k, db + 2 * k, idesc, 1u);
              else ptx::umma_f16(d_tmem, da + 2 * k, db + 2 * k, idesc, 1u);
            }
            if (CG == 2) { ptx::umma_commit_pair(&empty_bar[sa_stage]); if (!kOneSlot) ptx::umma_commit_pair(&empty_bar[stage]); }
            else { ptx::umma_commit(&empty_bar[sa_stage]); if (!kOneSlot) ptx::umma_commit(&empty_bar[stage]); }
            if (kb == kb2_blocks - 1) {
              if (CG == 2) ptx::umma_commit_pair(&tmem_full_bar[acc]); else ptx::umma_commit(&tmem_full_bar[acc]);
            }
          }
          __syncwarp();
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        continue;
      }
      for (int g = 0; g < num_groups; ++g) {
        if (tim) tq = clock64();
        ptx::mbar_wait(&full_bar[stage], phase);
        if (tim) w_b += clock64() - tq;
        ptx::tc_fence_after_sync();
        const int nsub = min(KSUB, num_kb - g * KSUB);
        if (ptx::elect_one()) {
          for (int j = 0; j < nsub; ++j) {
            if (p.dbg & 2) break;                          // diagnostics: barriers only
            const uint64_t da = ptx::make_sw128_kmajor_desc(ptx::smem_u32(smem_a + (stage * KSUB + j) * kAT));
            const uint64_t db = ptx::make_sw128_kmajor_desc(ptx::smem_u32(smem_b + (stage * KSUB + j) * Cfg::kBBytes));
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              // one MMA consumes 32 bytes of K (16 x 16-bit or 8 x tf32) of the 128-byte swizzle row:
              // advance the start address by 32 B = +2 in 16-byte units
              const uint32_t accum = (g | j | k) != 0 ? 1u : 0u;
              if (CG == 2) {
                if (kTf32) ptx::umma_tf32_pair(d_tmem, da + 2 * k, db + 2 * k, idesc, accum);
                else ptx::umma_f16_pair(d_tmem, da + 2 * k, db + 2 * k, idesc, accum);
              } else {
                if (kTf32) ptx::umma_tf32(d_tmem, da + 2 * k, db + 2 * k, idesc, accum);
                else ptx::umma_f16(d_tmem, da + 2 * k, db + 2 * k, idesc, accum);
              }
            }
          }
          // frees the smem slot (in both CTAs of a pair) when these MMAs retire
          if (CG == 2) ptx::umma_commit_pair(&empty_bar[stage]); else ptx::umma_commit(&empty_bar[stage]);
          if (g == num_groups - 1) {
            if (CG == 2) ptx::umma_commit_pair(&tmem_full_bar[acc]); else ptx::umma_commit(&tmem_full_bar[acc]);
          }
        }
        __syncwarp();
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
    if (tim && blockIdx.x == 0 && lane == 0)
      printf("gemm_tc<%d,cg%d,epi%d,slab%d> issuer: %lld cycles, %d tiles x %d k-blocks; waited: accumulator %lld, slab %lld, B stage %lld\n",
             BLOCK_N, CG, EPI, SLAB, clock64() - t_begin, (num_tiles - w_first + w_step - 1) / w_step, num_kb, w_acc, w_slab, w_b);
  } else if (warp >= 12 && xf) {
    // ------------------------------------------------------------ fused GroupNorm + SiLU (warps 12..19 of every CTA)
    // A slab is 180 lines of 128 bytes = 64 channels of one halo pixel each, 16-byte chunk j of line L stored at chunk
    // j ^ (L & 7).  Thread t of the 256 owns logical chunk c = t & 7 (channels 8c .. 8c+7 of the K block: its 16 scale /
    // shift values stay in registers) of the lines L = (t >> 3) + 32 i, all of which have the same L & 7: one fixed
    // physical chunk.  Packed fp32 arithmetic (FFMA2 / FMUL2 / FADD2), the same operations in the same order as
    // gn_apply_kernel + silu_nr (groupnorm.cu), so the operand the MMAs read is bit-identical to the one the streaming
    // kernel would have written to HBM and the conv read back: 4 bytes per element of traffic less per layer.
    // Only for 256-column tiles: a slab then feeds 4 608 cycles of MMAs, the transform costs ~3 000 warp instructions;
    // behind the 1 152 cycles of a 128-column slab it cannot hide (measured with two warps: 5.1 M cycles instead of 1.0 M).
    if constexpr (xf) {
      const int tl = (warp - 12) * 32 + lane;                            // 0 .. 255
      const int c = tl & 7, lg = tl >> 3;                                // lg = 0 .. 31
      const uint32_t chunk_off = (uint32_t)((c ^ (lg & 7)) << 4);
      const int C = p.k_per_tap;
      const int y_hi = p.xf_y_hi;
      int ss = 0;
      uint32_t sphase = 0;
      const bool tim = (p.dbg & 32) != 0;                          // CTA 0, first transform warp: waiting for slabs / transforming
      long long w_land = 0, w_work = 0, tq = 0;
      for (int tile = w_first; tile < num_tiles; tile += w_step) {
        const int mt = (tile / p.n_tiles_n) * CG + (int)rank;
        const int img = mt / tiles_per_img;
        const int rem = mt - img * tiles_per_img;
        const int ty = rem / p.tiles_x;
        const int tx = rem - ty * p.tiles_x;
        const int x0 = tx * p.TW - 1, y0 = ty * p.TH - 1;          // image coordinates of slab line 0
        const bool img_ok = img < p.n_img;
        for (int kb = 0; kb < kb_per_tap; ++kb) {
          float2 a2[4], b2[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int ch = kb * kElemsPerRow + c * 8 + 2 * e;
            const bool ok = img_ok && ch + 1 < C;
            a2[e].x = ok ? __ldg(p.xf_scale + (long long)img * C + ch) * p.xf_in_scale : 0.f;
            a2[e].y = ok ? __ldg(p.xf_scale + (long long)img * C + ch + 1) * p.xf_in_scale : 0.f;
            b2[e].x = ok ? __ldg(p.xf_shift + (long long)img * C + ch) : 0.f;
            b2[e].y = ok ? __ldg(p.xf_shift + (long long)img * C + ch + 1) : 0.f;
          }
          if (tim) tq = clock64();
          ptx::mbar_wait(&slab_full_bar[ss], sphase);
          if (tim) { const long long now = clock64(); w_land += now - tq; tq = now; }
          uint8_t* base = smem_slab + ss * Cfg::kSlabBuf + chunk_off;
          int r = lg / kSlabPitch, px = lg - r * kSlabPitch;       // slab row / pixel of line L = lg + 32 i
#pragma unroll 2
          for (int L = lg; L < kSlabRows * kSlabPitch; L += 32) {
            uint4* q = reinterpret_cast<uint4*>(base + L * kRowBytes);
            const int x = x0 + px, y = y0 + r;
            const bool inside = x >= 0 && x < p.W && y >= p.xf_y_lo && y < y_hi;
            uint4 v = *q;
            __half2* h = reinterpret_cast<__half2*>(&v);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float2 o = silu_nr2(f2_fma(__half22float2(h[e]), a2[e], b2[e]));
              h[e] = __floats2half2_rn(o.x, o.y);
            }
            if (!inside) v = make_uint4(0u, 0u, 0u, 0u);
            *q = v;
            px += 32 - 3 * kSlabPitch;                             // 32 lines on = 3 rows + 2 pixels
            r += 3;
            if (px >= kSlabPitch) { px -= kSlabPitch; ++r; }
          }
          ptx::fence_proxy_async();                                // generic-proxy writes -> visible to the tensor core's reads
          __syncwarp();
          if (lane == 0) {
            // plain remote arrive, as the epilogue's accumulator hand-back: each CTA's slab is read by its OWN SM's tensor
            // core, the leader's issuer only has to learn that it is ready.  (The release.cluster form compiles to
            // MEMBAR.ALL.GPU: ncu showed 30 % of the transform warps' samples stalled on it.)
            if (CG == 2) ptx::mbar_arrive_cluster(&slab_ready_bar[ss], 0);
            else ptx::mbar_arrive(&slab_ready_bar[ss]);
          }
          if (tim) w_work += clock64() - tq;
          if (++ss == Cfg::kSlabStages) { ss = 0; sphase ^= 1; }
        }
      }
      if (tim && blockIdx.x == 0 && warp == 12 && lane == 0)
        printf("gemm_tc<%d,cg%d,epi%d,slab%d> transform warp 0: waited for slabs to land %lld cycles, transformed them in %lld\n",
               BLOCK_N, CG, EPI, SLAB, w_land, w_work);
    }
  }
  } else {
  if (XF) ptx::reg_inc<kRegsEpilogueXf>(); else ptx::reg_inc<kRegsEpilogue>();
  if ((warp - 4) < kActiveEpiWarps) {
    // ------------------------------------------------------------ epilogue (8 warps; 128 TMEM lanes x 2 column halves)
    // TMEM hands every thread one accumulator ROW (pixel).  Writing rows straight to global memory makes each
    // warp-level access touch 32 different 128-byte lines (ncu: 31 sectors/request, LSU wavefront bound), so
    // each 32x32 chunk is transposed through a 4 KB swizzled shared-memory patch: afterwards 8 lanes cover 128
    // contiguous bytes of one pixel and a warp access touches 4 lines.  Bias, residual, GroupNorm statistics
    // and the stores all happen in that coalesced layout; the residual never goes through shared memory.
    // The feature set is a template parameter (EPI): the generic build keeps every switch at run time and cost
    // ~800 instructions per chunk (ncu: issue/latency bound); the specialised builds drop to ~250.
    constexpr bool kGen = (EPI & EPI_GENERIC) != 0;
    const bool out_f32 = kGen ? (p.out_dtype == DT_F32) : ((EPI & EPI_OUT16) == 0);
    const bool has_res_f32 = kGen ? (p.residual != nullptr && p.res_dtype == DT_F32) : ((EPI & EPI_RES) != 0);
    const bool has_res_16 = kGen ? (p.residual != nullptr && p.res_dtype != DT_F32) : ((EPI & EPI_RES16) != 0);
    const bool res_bf = p.res_dtype == DT_BF16;
    const bool has_out2 = kGen ? (p.out2 != nullptr) : ((EPI & EPI_OUT2) != 0);
    const bool has_stats = kGen ? (p.stats != nullptr) : ((EPI & EPI_STATS) != 0);
    const bool row_ops = kGen ? (p.bias_per_row != 0 || p.row_scale != nullptr) : ((EPI & EPI_ROWOPS) != 0);
    const bool do_round = kGen && p.round_tf32 != 0;
    const bool has_lrelu = kGen ? (p.lrelu != 0.f) : ((EPI & EPI_LRELU) != 0);
    const bool has_res2 = kGen ? (p.residual2 != nullptr) : ((EPI & EPI_RES2) != 0);
    const float lrelu = p.lrelu, res_scale = p.res_scale;
    const int n_store = p.n_store > 0 ? p.n_store : p.n_cols;
    const int q = warp & 3;                 // TMEM lane quarter this warp may access
    const int we = warp - 4;                // 0..7
    const int half = we >> 2;               // which half of the tile's columns this warp drains
    const int cpg = p.n_cols >> 5;          // channels per GroupNorm group (stats only: 4, 8 or 16 there)
    const int cpg_log2 = cpg >= 16 ? 4 : cpg >= 8 ? 3 : 2;
    const int slots_per_group = cpg >> 2;   // 1, 2 or 4
    const int slot = lane & 7;              // 4-channel slot inside the 32-column chunk
    const int sr = lane >> 3;               // pixel sub-row 0..3 handled by this lane in each iteration
    float4* patch = reinterpret_cast<float4*>(stage_s) + we * 256;      // [32 rows][8 float4], XOR-swizzled
    constexpr int kChunksPerWarp = BLOCK_N >= 64 ? BLOCK_N / 64 : 1;
    const float alpha = p.alpha;
    const bool out16_bf = p.out_dtype == DT_BF16, out2_bf = p.out2_dtype == DT_BF16;
    const float s2 = p.out2_scale;
    const float s16 = p.out_scale != 0.f ? p.out_scale : 1.f;
    float* const outf = reinterpret_cast<float*>(p.out);
    uint16_t* const outh = reinterpret_cast<uint16_t*>(p.out);
    uint16_t* const out2h = reinterpret_cast<uint16_t*>(p.out2);
    const float* const resf = reinterpret_cast<const float*>(p.residual);
    const long long px_step = (long long)p.sx * p.out_px_stride;
    // the second output may live in a tensor with different strides (a channel slice of a concat buffer)
    const bool out2_own = p.out2_px_stride != 0;
    const long long o2_img = out2_own ? p.out2_img_stride : p.out_img_stride;
    const long long o2_row = out2_own ? p.out2_row_stride : p.out_row_stride;
    const long long o2_px = out2_own ? p.out2_px_stride : p.out_px_stride;
    const bool wide = p.tw_log2 >= 5;       // a warp's 32 pixels are consecutive in x (all but tiny images)
    // Fast path (specialised builds, tiles that lie wholly inside the image): the element offset of this lane's 4 columns
    // of pixel `it` relative to the tile origin is the same for every tile, so it is computed once per kernel; a tile
    // then costs one (warp-uniform) origin and no per-pixel address arithmetic or bounds masks.
    constexpr bool kFastBuild = !kGen && (EPI & EPI_ROWOPS) == 0;
    uint32_t lo[8], lo2[8];
#pragma unroll
    for (int it = 0; it < 8; ++it) {
      const int row = q * 32 + it * 4 + sr;
      const int yy = (row >> p.tw_log2) * p.sy, xx = (row & (p.TW - 1)) * p.sx;
      lo[it] = (uint32_t)((long long)yy * p.out_row_stride + (long long)xx * p.out_px_stride) + half * (BLOCK_N / 2) + slot * 4;
      lo2[it] = (uint32_t)((long long)yy * o2_row + (long long)xx * o2_px) + half * (BLOCK_N / 2) + slot * 4;
    }
    float4 rres_a[8];                       // residual of the chunk in hand
    int acc = 0;
    uint32_t acc_phase = 0;
    const bool tim = (p.dbg & 32) != 0;     // CTA 0, first epilogue warp: cycles waiting for accumulators / draining them
    long long w_full = 0, w_drain = 0, tq = 0;
    for (int tile = w_first; tile < num_tiles; tile += w_step) {
      const int nt = tile % p.n_tiles_n;
      const int mt = (tile / p.n_tiles_n) * CG + (int)rank;
      const bool tile_live = mt < m_tiles;                 // false: the pair's padding tile, nothing to store
      const int img = mt / tiles_per_img;
      const int rem = mt - img * tiles_per_img;
      const int ty = rem / p.tiles_x;
      const int tx = rem - ty * p.tiles_x;
      const int n0 = nt * BLOCK_N;
      const int cbase = half * (BLOCK_N / 2);
      const long long img_off = (long long)img * p.out_img_stride + n0;
      // GroupNorm partial record of this warp: one per (tile, TMEM lane quarter), [32 groups][2]
      float* const stat_rec = has_stats ? p.stats + (((long long)img * p.stats_chunks_per_img + p.stats_chunk0 + rem * 4 + q) * 32) * 2 : nullptr;

      if constexpr (kFastBuild) {
        if (tile_live && (ty + 1) * p.TH <= p.H && (tx + 1) * p.TW <= p.W && n0 + BLOCK_N <= n_store) {
          const uint32_t t_acc = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * BLOCK_N + cbase;
          const long long ty_off = (long long)(ty * p.TH * p.sy + p.py), tx_off = (long long)(tx * p.TW * p.sx + p.px);
          const long long org = img_off + ty_off * p.out_row_stride + tx_off * p.out_px_stride;
          const long long org2 = (long long)img * o2_img + n0 + ty_off * o2_row + tx_off * o2_px;
          float4 rres2[8];
          uint2 rres16[8];
          auto fetch_res = [&](long long origin, int ci, float4 (&dst)[8]) {
            if constexpr ((EPI & EPI_RES) != 0) {
              const float* r = resf + origin + ci * 32;   // plain loads: the residual may alias the output
#pragma unroll
              for (int it = 0; it < 8; ++it) dst[it] = *reinterpret_cast<const float4*>(r + lo[it]);
            }
            if constexpr ((EPI & EPI_RES16) != 0) {
              const uint16_t* r = reinterpret_cast<const uint16_t*>(p.residual) + origin + ci * 32;
#pragma unroll
              for (int it = 0; it < 8; ++it) rres16[it] = *reinterpret_cast<const uint2*>(r + lo[it]);
            }
          };
          fetch_res(org, 0, rres_a);
          if (tim) tq = clock64();
          ptx::mbar_wait(&tmem_full_bar[acc], acc_phase);
          if (tim) { const long long now = clock64(); w_full += now - tq; tq = now; }
          ptx::tc_fence_after_sync();
          uint32_t v[32];
          ptx::tmem_ld_32x32(t_acc, v);
          const float2 alpha2 = make_float2(alpha, alpha), rs2 = make_float2(res_scale, res_scale);
          const float2 s16_2 = make_float2(s16, s16), s2_2 = make_float2(s2, s2);
          // one 32 x 32 chunk: accumulator -> transpose patch -> (+ residual rr) -> global, + GroupNorm partials
          auto do_chunk = [&](const int ci, const float4 (&rr)[8]) {
            if constexpr ((EPI & EPI_RES2) != 0) {
              const float* r = p.residual2 + org + ci * 32;
#pragma unroll
              for (int it = 0; it < 8; ++it) rres2[it] = *reinterpret_cast<const float4*>(r + lo[it]);
            }
            float4 bias4 = make_float4(0.f, 0.f, 0.f, 0.f);
            if (p.bias != nullptr) bias4 = __ldg(reinterpret_cast<const float4*>(p.bias + n0 + cbase + ci * 32 + slot * 4));
            const float2 b01 = make_float2(bias4.x, bias4.y), b23 = make_float2(bias4.z, bias4.w);
            ptx::tmem_ld_wait(v);
            __syncwarp();                                 // previous chunk's readers are done with the patch
#pragma unroll
            for (int j = 0; j < 8; ++j)
              patch[lane * 8 + (j ^ (lane & 7))] = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                                                               __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
            if (ci + 1 < kChunksPerWarp) {
              ptx::tmem_ld_32x32(t_acc + (ci + 1) * 32, v);   // v has been consumed: start the next chunk's loads now
            } else {
              ptx::tc_fence_before_sync();                // the accumulator has been read out: hand it back already
            }
            __syncwarp();
            if (ci + 1 == kChunksPerWarp && lane == 0) {
              if (CG == 2) ptx::mbar_arrive_cluster(&tmem_empty_bar[acc], 0);
              else ptx::mbar_arrive(&tmem_empty_bar[acc]);
            }
            float4 a[8];
#pragma unroll
            for (int it = 0; it < 8; ++it) {
              const int rw = it * 4 + sr;
              a[it] = patch[rw * 8 + (slot ^ (rw & 7))];
            }
            float2 sum2 = make_float2(0.f, 0.f), sq2 = make_float2(0.f, 0.f);
            const long long ob = org + ci * 32, ob2 = org2 + ci * 32;
#pragma unroll
            for (int it = 0; it < 8; ++it) {
              float2 t01 = f2_fma(make_float2(a[it].x, a[it].y), alpha2, b01);
              float2 t23 = f2_fma(make_float2(a[it].z, a[it].w), alpha2, b23);
              if constexpr ((EPI & EPI_RES) != 0) {
                t01 = f2_fma(make_float2(rr[it].x, rr[it].y), rs2, t01);
                t23 = f2_fma(make_float2(rr[it].z, rr[it].w), rs2, t23);
              }
              if constexpr ((EPI & EPI_RES2) != 0) {
                t01 = f2_add(t01, make_float2(rres2[it].x, rres2[it].y));
                t23 = f2_add(t23, make_float2(rres2[it].z, rres2[it].w));
              }
              if constexpr ((EPI & EPI_RES16) != 0) {
                float2 r01, r23;
                if (res_bf) {
                  r01 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&rres16[it].x));
                  r23 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&rres16[it].y));
                } else {
                  r01 = __half22float2(*reinterpret_cast<const __half2*>(&rres16[it].x));
                  r23 = __half22float2(*reinterpret_cast<const __half2*>(&rres16[it].y));
                }
                t01 = f2_fma(r01, rs2, t01);
                t23 = f2_fma(r23, rs2, t23);
              }
              if constexpr ((EPI & EPI_LRELU) != 0) {
                t01.x = t01.x < 0.f ? t01.x * lrelu : t01.x; t01.y = t01.y < 0.f ? t01.y * lrelu : t01.y;
                t23.x = t23.x < 0.f ? t23.x * lrelu : t23.x; t23.y = t23.y < 0.f ? t23.y * lrelu : t23.y;
              }
              if constexpr ((EPI & EPI_OUT2) != 0) {
                const float2 u01 = f2_mul(t01, s2_2), u23 = f2_mul(t23, s2_2);
                uint2 o2;
                if (out2_bf) { o2.x = pack_bf16x2(u01.x, u01.y); o2.y = pack_bf16x2(u23.x, u23.y); }
                else { o2.x = pack_f16x2(u01.x, u01.y); o2.y = pack_f16x2(u23.x, u23.y); }
                *reinterpret_cast<uint2*>(out2h + ob2 + lo2[it]) = o2;
              }
              if constexpr ((EPI & EPI_OUT16) != 0) {
                const float2 u01 = f2_mul(t01, s16_2), u23 = f2_mul(t23, s16_2);
                uint2 o;
                if (out16_bf) { o.x = pack_bf16x2(u01.x, u01.y); o.y = pack_bf16x2(u23.x, u23.y); }
                else { o.x = pack_f16x2(u01.x, u01.y); o.y = pack_f16x2(u23.x, u23.y); }
                *reinterpret_cast<uint2*>(outh + ob + lo[it]) = o;
              } else {
                *reinterpret_cast<float4*>(outf + ob + lo[it]) = make_float4(t01.x, t01.y, t23.x, t23.y);
              }
              if constexpr ((EPI & EPI_STATS) != 0) {
                sum2 = f2_add(sum2, t01); sum2 = f2_add(sum2, t23);
                sq2 = f2_fma(t01, t01, sq2); sq2 = f2_fma(t23, t23, sq2);
              }
            }
            if constexpr ((EPI & EPI_STATS) != 0) {
              // this lane: (sum, sum of squares) of 4 channels x 8 pixels; fold the 4 pixel sub-rows (lanes +8, +16, +24),
              // then the slots that share a group; the group's first slot writes the warp's partial straight to its record
              float s_acc = sum2.x + sum2.y, q_acc = sq2.x + sq2.y;
              s_acc += __shfl_xor_sync(0xffffffffu, s_acc, 8);  q_acc += __shfl_xor_sync(0xffffffffu, q_acc, 8);
              s_acc += __shfl_xor_sync(0xffffffffu, s_acc, 16); q_acc += __shfl_xor_sync(0xffffffffu, q_acc, 16);
              if (cpg >= 8) { s_acc += __shfl_xor_sync(0xffffffffu, s_acc, 1); q_acc += __shfl_xor_sync(0xffffffffu, q_acc, 1); }
              if (cpg >= 16) { s_acc += __shfl_xor_sync(0xffffffffu, s_acc, 2); q_acc += __shfl_xor_sync(0xffffffffu, q_acc, 2); }
              if (lane < 8 && (slot & (slots_per_group - 1)) == 0) {
                const int gg = (n0 + cbase + ci * 32 + slot * 4) >> cpg_log2;      // group index in the layer
                if (gg < 32) *reinterpret_cast<float2*>(stat_rec + gg * 2) = make_float2(s_acc, q_acc);
              }
            }
          };
          // (Round 2 also tried requesting the residual a whole chunk — and, across tiles, a whole tile — ahead: double
          // buffers, 64 more registers.  No change: 1.449 M against 1.432 M cycles for the 128-channel in-place conv, whose
          // issuer waits for accumulators 28 % of the time.  The fp32 stream's read + write bytes pace that epilogue (4.9 of
          // the 6.55 TB/s a plain copy reaches), not its latency.)
#pragma unroll 1
          for (int ci = 0; ci < kChunksPerWarp; ++ci) {
            if (ci > 0) fetch_res(org, ci, rres_a);       // issued first: overlaps the TMEM wait and the transpose
            do_chunk(ci, rres_a);
          }
          if (tim) w_drain += clock64() - tq;
          if (++acc == 2) { acc = 0; acc_phase ^= 1; }
          continue;
        }
      }

      // coalesced-layout geometry of the 8 pixels this lane touches per chunk
      long long poff[8];
      uint32_t pmask = 0;                   // bit it: pixel it is inside the image
      int x_first = 0;                      // x of pixel it = 0 (wide case), for per-row bias / scale lookups
      if (wide) {
        const int row0 = q * 32 + sr;
        const int y = ty * p.TH + (row0 >> p.tw_log2);
        const int x = tx * p.TW + (row0 & (p.TW - 1));
        x_first = x;
        const long long o0 = img_off + (long long)(y * p.sy + p.py) * p.out_row_stride + (long long)(x * p.sx + p.px) * p.out_px_stride;
        const bool row_live = tile_live && y < p.H;
#pragma unroll
        for (int it = 0; it < 8; ++it) {
          poff[it] = o0 + it * 4 * px_step;
          if (row_live && (x + it * 4) < p.W) pmask |= 1u << it;
        }
      } else {
#pragma unroll
        for (int it = 0; it < 8; ++it) {
          const int row = q * 32 + it * 4 + sr;
          const int y = ty * p.TH + (row >> p.tw_log2);
          const int x = tx * p.TW + (row & (p.TW - 1));
          if (tile_live && y < p.H && x < p.W) pmask |= 1u << it;
          poff[it] = img_off + (long long)(y * p.sy + p.py) * p.out_row_stride + (long long)(x * p.sx + p.px) * p.out_px_stride;
        }
      }

      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * BLOCK_N;
      // Software pipeline over the warp's chunks: the TMEM load of chunk ci+1 is issued as soon as the registers of
      // chunk ci have gone to the transpose patch, so it overlaps the store phase.  ncu on the in-place-residual
      // 128 -> 128 conv (profiles/r02_ncu_conv128_residual_summary.txt): tensor pipe 50 %, DRAM 48 %, the epilogue warps
      // stall on the first use of the second chunk's residual (long scoreboard, 12 % of all samples).  Both ways of
      // fetching it earlier were measured SLOWER: issuing the next chunk's loads in the middle of a chunk (-13 %, round 1:
      // they queue behind the stores) and fetching the whole tile's residual before the accumulator wait (kPre = 2:
      // 1.55 -> 2.0 ms, round 2: 64 more live registers spill at the 168-register cap of a 320-thread CTA).
      constexpr int kPre = 1;
      float4 rres_buf[kPre][8];
      auto load_res = [&](int ci, float4 (&dst)[8]) {
        if (!has_res_f32) return;
        const int colx = cbase + ci * 32 + slot * 4;
        const uint32_t cm = (n0 + colx) < n_store ? pmask : 0u;
#pragma unroll
        for (int it = 0; it < 8; ++it)
          dst[it] = (cm >> it & 1) ? *reinterpret_cast<const float4*>(resf + poff[it] + colx)   // plain load: may alias out
                                   : make_float4(0.f, 0.f, 0.f, 0.f);
      };
      load_res(0, rres_buf[0]);
      if (kPre == 2) load_res(1, rres_buf[kPre - 1]);
      if (tim) tq = clock64();
      ptx::mbar_wait(&tmem_full_bar[acc], acc_phase);
      if (tim) { const long long now = clock64(); w_full += now - tq; tq = now; }
      ptx::tc_fence_after_sync();
      uint32_t v[32];
      ptx::tmem_ld_32x32(t_row + cbase, v);
#pragma unroll(kPre == 2 ? 2 : 1)
      for (int ci = 0; ci < kChunksPerWarp; ++ci) {
        const int c0 = cbase + ci * 32;
        const int col = c0 + slot * 4;                    // first of this lane's 4 columns (tile-relative)
        const uint32_t cmask = (n0 + col) < n_store ? pmask : 0u;   // n_cols % 32 == 0 and n_store % 4 == 0 on every call site
        float4 (&rres)[8] = rres_buf[kPre == 2 ? ci : 0];
        if (ci > 0 && kPre == 1) load_res(ci, rres);      // residual: issued first, overlaps the TMEM wait / transpose
        float4 rres2[8];
        if (has_res2) {
#pragma unroll
          for (int it = 0; it < 8; ++it)
            rres2[it] = (cmask >> it & 1) ? *reinterpret_cast<const float4*>(p.residual2 + poff[it] + col) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        float4 bias4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (!(row_ops && p.bias_per_row) && p.bias != nullptr && cmask != 0u) bias4 = __ldg(reinterpret_cast<const float4*>(p.bias + n0 + col));
        ptx::tmem_ld_wait(v);
        __syncwarp();                                     // previous chunk's readers are done with the patch
#pragma unroll
        for (int j = 0; j < 8; ++j)
          patch[lane * 8 + (j ^ (lane & 7))] = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                                                           __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
        if (ci + 1 < kChunksPerWarp) {                    // v has been consumed: start the next chunk's loads now
          ptx::tmem_ld_32x32(t_row + c0 + 32, v);
        }
        __syncwarp();
        // All 8 patch reads are issued back to back and the arithmetic is branch-free (only the stores are predicated):
        // with a branch per pixel the compiler serialised load -> use 8 times per chunk and the two epilogue warps of
        // a scheduler could not cover the latency (ncu round 2: 22 % of all stall samples on the first use of each read;
        // the 128 -> 128 convs were epilogue-paced at 72 % tensor-pipe activity while 256 -> 128 reached 92 %).
        float4 a[8];
#pragma unroll
        for (int it = 0; it < 8; ++it) {
          const int rr = it * 4 + sr;
          a[it] = patch[rr * 8 + (slot ^ (rr & 7))];
        }
        float s_acc = 0.f, q_acc = 0.f;
#pragma unroll
        for (int it = 0; it < 8; ++it) {
          const bool live = (cmask >> it & 1) != 0;
          float4 t = a[it];
          float scale = alpha;
          if (row_ops && live) {
            // per-row scale / bias (attention GEMMs); x of this pixel: rows are consecutive there (H = 1)
            const int xr = x_first + it * 4;
            if (p.row_scale != nullptr) scale *= __ldg(p.row_scale + xr);
            if (p.bias_per_row) {
              const float rb = p.bias != nullptr ? __ldg(p.bias + xr) : 0.f;
              bias4 = make_float4(rb, rb, rb, rb);
            }
          }
          t.x = fmaf(t.x, scale, bias4.x); t.y = fmaf(t.y, scale, bias4.y);
          t.z = fmaf(t.z, scale, bias4.z); t.w = fmaf(t.w, scale, bias4.w);
          if (has_res_f32) {
            t.x = fmaf(rres[it].x, res_scale, t.x); t.y = fmaf(rres[it].y, res_scale, t.y);
            t.z = fmaf(rres[it].z, res_scale, t.z); t.w = fmaf(rres[it].w, res_scale, t.w);
          }
          if (has_res2) { t.x += rres2[it].x; t.y += rres2[it].y; t.z += rres2[it].z; t.w += rres2[it].w; }
          if (has_res_16 && live) {
            // 16-bit residual (the scaled 16-bit residual stream, or the test entry); plain load: it may alias the output
            const uint2 r = *reinterpret_cast<const uint2*>(reinterpret_cast<const uint16_t*>(p.residual) + poff[it] + col);
            float2 lo, hi;
            if (p.res_dtype == DT_BF16) {
              lo = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&r.x));
              hi = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&r.y));
            } else {
              lo = __half22float2(*reinterpret_cast<const __half2*>(&r.x));
              hi = __half22float2(*reinterpret_cast<const __half2*>(&r.y));
            }
            t.x = fmaf(lo.x, res_scale, t.x); t.y = fmaf(lo.y, res_scale, t.y);
            t.z = fmaf(hi.x, res_scale, t.z); t.w = fmaf(hi.y, res_scale, t.w);
          }
          if (has_lrelu) {
            t.x = t.x < 0.f ? t.x * lrelu : t.x; t.y = t.y < 0.f ? t.y * lrelu : t.y;
            t.z = t.z < 0.f ? t.z * lrelu : t.z; t.w = t.w < 0.f ? t.w * lrelu : t.w;
          }
          if (has_out2) {
            // second, scaled 16-bit copy of the output: the tensor-core operand of a conv that consumes this
            // (un-normalised) tensor directly; the power-of-two scale keeps fp16 far from overflow
            uint2 o2;
            if (out2_bf) { o2.x = pack_bf16x2(t.x * s2, t.y * s2); o2.y = pack_bf16x2(t.z * s2, t.w * s2); }
            else { o2.x = pack_f16x2(t.x * s2, t.y * s2); o2.y = pack_f16x2(t.z * s2, t.w * s2); }
            long long off2 = poff[it];
            if (out2_own) {
              const int row = wide ? q * 32 + sr + it * 4 : q * 32 + it * 4 + sr;
              const int y2 = ty * p.TH + (row >> p.tw_log2), x2 = tx * p.TW + (row & (p.TW - 1));
              off2 = (long long)img * o2_img + n0 + (long long)(y2 * p.sy + p.py) * o2_row + (long long)(x2 * p.sx + p.px) * o2_px;
            }
            if (live) *reinterpret_cast<uint2*>(out2h + off2 + col) = o2;
          }
          if (out_f32) {
            if (do_round) { t.x = round_tf32(t.x); t.y = round_tf32(t.y); t.z = round_tf32(t.z); t.w = round_tf32(t.w); }
            if (live) *reinterpret_cast<float4*>(outf + poff[it] + col) = t;
          } else {
            uint2 o;
            if (out16_bf) { o.x = pack_bf16x2(t.x * s16, t.y * s16); o.y = pack_bf16x2(t.z * s16, t.w * s16); }
            else { o.x = pack_f16x2(t.x * s16, t.y * s16); o.y = pack_f16x2(t.z * s16, t.w * s16); }
            if (live) *reinterpret_cast<uint2*>(outh + poff[it] + col) = o;
          }
          if (has_stats) {
            const float s4 = (t.x + t.y) + (t.z + t.w);
            const float q4 = (t.x * t.x + t.y * t.y) + (t.z * t.z + t.w * t.w);
            s_acc += live ? s4 : 0.f;
            q_acc += live ? q4 : 0.f;
          }
        }
        if (has_stats) {
          // GroupNorm partials of what was just written: this lane holds (sum, sum of squares) of 4 channels x 8
          // pixels; fold the 4 pixel sub-rows (lanes +8, +16, +24), then the slots that share a group
          s_acc += __shfl_xor_sync(0xffffffffu, s_acc, 8);  q_acc += __shfl_xor_sync(0xffffffffu, q_acc, 8);
          s_acc += __shfl_xor_sync(0xffffffffu, s_acc, 16); q_acc += __shfl_xor_sync(0xffffffffu, q_acc, 16);
          if (cpg >= 8) { s_acc += __shfl_xor_sync(0xffffffffu, s_acc, 1); q_acc += __shfl_xor_sync(0xffffffffu, q_acc, 1); }
          if (cpg >= 16) { s_acc += __shfl_xor_sync(0xffffffffu, s_acc, 2); q_acc += __shfl_xor_sync(0xffffffffu, q_acc, 2); }
          if (lane < 8 && (slot & (slots_per_group - 1)) == 0 && tile_live) {
            const int gg = (n0 + c0 + slot * 4) >> cpg_log2;       // group index in the layer
            if (gg < 32) *reinterpret_cast<float2*>(stat_rec + gg * 2) = make_float2(s_acc, q_acc);
          }
        }
      }
      ptx::tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) {
        if (CG == 2) ptx::mbar_arrive_cluster(&tmem_empty_bar[acc], 0);   // the leader's MMA thread owns the accumulators
        else ptx::mbar_arrive(&tmem_empty_bar[acc]);
      }
      if (tim) w_drain += clock64() - tq;
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
    if (tim && blockIdx.x == 0 && warp == 4 && lane == 0)
      printf("gemm_tc<%d,cg%d,epi%d,slab%d> epilogue warp 0: waited for accumulators %lld cycles, drained them in %lld\n",
             BLOCK_N, CG, EPI, SLAB, w_full, w_drain);
  }
  }

  ptx::tc_fence_before_sync();
  if (CG == 2) ptx::cluster_sync_all(); else __syncthreads();    // the peer may still be read by the leader's MMAs
  if (warp == 1) {
    ptx::tc_fence_after_sync();
    if (CG == 2) ptx::tmem_dealloc_pair<Cfg::kTmemCols>(tmem_base);
    else ptx::tmem_dealloc<Cfg::kTmemCols>(tmem_base);
  }
}

// ---------------------------------------------------------------------------- host side
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                    CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                    CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode_fn() {
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

static int make_maps(const GemmParams& p, int block_n, TensorMapPair* maps, int slab = 0) {
  PFN_encodeTiled enc = get_encode_fn();
  HDRVAE_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled entry point not available");
  const int eb = dt_bytes(p.ab_dtype);
  const int vec = 16 / eb;
  const int row_elems = kRowBytes / eb;
  const CUtensorMapDataType dt = p.ab_dtype == DT_F32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                               : p.ab_dtype == DT_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  HDRVAE_REQUIRE((reinterpret_cast<uintptr_t>(p.a) & 15) == 0 && (reinterpret_cast<uintptr_t>(p.b) & 15) == 0,
                 "gemm_tc: operand pointers must be 16-byte aligned");
  HDRVAE_REQUIRE(p.a_px_stride % vec == 0 && p.a_row_stride % vec == 0 && p.a_img_stride % vec == 0 && p.b_row_stride % vec == 0,
                 "gemm_tc: strides must be multiples of 16 bytes");
  {
    // A: {C, W, H, N}; the channel extent visible to TMA is k_per_tap (columns beyond are never addressed)
    cuuint64_t dims[4] = {(cuuint64_t)(p.a_k_valid > 0 ? p.a_k_valid : p.k_per_tap), (cuuint64_t)p.W, (cuuint64_t)(p.H + 2 * p.y_pad), (cuuint64_t)p.n_img};
    cuuint64_t strides[3] = {(cuuint64_t)p.a_px_stride * eb, (cuuint64_t)p.a_row_stride * eb,
                             (cuuint64_t)p.a_img_stride * eb};
    cuuint32_t box[4] = {(cuuint32_t)row_elems, (cuuint32_t)p.TW, (cuuint32_t)p.TH, 1};
    if (slab) { box[1] = kSlabPitch; box[2] = kSlabRows; }
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = enc(&maps->a, dt, 4, const_cast<void*>(p.a), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    HDRVAE_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(A) failed: %d (W=%d H=%d N=%d K=%d)", (int)r, p.W, p.H,
                   p.n_img, p.k_per_tap);
  }
  if (slab) {
    // B as {K of one tap, Cout rows, 9 taps}: one box brings the 9 taps' [rows][64] tiles of a K block, tap-major
    cuuint64_t dims[3] = {(cuuint64_t)p.k_per_tap, (cuuint64_t)(p.b_rows > 0 ? p.b_rows : p.n_cols), (cuuint64_t)p.ntaps};
    cuuint64_t strides[2] = {(cuuint64_t)p.b_row_stride * eb, (cuuint64_t)p.k_per_tap * eb};
    cuuint32_t box[3] = {(cuuint32_t)row_elems, (cuuint32_t)block_n, (cuuint32_t)slab};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(&maps->b, dt, 3, const_cast<void*>(p.b), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    HDRVAE_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(B, slab) failed: %d (K=%d cols=%d)", (int)r, p.k_per_tap, p.n_cols);
  } else {
    cuuint64_t dims[2] = {(cuuint64_t)p.k_per_tap * p.ntaps, (cuuint64_t)(p.b_rows > 0 ? p.b_rows : p.n_cols)};
    cuuint64_t strides[1] = {(cuuint64_t)p.b_row_stride * eb};
    cuuint32_t box[2] = {(cuuint32_t)row_elems, (cuuint32_t)block_n};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(&maps->b, dt, 2, const_cast<void*>(p.b), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    HDRVAE_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(B) failed: %d (K=%d cols=%d)", (int)r,
                   p.k_per_tap * p.ntaps, p.n_cols);
  }
  memset(&maps->a2, 0, sizeof maps->a2);
  memset(&maps->b2, 0, sizeof maps->b2);
  if (p.k2 > 0) {
    HDRVAE_REQUIRE(slab && eb == 2 && p.k2 % row_elems == 0 && p.a2 != nullptr && p.b2 != nullptr,
                   "gemm_tc: the fused second tensor needs the 16-bit slab form and whole K blocks");
    HDRVAE_REQUIRE((reinterpret_cast<uintptr_t>(p.a2) & 15) == 0 && (reinterpret_cast<uintptr_t>(p.b2) & 15) == 0 &&
                   p.a2_px_stride % vec == 0 && p.a2_row_stride % vec == 0 && p.a2_img_stride % vec == 0 && p.b2_row_stride % vec == 0,
                   "gemm_tc: second-tensor pointers / strides must be 16-byte aligned");
    cuuint64_t dims[4] = {(cuuint64_t)p.k2, (cuuint64_t)p.W, (cuuint64_t)(p.H + 2 * p.y_pad), (cuuint64_t)p.n_img};
    cuuint64_t strides[3] = {(cuuint64_t)p.a2_px_stride * eb, (cuuint64_t)p.a2_row_stride * eb, (cuuint64_t)p.a2_img_stride * eb};
    cuuint32_t box[4] = {(cuuint32_t)row_elems, 8, 16, 1};      // the tile's own 8 x 16 pixels: a 1x1 conv needs no halo
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = enc(&maps->a2, dt, 4, const_cast<void*>(p.a2), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    HDRVAE_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(A2) failed: %d", (int)r);
    cuuint64_t bdims[2] = {(cuuint64_t)p.k2, (cuuint64_t)(p.b_rows > 0 ? p.b_rows : p.n_cols)};
    cuuint64_t bstrides[1] = {(cuuint64_t)p.b2_row_stride * eb};
    cuuint32_t bbox[2] = {(cuuint32_t)row_elems, (cuuint32_t)block_n};
    cuuint32_t bestr[2] = {1, 1};
    r = enc(&maps->b2, dt, 2, const_cast<void*>(p.b2), bdims, bstrides, bbox, bestr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    HDRVAE_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(B2) failed: %d", (int)r);
  }
  return 0;
}

// Chooses the pixel-patch shape (TW x TH = 128) that wastes the fewest MMA rows.
void choose_tile(int H, int W, GemmParams* p) {
  long long best = -1;
  for (int lg = 7; lg >= 0; --lg) {
    const int tw = 1 << lg, th = 128 >> lg;
    const long long cover = (long long)((W + tw - 1) / tw) * tw * ((H + th - 1) / th) * th;
    if (best < 0 || cover < best) {
      best = cover;
      p->tw_log2 = lg; p->TW = tw; p->TH = th;
    }
  }
  p->tiles_x = (W + p->TW - 1) / p->TW;
  p->tiles_y = (H + p->TH - 1) / p->TH;
}

template <int BLOCK_N, bool kTf32, int CG, int EPI, int SLAB = 0, bool XF = false>
static int launch_tc(const GemmParams& p_in, int num_sms, cudaStream_t stream) {
  // two k-sub-blocks per pipeline stage for the 128-column tiles (their MMAs are short: 64 cycles each)
  constexpr int KSUB = SLAB ? 1 : (BLOCK_N <= 128) ? 2 : 1;
  GemmParams p = p_in;
  if (p.res_scale == 0.f) p.res_scale = 1.f;
  using Cfg = TcConfig<BLOCK_N, CG, KSUB, SLAB>;
  p.dbg = switches().gemm_dbg;
  p.n_tiles_n = (p.n_cols + BLOCK_N - 1) / BLOCK_N;
  TensorMapPair maps;
  HDRVAE_TRY(make_maps(p, BLOCK_N / CG, &maps, SLAB));  // a CTA of a pair stages half of the B rows
  static PerDeviceOnce attr_once;
  if (attr_once.first())
    HDRVAE_CUDA_OK(cudaFuncSetAttribute(gemm_tc_kernel<BLOCK_N, kTf32, CG, EPI, KSUB, SLAB, XF>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        Cfg::kSmemBytes));
  const long long m_tiles = (long long)p.n_img * p.tiles_x * p.tiles_y;
  const long long work = ((m_tiles + CG - 1) / CG) * p.n_tiles_n;
  long long groups = num_sms / CG;
  if (work < groups) groups = work;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof cfg);
  cfg.gridDim = dim3((unsigned)(groups * CG));
  cfg.blockDim = dim3(XF ? kXfThreads : kNumThreads);
  cfg.dynamicSmemBytes = Cfg::kSmemBytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CG;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  HDRVAE_REQUIRE(p.k2 == 0 || (SLAB > 0 && Cfg::kFusedTensorFits), "gemm_tc: a fused second tensor needs the slab form with >= 16 KB ring slots");
  HDRVAE_REQUIRE((p.xf_scale != nullptr) == XF, "gemm_tc: fused-GroupNorm parameters and kernel build do not match");
  HDRVAE_REQUIRE(!XF || (SLAB > 0 && p.ab_dtype == DT_F16 && p.xf_shift != nullptr && p.a_k_valid == 0),
                 "gemm_tc: the fused GroupNorm needs the slab form and a dense fp16 activation tensor");
  HDRVAE_CUDA_OK(cudaLaunchKernelEx(&cfg, gemm_tc_kernel<BLOCK_N, kTf32, CG, EPI, KSUB, SLAB, XF>, maps.a, maps.b, maps.a2, maps.b2, p));
  HDRVAE_LAUNCHED();
  HDRVAE_CUDA_OK(cudaGetLastError());
  return 0;
}

int launch_gemm_tc(const GemmParams& p, int num_sms, cudaStream_t stream) {
  const int row_elems = kRowBytes / dt_bytes(p.ab_dtype);
  HDRVAE_REQUIRE(p.k_per_tap % row_elems == 0 && p.k_per_tap > 0, "gemm_tc: K per tap (%d) must be a multiple of %d",
                 p.k_per_tap, row_elems);
  HDRVAE_REQUIRE(p.n_cols % 32 == 0, "gemm_tc: output columns (%d) must be a multiple of 32", p.n_cols);
  HDRVAE_REQUIRE(p.TW * p.TH == kBlockM, "gemm_tc: tile must cover 128 pixels");
  HDRVAE_REQUIRE(!(p.bias_per_row || p.row_scale) || p.tw_log2 >= 5, "gemm_tc: per-row bias/scale needs row-major tiles");
  HDRVAE_REQUIRE(p.stats == nullptr || (p.n_cols % 128 == 0 && p.n_cols <= 512),
                 "gemm_tc: GroupNorm statistics need 128/256/512 output channels");
  HDRVAE_REQUIRE(p.stats == nullptr || (p.n_cols & (p.n_cols - 1)) == 0, "gemm_tc: GroupNorm statistics need 128/256/512 output channels");
  const bool tf32 = p.ab_dtype == DT_F32;
  const int use_cg = p.cta_group > 0 ? p.cta_group : 2;     // CTA pairs by default
  const bool n128 = p.n_cols <= 128;
  if (p.n_cols <= 64 && !tf32) {
    // narrow tiles (the upscaler's 32- and 64-channel convs): 32 / 64 accumulator columns instead of 128, so the
    // MMAs do no work on padding columns
    const bool n32 = p.n_cols <= 32;
    int epi = -1;
    if (use_cg == 2 && !p.round_tf32 && p.stats == nullptr && !p.bias_per_row && p.row_scale == nullptr &&
        (p.residual == nullptr || p.res_dtype == DT_F32)) {
      epi = (p.out_dtype != DT_F32 ? EPI_OUT16 : 0) | (p.residual ? EPI_RES : 0) | (p.residual2 ? EPI_RES2 : 0) |
            (p.out2 ? EPI_OUT2 : 0) | (p.lrelu != 0.f ? EPI_LRELU : 0);
    }
    if (p.slab) {
      HDRVAE_REQUIRE(p.ntaps == 9 && p.TW == 8 && p.TH == 16,
                     "gemm_tc: the slab variant is a 3x3 conv on 8x16-pixel tiles");
      if (use_cg == 2) {
        if (n32) {
          if (epi == (EPI_OUT16 | EPI_LRELU)) return launch_tc<32, false, 2, EPI_OUT16 | EPI_LRELU, 9>(p, num_sms, stream);
          if (epi == 0) return launch_tc<32, false, 2, 0, 9>(p, num_sms, stream);
          return launch_tc<32, false, 2, EPI_GENERIC, 9>(p, num_sms, stream);
        }
        if (epi == (EPI_OUT16 | EPI_LRELU)) return launch_tc<64, false, 2, EPI_OUT16 | EPI_LRELU, 9>(p, num_sms, stream);
        if (epi == (EPI_RES | EPI_OUT2)) return launch_tc<64, false, 2, EPI_RES | EPI_OUT2, 9>(p, num_sms, stream);
        if (epi == (EPI_RES | EPI_RES2 | EPI_OUT2)) return launch_tc<64, false, 2, EPI_RES | EPI_RES2 | EPI_OUT2, 9>(p, num_sms, stream);
        if (epi == EPI_OUT2) return launch_tc<64, false, 2, EPI_OUT2, 9>(p, num_sms, stream);
        return launch_tc<64, false, 2, EPI_GENERIC, 9>(p, num_sms, stream);
      }
      // single CTAs: 64 columns x 9 taps of B do not leave room for two slab stages; 8x16 tiles also work tap by tap
      return n32 ? launch_tc<32, false, 1, EPI_GENERIC, 9>(p, num_sms, stream)
                 : launch_tc<64, false, 1, EPI_GENERIC>(p, num_sms, stream);
    }
    if (n32) {
      if (epi == (EPI_OUT16 | EPI_LRELU)) return launch_tc<32, false, 2, EPI_OUT16 | EPI_LRELU>(p, num_sms, stream);
      if (epi == 0) return launch_tc<32, false, 2, 0>(p, num_sms, stream);
      return use_cg == 2 ? launch_tc<32, false, 2, EPI_GENERIC>(p, num_sms, stream)
                         : launch_tc<32, false, 1, EPI_GENERIC>(p, num_sms, stream);
    }
    if (epi == (EPI_OUT16 | EPI_LRELU)) return launch_tc<64, false, 2, EPI_OUT16 | EPI_LRELU>(p, num_sms, stream);
    if (epi == (EPI_RES | EPI_OUT2)) return launch_tc<64, false, 2, EPI_RES | EPI_OUT2>(p, num_sms, stream);
    if (epi == (EPI_RES | EPI_RES2 | EPI_OUT2)) return launch_tc<64, false, 2, EPI_RES | EPI_RES2 | EPI_OUT2>(p, num_sms, stream);
    if (epi == EPI_OUT2) return launch_tc<64, false, 2, EPI_OUT2>(p, num_sms, stream);
    return use_cg == 2 ? launch_tc<64, false, 2, EPI_GENERIC>(p, num_sms, stream)
                       : launch_tc<64, false, 1, EPI_GENERIC>(p, num_sms, stream);
  }
  const bool res16 = p.residual != nullptr && p.res_dtype != DT_F32;
  if (use_cg == 2 && !tf32 && p.lrelu == 0.f && p.residual2 == nullptr && (p.res_scale == 0.f || p.res_scale == 1.f || res16)) {
    // specialised epilogues for what the decoder launches; anything else takes the generic build
    int epi = 0;
    const bool simple_res = p.residual == nullptr || p.res_dtype == DT_F32;
    const bool rowops = p.bias_per_row != 0 || p.row_scale != nullptr;
    if (simple_res && !p.round_tf32) {
      if (p.out_dtype == DT_F32 && !rowops) {
        epi = (p.residual ? EPI_RES : 0) | (p.out2 ? EPI_OUT2 : 0) | (p.stats ? EPI_STATS : 0);
        if ((epi & EPI_OUT2) && !(epi & EPI_STATS)) epi = -1;        // not a decoder combination
      } else if (p.out_dtype != DT_F32 && p.residual == nullptr && p.out2 == nullptr && !(p.stats && rowops)) {
        epi = EPI_OUT16 | (rowops ? EPI_ROWOPS : 0) | (p.stats ? EPI_STATS : 0);
      } else {
        epi = -1;
      }
    } else if (res16 && !p.round_tf32 && p.out_dtype == p.res_dtype && p.out2 == nullptr && !rowops && p.stats != nullptr) {
      epi = EPI_OUT16 | EPI_RES16 | EPI_STATS;     // the scaled 16-bit residual stream, updated in place
    } else {
      epi = -1;
    }
    if (p.slab && n128 && p.ntaps == 9 && p.TW == 8 && p.TH == 16) {
      // the decoder's 128-channel 3x3 convs: slab variant, weights in groups of 3 taps
      if (epi == EPI_STATS) return launch_tc<128, false, 2, EPI_STATS, 3>(p, num_sms, stream);
      if (epi == (EPI_OUT16 | EPI_STATS)) return launch_tc<128, false, 2, EPI_OUT16 | EPI_STATS, 3>(p, num_sms, stream);
      if (epi == (EPI_RES | EPI_STATS)) return launch_tc<128, false, 2, EPI_RES | EPI_STATS, 3>(p, num_sms, stream);
      if (epi == (EPI_RES | EPI_OUT2 | EPI_STATS)) return launch_tc<128, false, 2, EPI_RES | EPI_OUT2 | EPI_STATS, 3>(p, num_sms, stream);
      if (epi == (EPI_OUT16 | EPI_RES16 | EPI_STATS)) return launch_tc<128, false, 2, EPI_OUT16 | EPI_RES16 | EPI_STATS, 3>(p, num_sms, stream);
      if (epi == 0) return launch_tc<128, false, 2, 0, 3>(p, num_sms, stream);
      if (epi == EPI_RES) return launch_tc<128, false, 2, EPI_RES, 3>(p, num_sms, stream);
    }
    if (p.slab && !n128 && p.ntaps == 4 && p.TW == 8 && p.TH == 16) {
      // one output phase of an upsample conv: 4 taps of the same halo slab (tap-reload form: L2 -> SM bound, the issuer
      // waited for operands 60 % of the time)
      if (epi == (EPI_OUT2 | EPI_STATS)) return launch_tc<256, false, 2, EPI_OUT2 | EPI_STATS, 1>(p, num_sms, stream);
      if (epi == EPI_STATS) return launch_tc<256, false, 2, EPI_STATS, 1>(p, num_sms, stream);
      if (epi == (EPI_OUT16 | EPI_STATS)) return launch_tc<256, false, 2, EPI_OUT16 | EPI_STATS, 1>(p, num_sms, stream);
      HDRVAE_REQUIRE(false, "gemm_tc: no slab build for this upsample epilogue (%d)", epi);
    }
    if (p.xf_scale != nullptr) {
      HDRVAE_REQUIRE(p.slab && !n128 && p.ntaps == 9 && p.TW == 8 && p.TH == 16 && p.k2 == 0,
                     "gemm_tc: the fused GroupNorm exists for the 256-column 3x3 slab convs");
      if (epi == (EPI_OUT16 | EPI_STATS)) return launch_tc<256, false, 2, EPI_OUT16 | EPI_STATS, 1, true>(p, num_sms, stream);
      if (epi == (EPI_OUT16 | EPI_RES16 | EPI_STATS)) return launch_tc<256, false, 2, EPI_OUT16 | EPI_RES16 | EPI_STATS, 1, true>(p, num_sms, stream);
      HDRVAE_REQUIRE(false, "gemm_tc: no fused-GroupNorm build for this epilogue (%d)", epi);
    }
    if (p.slab && !n128 && p.ntaps == 9 && p.TW == 8 && p.TH == 16) {
      // 256-column tiles: slab variant with one tap of weights per stage
      if (epi == EPI_STATS) return launch_tc<256, false, 2, EPI_STATS, 1>(p, num_sms, stream);
      if (epi == (EPI_OUT16 | EPI_STATS)) return launch_tc<256, false, 2, EPI_OUT16 | EPI_STATS, 1>(p, num_sms, stream);
      if (epi == (EPI_RES | EPI_STATS)) return launch_tc<256, false, 2, EPI_RES | EPI_STATS, 1>(p, num_sms, stream);
      if (epi == (EPI_RES | EPI_OUT2 | EPI_STATS)) return launch_tc<256, false, 2, EPI_RES | EPI_OUT2 | EPI_STATS, 1>(p, num_sms, stream);
      if (epi == (EPI_OUT16 | EPI_RES16 | EPI_STATS)) return launch_tc<256, false, 2, EPI_OUT16 | EPI_RES16 | EPI_STATS, 1>(p, num_sms, stream);
    }
#define HDRVAE_EPI_CASE(E)                                                                       \
    case E:                                                                                      \
      return n128 ? launch_tc<128, false, 2, E>(p, num_sms, stream) : launch_tc<256, false, 2, E>(p, num_sms, stream);
    switch (epi) {
      HDRVAE_EPI_CASE(0)
      HDRVAE_EPI_CASE(EPI_RES)
      HDRVAE_EPI_CASE(EPI_STATS)
      HDRVAE_EPI_CASE(EPI_RES | EPI_STATS)
      HDRVAE_EPI_CASE(EPI_OUT2 | EPI_STATS)
      HDRVAE_EPI_CASE(EPI_RES | EPI_OUT2 | EPI_STATS)
      HDRVAE_EPI_CASE(EPI_OUT16)
      HDRVAE_EPI_CASE(EPI_OUT16 | EPI_STATS)
      HDRVAE_EPI_CASE(EPI_OUT16 | EPI_ROWOPS)
      HDRVAE_EPI_CASE(EPI_OUT16 | EPI_RES16 | EPI_STATS)
      default: break;
    }
#undef HDRVAE_EPI_CASE
  }
  if (use_cg == 2) {
    if (n128) return tf32 ? launch_tc<128, true, 2, EPI_GENERIC>(p, num_sms, stream) : launch_tc<128, false, 2, EPI_GENERIC>(p, num_sms, stream);
    return tf32 ? launch_tc<256, true, 2, EPI_GENERIC>(p, num_sms, stream) : launch_tc<256, false, 2, EPI_GENERIC>(p, num_sms, stream);
  }
  if (n128) return tf32 ? launch_tc<128, true, 1, EPI_GENERIC>(p, num_sms, stream) : launch_tc<128, false, 1, EPI_GENERIC>(p, num_sms, stream);
  return tf32 ? launch_tc<256, true, 1, EPI_GENERIC>(p, num_sms, stream) : launch_tc<256, false, 1, EPI_GENERIC>(p, num_sms, stream);
}

}  // namespace hdrvae
