// C ABI of libhdrvae.so (include/hdrvae.h): context, weight repack, the decoder layer program and
// the entry points.  The layer program restates the Flux.1 AE decoder graph that the reference
// drives through vae.decode (hdr_vae_decode.py:859,:1022; graph in SURVEY.md §8 a3).
//
// Numeric plan (DESIGN.md "Precision"): tensor-core operands are 16-bit (fp16 by default, bf16 selectable)
// for everything that is normalised or bounded (GroupNorm outputs, weights, attention q/k/v/probabilities).
// The un-normalised tensors are stored in the 16-bit operand type scaled by 2^-4 on the tcgen05 kernels: the conv1
// outputs h (h_is_16bit), and with fp16 operands the residual stream x too (x_is_16bit), which the five convs that
// consume the raw stream (3 upsample convs, 2 nin_shortcuts fused into conv2) then read directly.  An fp32 x (bf16 and
// high precision, the validation kernels, HDRVAE_X16=0) comes with a scaled 16-bit copy that the producing conv's
// epilogue writes next to it for those convs (kind::tf32 on the fp32 tensor itself is also implemented in gemm_tc.cu and
// reachable through hdrvae_conv2d, at half the MMA rate).  The single-GPU and the row-tiled decode are issued by one
// layer program (Decoder below).
#include <stdarg.h>
#include <string.h>

#include <algorithm>
#include <functional>
#include <map>
#include <string>
#include <vector>

#include "engine.cuh"

namespace hdrvae {

// ---- error channel ----------------------------------------------------------------------------
static thread_local std::string g_last_error;
long long g_launch_count = 0;
void set_error(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_last_error = buf;
}

bool g_prof_on = false;
std::vector<ProfEntry> g_prof;

// ---- environment switches: the only place the library reads the environment ---------------------
const Switches& switches() {
  static const Switches sw = [] {
    auto off = [](const char* e) { return e != nullptr && atoi(e) == 0; };
    Switches w;
    w.h16 = !off(getenv("HDRVAE_H16"));
    w.x16 = !off(getenv("HDRVAE_X16"));
    w.fuse_nin = !off(getenv("HDRVAE_FUSE_NIN"));
    w.fuse_gn = !off(getenv("HDRVAE_FUSE_GN"));
    const char* no_graph = getenv("HDRVAE_NO_GRAPH");
    w.graphs = !(no_graph != nullptr && atoi(no_graph) != 0);
    const char* impl = getenv("HDRVAE_CONV_IMPL");
    w.conv_direct = impl != nullptr && strcmp(impl, "direct") == 0;
    const char* dbg = getenv("HDRVAE_GEMM_DBG");
    w.gemm_dbg = dbg != nullptr ? atoi(dbg) : 0;
    return w;
  }();
  return sw;
}

}  // namespace hdrvae

using namespace hdrvae;

namespace hdrvae {

int dev_alloc(hdrvae_ctx* ctx, size_t bytes, void** out) {
  HDRVAE_CUDA_OK(cudaMalloc(out, bytes ? bytes : 16));
  ctx->owned.push_back(*out);
  return 0;
}

// 3x3 taps in (ky,kx) row-major order; dy = ky-1, dx = kx-1
static void fill_taps_3x3(GemmParams* p) {
  p->ntaps = 9;
  for (int t = 0; t < 9; ++t) { p->tap_dy[t] = t / 3 - 1; p->tap_dx[t] = t % 3 - 1; }
}
// Upsample phase (py,px): 2x2 taps on the source grid.  Rows: py=0 -> {dy=-1: ky 0 | dy=0: ky 1,2},
// py=1 -> {dy=0: ky 0,1 | dy=+1: ky 2}; columns alike.
static void phase_taps(int py, int px, int* dy, int* dx, int* mask) {
  const int rdy[2][2] = {{-1, 0}, {0, 1}};
  const int rmask[2][2] = {{0b001, 0b110}, {0b011, 0b100}};   // bit ky (or kx)
  for (int a = 0; a < 2; ++a)
    for (int b = 0; b < 2; ++b) {
      const int t = a * 2 + b;
      dy[t] = rdy[py][a];
      dx[t] = rdy[px][b];
      int m = 0;
      for (int ky = 0; ky < 3; ++ky)
        for (int kx = 0; kx < 3; ++kx)
          if ((rmask[py][a] >> ky & 1) && (rmask[px][b] >> kx & 1)) m |= 1 << (ky * 3 + kx);
      mask[t] = m;
    }
}

int pack_conv(hdrvae_ctx* ctx, const float* w, const float* bias, int cout, int cin, int ks, bool upsample,
                     float scale, int w_dtype, PackedConv* pc, cudaStream_t s, bool split3) {
  pc->cin = cin; pc->cout = cout; pc->ks = ks; pc->upsample = upsample; pc->w_dtype = w_dtype;
  pc->kmul = split3 ? 3 : 1;
  HDRVAE_REQUIRE(!split3 || w_dtype == DT_F16, "pack_conv: the hi|hi|lo operand is fp16");
  pc->cin_pad = (cin + 63) / 64 * 64;
  pc->cout_pad = (cout + 31) / 32 * 32;
  const size_t eb = dt_bytes(w_dtype);
  if (bias != nullptr) {
    HDRVAE_TRY(dev_alloc(ctx, pc->cout_pad * sizeof(float), (void**)&pc->bias));
    HDRVAE_CUDA_OK(cudaMemsetAsync(pc->bias, 0, pc->cout_pad * sizeof(float), s));
    HDRVAE_CUDA_OK(cudaMemcpyAsync(pc->bias, bias, cout * sizeof(float), cudaMemcpyDeviceToDevice, s));
  }
  if (!upsample) {
    const int ntaps = ks * ks;
    int mask[9];
    for (int t = 0; t < ntaps; ++t) mask[t] = 1 << t;
    HDRVAE_TRY(dev_alloc(ctx, (size_t)cout * ntaps * pc->cin_pad * pc->kmul * eb, &pc->w[0]));
    HDRVAE_TRY(launch_pack_weight(w, pc->w[0], w_dtype, cout, cin, ks, ntaps, pc->cin_pad, mask, scale, s, split3 ? 1 : 0));
  } else {
    HDRVAE_REQUIRE(ks == 3, "upsample folding needs a 3x3 kernel");
    for (int ph = 0; ph < 4; ++ph) {
      int dy[4], dx[4], mask[4];
      phase_taps(ph >> 1, ph & 1, dy, dx, mask);
      HDRVAE_TRY(dev_alloc(ctx, (size_t)cout * 4 * pc->cin_pad * pc->kmul * eb, &pc->w[ph]));
      HDRVAE_TRY(launch_pack_weight(w, pc->w[ph], w_dtype, cout, cin, 3, 4, pc->cin_pad, mask, scale, s, split3 ? 1 : 0));
    }
  }
  return 0;
}

// Upper bound of the m-tiles (= GroupNorm partial chunks) a conv over an H x W image is split into: the 128-pixel
// patch choose_tile picks, or the 8 x 16 tiles of the slab variant.
// A conv writes one partial record per (m-tile, TMEM lane quarter = 32 pixels): 4 per tile (gemm_tc.cu epilogue).
constexpr int kStatRecordsPerTile = 4;
static int tiles_for(int H, int W) {
  GemmParams p;
  choose_tile(H, W, &p);
  return kStatRecordsPerTile * std::max(p.tiles_x * p.tiles_y, ((W + 7) / 8) * ((H + 15) / 16));
}


int run_conv(hdrvae_ctx* ctx, const PackedConv& pc, const ConvIO& io, int B, int H, int W, int impl,
                    cudaStream_t s) {
  if (pc.kmul == 3 && io.y2 != nullptr) {
    // "precision high": the scaled operand copy of the output is the hi|lo|hi split of the fp32 tensor (separate pass)
    HDRVAE_REQUIRE(io.y_dtype == DT_F32 && io.y_channels == 0 && io.y_pad == 0, "run_conv: split operand copy needs a dense fp32 output");
    ConvIO c = io; c.y2 = nullptr;
    HDRVAE_TRY(run_conv(ctx, pc, c, B, H, W, impl, s));
    const long long px = (long long)B * H * W * (pc.upsample ? 4 : 1);
    return launch_split3(reinterpret_cast<const float*>(io.y), pc.cout, io.y2, 3 * pc.cout, px, pc.cout, io.y2_scale, 0, s);
  }
  const int kpad = pc.cin_pad * pc.kmul;            // K per tap as the GEMM sees it
  char pname[96];
  snprintf(pname, sizeof pname, "conv%dx%d%s%s %d->%d @%dx%dx%d", pc.ks, pc.ks, pc.upsample ? "up" : "",
           pc.w_dtype == DT_F32 ? " tf32" : "", pc.cin, pc.cout, B, H, W);
  const double out_px = (double)B * H * W * (pc.upsample ? 4 : 1);
  ProfScope prof(pname, 2.0 * out_px * pc.cout * pc.cin * pc.ks * pc.ks,
                 (double)B * H * W * kpad * dt_bytes(pc.w_dtype) +
                     out_px * pc.cout * (dt_bytes(io.y_dtype) + (io.residual ? dt_bytes(io.res_dtype) : 0)), s);
  GemmParams p;
  memset(&p, 0, sizeof p);
  p.a = io.x;
  p.ab_dtype = pc.w_dtype;
  const int xch = io.x_channels > 0 ? io.x_channels : kpad;
  p.a_px_stride = xch; p.a_row_stride = (long long)W * xch;
  p.a_img_stride = (long long)(H + 2 * io.x_pad) * W * xch;
  p.a_k_valid = io.x_channels > 0 ? pc.cin : 0;
  p.y_pad = io.x_pad;
  p.n_img = B; p.H = H; p.W = W;
  p.k_per_tap = kpad;
  p.n_cols = pc.cout_pad;
  p.n_store = io.n_store > 0 ? io.n_store : (pc.cout_pad != pc.cout ? (pc.cout + 3) / 4 * 4 : 0);
  p.res_scale = io.res_scale; p.lrelu = io.lrelu; p.act_slope = io.act_slope; p.act = io.act;
  p.out_dtype = io.y_dtype;
  p.out_scale = io.y_scale;
  p.bias = io.bias != nullptr ? io.bias : pc.bias; p.bias_per_row = 0; p.res_dtype = io.res_dtype; p.alpha = io.alpha;
  p.round_tf32 = io.round_tf32 ? 1 : 0;
  p.out2_dtype = io.y2_dtype; p.out2_scale = io.y2_scale;
  p.cta_group = ctx->cta_group;
  choose_tile(H, W, &p);
  if (conv_takes_slab(pc, io, H, W, impl)) {
    p.slab = 1;
    p.tw_log2 = 3; p.TW = 8; p.TH = 16;
    p.tiles_x = (W + 7) / 8; p.tiles_y = (H + 15) / 16;
  }
  if (io.xf_scale != nullptr) {
    HDRVAE_REQUIRE(p.slab && pc.w_dtype == DT_F16 && io.x_channels == 0, "run_conv: the fused GroupNorm needs the slab form and fp16 operands");
    p.xf_scale = io.xf_scale; p.xf_shift = io.xf_shift; p.xf_in_scale = io.xf_in_scale;
    p.xf_y_lo = io.xf_y_lo; p.xf_y_hi = io.xf_y_hi < 0 ? H : io.xf_y_hi;
  }
  if (io.x2 != nullptr) {
    HDRVAE_REQUIRE(p.slab && io.pc2 != nullptr && io.pc2->ks == 1 && io.pc2->w_dtype == pc.w_dtype && io.pc2->kmul == 1 &&
                   io.pc2->cout == pc.cout, "run_conv: the fused 1x1 conv needs the slab form");
    const int c2 = io.pc2->cin_pad;
    p.a2 = io.x2; p.k2 = c2;
    p.a2_px_stride = c2; p.a2_row_stride = (long long)W * c2; p.a2_img_stride = (long long)(H + 2 * io.x_pad) * W * c2;
    p.b2 = io.pc2->w[0]; p.b2_row_stride = c2;
  }
  const int phases = pc.upsample ? 4 : 1;
  const int OH = pc.upsample ? 2 * H : H, OW = pc.upsample ? 2 * W : W;
  const int ych = io.y_channels > 0 ? io.y_channels : pc.cout;
  p.out_px_stride = ych; p.out_row_stride = (long long)OW * ych;
  p.out_img_stride = (long long)(OH + 2 * io.y_pad) * OW * ych;
  {
    // interior of the output slab(s): skip the y_pad halo rows
    const size_t skip = (size_t)io.y_pad * OW * ych + io.y_chan_off;
    p.out = reinterpret_cast<uint8_t*>(io.y) + skip * dt_bytes(io.y_dtype);
    p.residual = io.residual ? reinterpret_cast<const uint8_t*>(io.residual) + skip * dt_bytes(io.res_dtype) : nullptr;
    p.residual2 = io.residual2 ? io.residual2 + skip : nullptr;
    if (io.y2 != nullptr && io.y2_channels > 0) {
      p.out2_px_stride = io.y2_channels; p.out2_row_stride = (long long)OW * io.y2_channels;
      p.out2_img_stride = (long long)(OH + 2 * io.y_pad) * OW * io.y2_channels;
      p.out2 = reinterpret_cast<uint8_t*>(io.y2) + ((size_t)io.y_pad * OW * io.y2_channels + io.y2_chan_off) * 2;
    } else {
      p.out2 = io.y2 ? reinterpret_cast<uint8_t*>(io.y2) + skip * 2 : nullptr;
    }
  }
  const int tiles = p.tiles_x * p.tiles_y * kStatRecordsPerTile;      // GroupNorm partial records of one phase
  p.stats = io.stats;
  p.stats_chunks_per_img = phases * tiles;
  if (io.stats_chunks != nullptr) *io.stats_chunks = io.stats != nullptr ? phases * tiles : 0;
  for (int ph = 0; ph < phases; ++ph) {
    if (pc.upsample) {
      int mask[4];
      p.ntaps = 4;
      phase_taps(ph >> 1, ph & 1, p.tap_dy, p.tap_dx, mask);
      p.sy = p.sx = 2; p.py = ph >> 1; p.px = ph & 1;
    } else {
      if (pc.ks == 3) fill_taps_3x3(&p);
      else { p.ntaps = 1; p.tap_dy[0] = p.tap_dx[0] = 0; }
      p.sy = p.sx = 1; p.py = p.px = 0;
    }
    p.stats_chunk0 = ph * tiles;
    p.b = pc.w[ph];
    p.b_row_stride = (long long)p.ntaps * kpad;
    p.b_rows = pc.cout;
    if (impl == HDRVAE_CONV_DIRECT) {
      HDRVAE_REQUIRE(io.stats == nullptr, "the validation conv kernel does not emit GroupNorm statistics");
      HDRVAE_TRY(launch_gemm_direct(p, s));
    } else {
      HDRVAE_TRY(launch_gemm_tc(p, ctx->num_sms, s));
    }
  }
  return 0;
}

// Which convs take the slab form (gemm_tc.cu): every 3x3 conv of the decoder and the upscaler that is not an upsample
// conv (same-box A/B of the C2 step: 44.3 -> 43.4 ms; the chip runs at its power cap, so the 4x lower L2 -> SM operand
// traffic also buys clock).  The 128-column convs that add the residual in place were the exception in round 1 (8 x 16
// tiles: 1.76 vs 1.57 ms, their epilogue was the bound); with the round-2 epilogue the slab form wins there too
// (1.21 vs 1.44 ms).
static constexpr int kSlabMaxCols = 512;   // widest slab conv: the decoder's 512-channel convs
bool conv_takes_slab(const PackedConv& pc, const ConvIO& io, int H, int W, int impl) {
  if (pc.upsample)    // the decoder's upsample convs (256-column tiles, statistics [+ scaled operand copy] epilogues)
    return pc.ks == 3 && pc.w_dtype != DT_F32 && pc.kmul == 1 && impl == HDRVAE_CONV_TCGEN05 && H * W >= 128 &&
           pc.cout_pad >= 256 && pc.cout_pad <= kSlabMaxCols && io.residual == nullptr && io.stats != nullptr &&
           (io.y_dtype == DT_F32 || io.y2 == nullptr) && io.lrelu == 0.f && io.residual2 == nullptr;
  return pc.ks == 3 && pc.w_dtype != DT_F32 && impl != HDRVAE_CONV_DIRECT && H * W >= 128 && pc.cout_pad <= kSlabMaxCols;
}

// Plain K-major GEMM: out[M][n_cols] = row_scale[m] * alpha * A[M][K] * Bm[n_cols][K]^T (+ bias) on the same kernel.
static int run_gemm(hdrvae_ctx* ctx, int ab_dtype, const void* A, long long lda, int M, int K, const void* Bm,
                    long long ldb, int b_rows, int n_cols, void* out, long long ldo, int out_dtype, const float* bias,
                    bool bias_per_row, float alpha, const float* row_scale, int impl, cudaStream_t s) {
  GemmParams p;
  memset(&p, 0, sizeof p);
  p.a = A; p.ab_dtype = ab_dtype;
  p.a_px_stride = lda; p.a_row_stride = (long long)M * lda; p.a_img_stride = (long long)M * lda;
  p.n_img = 1; p.H = 1; p.W = M;
  p.k_per_tap = K; p.ntaps = 1;
  p.b = Bm; p.b_row_stride = ldb; p.b_rows = b_rows; p.n_cols = n_cols;
  p.out = out; p.out_dtype = out_dtype;
  p.out_px_stride = ldo; p.out_row_stride = 0; p.out_img_stride = 0;
  p.sy = p.sx = 1;
  p.bias = bias; p.bias_per_row = bias_per_row ? 1 : 0; p.alpha = alpha; p.row_scale = row_scale;
  p.cta_group = ctx->cta_group;
  p.tw_log2 = 7; p.TW = 128; p.TH = 1; p.tiles_x = (M + 127) / 128; p.tiles_y = 1;
  if (impl == HDRVAE_CONV_DIRECT) return launch_gemm_direct(p, s);
  return launch_gemm_tc(p, ctx->num_sms, s);
}

// The fused attention kernel runs with the tensor-core convs; the CUDA-core validation build takes the GEMM-level form
// (fp32 S, row soft-max kernel, P through HBM, PV GEMM) that the fused kernel replaced.
static bool attention_fused_enabled(hdrvae_ctx* ctx) { return ctx->conv_impl == HDRVAE_CONV_TCGEN05; }
static int attention_cta_group(hdrvae_ctx* ctx) { return ctx->cta_group == 1 ? 1 : 2; }

// ---- workspace plan -----------------------------------------------------------------------------
struct Plan {
  int B, h, w, T, Tp, s_rows, gn_chunks;
  size_t off_lat, off_x, off_h, off_t, off_x16, off_x16b, off_gn, off_qk, off_vt, off_o, off_f32, off_s, off_p, off_inv, off_epi, off_lat_in, off_img, total;
};
static constexpr long long kScoreBudgetElems = 1024ll << 20;  // fp32 score chunk <= 4 GiB (K and V^T are re-read once per chunk)

// Rows of one score / probability chunk of the GEMM-level attention (n_q query rows against Tp keys).
static int score_chunk_rows(int n_q, int Tp) {
  long long rows = kScoreBudgetElems / Tp;
  rows = rows / 128 * 128;
  if (rows < 128) rows = 128;
  const long long q128 = (n_q + 127) / 128 * 128;
  return (int)std::min(rows, q128);
}

// GroupNorm partial chunks per image that the decoder's convs can write for an h x w latent.
static int gn_chunk_capacity(int h, int w) {
  int chunks = 1184;
  for (int l = 1; l <= 8; l *= 2) chunks = std::max(chunks, 4 * tiles_for(l * h, l * w));
  return chunks;
}

// Workspace of a decode of B latents of h x w on this context.
static Plan decode_plan(hdrvae_ctx* ctx, int B, int h, int w) {
  Plan pl;
  const bool high = ctx->high;
  const size_t km = high ? 3 : 1;                              // hi|lo|hi operands are 3x as wide
  pl.B = B; pl.h = h; pl.w = w;
  pl.T = h * w;
  pl.Tp = (pl.T + 63) / 64 * 64;
  pl.s_rows = score_chunk_rows(pl.T, pl.Tp);
  pl.gn_chunks = gn_chunk_capacity(h, w);
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off += align_up(bytes, 1024); return o; };
  const size_t widest = (size_t)B * pl.T * 64 * 256;   // elements of [B, 8h, 8w, 256]
  pl.off_lat = take((size_t)B * pl.T * 64 * 2 * km);
  pl.off_x = take(widest * 4);       // residual stream, fp32
  pl.off_h = take(widest * 4);       // conv1 / shortcut / upsample outputs, fp32
  pl.off_t = take(widest * 2 * km);  // GroupNorm outputs: 16-bit tensor-core operands
  pl.off_x16 = take(widest / 2 * km);  // scaled 16-bit copy of x feeding an upsample conv (<= [B,4h,4w,256] elements)
  pl.off_x16b = take(widest * 2 * km); // scaled 16-bit copy of an upsample output feeding a nin_shortcut (<= [B,8h,8w,256])
  pl.off_gn = take(gn_scratch_bytes(B, 512, pl.gn_chunks));
  pl.off_qk = take((size_t)B * pl.Tp * 1024 * 2 * km);
  pl.off_vt = take((size_t)B * 512 * pl.Tp * 2 * km);
  pl.off_o = take((size_t)B * pl.T * 512 * 2 * km);
  pl.off_f32 = take(high ? (size_t)pl.Tp * 1536 * 4 + (size_t)B * 64 * pl.T * 4 : 0);   // high: fp32 q|k, v^T / o of one image; fp32 NHWC latent
  // score / probability chunks and row sums exist only for the GEMM-level attention (validation build, high precision):
  // the fused kernel keeps S and P on the SM (up to 6.1 GiB less at 4096^2).  Its key-split partials borrow off_h
  // (attend_dense).
  const bool gemm_attention = high || !attention_fused_enabled(ctx);
  pl.off_s = take(gemm_attention ? (size_t)pl.s_rows * pl.Tp * 4 : 0);
  pl.off_p = take(gemm_attention ? (size_t)pl.s_rows * pl.Tp * 2 * km : 0);
  pl.off_inv = take(gemm_attention ? (size_t)pl.s_rows * 4 : 0);          // 1 / row sum
  pl.off_epi = take(epilogue_scratch_bytes(B, 8 * h, 8 * w));
  pl.off_lat_in = take((size_t)B * ctx->c_lat * pl.T * 4);       // graph input: fp32 latent copy
  pl.off_img = take((size_t)B * 64 * pl.T * 3 * 4);        // graph output: fp32 BHWC image
  pl.total = off;
  return pl;
}

// ---- numeric plan ---------------------------------------------------------------------------------
// Un-normalised tensors that feed a conv directly (upsample convs, nin_shortcuts) are handed over as a
// 16-bit copy scaled by 2^-4: fp16 then covers |x| < 1e6 (no overflow for any sane activation) and loses
// precision only below 1e-3 (absolute error < 5e-7); the consuming conv multiplies its accumulator by 2^4.
static constexpr float kRawOperandScale = 1.0f / 16.0f;

// The block-internal tensor h = conv1(...) is never on the residual path: it is stored ONLY as the scaled 16-bit operand
// type (2 B instead of 4 written by conv1, 2 instead of 4 read by norm2; its GroupNorm statistics still come from the
// fp32 accumulators).  HDRVAE_H16=0 keeps it fp32.  Not used by the high-precision mode or the validation kernels.
static bool h_is_16bit(hdrvae_ctx* ctx) {
  return switches().h16 && !ctx->high && ctx->conv_impl == HDRVAE_CONV_TCGEN05;
}

// nin_shortcut fused into conv2 (extra K blocks of the slab conv kernel: K = 9 * Cout + Cin) instead of a separate 1x1 conv
// whose fp32 output conv2 then reads back as its residual.  HDRVAE_FUSE_NIN=0 keeps the two launches.
static bool nin_is_fused(hdrvae_ctx* ctx, const ResW& rw, int H, int W) {
  ConvIO probe;
  return switches().fuse_nin && rw.has_nin && !ctx->high && rw.nin_x16.w[0] != nullptr && conv_takes_slab(rw.c2, probe, H, W, ctx->conv_impl);
}

// The residual stream x itself is stored as fp16 scaled by 2^-4 (what the raw-stream convs read anyway): conv2 / proj_out
// read and write 2 + 2 bytes per element instead of 4 + 4 (+ 2 for the operand copy), norm1 reads 2 instead of 4, the
// upsample convs and shortcuts read x directly.  The step runs at its power cap, where bytes are what counts: same-box A/B
// 39.7 -> 36.8 ms.  Cost: one more fp16 rounding per block on the residual path (features 1.9e-3 -> 2.4e-3 rel-L2 against
// the fp32 oracle; every parity test keeps its 1e-2 bound).  HDRVAE_X16=0 keeps the fp32 stream.  Needs the fused
// shortcut and fp16 operands; not used by the bf16 and high-precision modes or the validation kernels.
static bool x_is_16bit(hdrvae_ctx* ctx) {
  return switches().x16 && switches().fuse_nin && !ctx->high && ctx->op_dtype == DT_F16 && ctx->conv_impl == HDRVAE_CONV_TCGEN05 && h_is_16bit(ctx);
}

// GroupNorm + SiLU applied inside the consuming conv (GemmParams::xf_*) instead of by the streaming kernel: for the 3x3
// slab convs whose input is a scaled fp16 tensor (x and h in the default mode).  HDRVAE_FUSE_GN=0 keeps the streaming kernel.
static bool gn_is_fused(hdrvae_ctx* ctx, const PackedConv& pc, const ConvIO& io, int x_dtype, int H, int W) {
  // (256-column tiles only: a 128-column slab's MMAs are too short to hide the transform behind, gemm_tc.cu; the fused
  // builds are CTA-pair builds)
  return switches().fuse_gn && x_is_16bit(ctx) && x_dtype == DT_F16 && pc.w_dtype == DT_F16 && pc.kmul == 1 && !pc.upsample && pc.ks == 3 &&
         pc.cout_pad >= 256 && pc.cin_pad % 64 == 0 && ctx->cta_group != 1 && io.x2 == nullptr && io.y_dtype == DT_F16 &&
         io.stats != nullptr && conv_takes_slab(pc, io, H, W, ctx->conv_impl);
}

// One chunk of the GEMM-level attention's scratch: `rows` query rows against Tp keys, fp32 scores S [rows][Tp], probabilities
// P [rows][km Tp] (km = 3 for the [hi|lo|hi] operand of the high-precision mode) and 1 / row sum [rows].
struct AttnChunk { float* S; void* P; float* inv; int rows; };
static AttnChunk plan_chunk(const Plan& pl, uint8_t* ws) {
  return {reinterpret_cast<float*>(ws + pl.off_s), ws + pl.off_p, reinterpret_cast<float*>(ws + pl.off_inv), pl.s_rows};
}

// The fused kernel (attention.cu: ONE launch, scores and probabilities never leave the SM) over n_img images: q and k
// 16-bit with row stride 1024 in a [n_img][Tp][1024] buffer (key rows >= T zero up to Tp), v^T [n_img][512][Tp], n_q query
// rows per image, o 16-bit [n_img][n_q][512].  ksplit: memory for the key-split partials ([splits][n_img n_q][512] fp32,
// then [splits][n_img n_q][2] (m, l)), needed only when T takes more than one split.
static int attention_fused(hdrvae_ctx* ctx, const uint16_t* q, const uint16_t* k, const uint16_t* vt, int n_img, int n_q,
                           int T, int Tp, void* o, float alpha, void* ksplit, size_t ksplit_bytes, cudaStream_t s) {
  const int ksp = attention_key_splits(T);
  const size_t rows = (size_t)n_img * n_q, need = (size_t)ksp * rows * (512 + 2) * 4;
  HDRVAE_REQUIRE(ksp == 1 || (ksplit != nullptr && ksplit_bytes >= need), "attention: key-split scratch too small (%zu < %zu bytes)",
                 ksplit_bytes, need);
  float* part = ksp > 1 ? reinterpret_cast<float*>(ksplit) : nullptr;
  return launch_attention_fused(q, 1024, (long long)Tp * 1024, n_q, k, 1024, (long long)Tp * 1024, Tp, vt, Tp, (long long)512 * Tp,
                                T, o, (long long)n_q * 512, n_img, ctx->op_dtype, alpha, attention_cta_group(ctx), ctx->num_sms,
                                part, part ? part + (size_t)ksp * rows * 512 : nullptr, (long long)ksp * rows, s);
}

// GEMM-level attention of n_q query rows (q, row stride ldq) against T keys (k, row stride ldk, rows >= T zero up to Tp) and
// v^T [512][ldv], in chunks of c.rows query rows: S = alpha q k^T in fp32 (the padded key columns give 0 and are masked by
// the soft-max), P = exp(S - rowmax) and inv = 1 / rowsum (launch_softmax_rows), o = inv * (P V) (o_dtype, row stride ldo).
// p_dtype is P's type: the 16-bit operand type, or DT_F16X3 for the high-precision mode, whose fp16 hi|lo operands q, k, v^T
// and P are three times as wide.
static int attention_gemm(hdrvae_ctx* ctx, const uint16_t* q, long long ldq, const uint16_t* k, long long ldk, const uint16_t* vt,
                          long long ldv, int n_q, int T, int Tp, int p_dtype, void* o, int o_dtype, long long ldo, float alpha,
                          const AttnChunk& c, cudaStream_t s) {
  const int km = p_dtype == DT_F16X3 ? 3 : 1, ab = p_dtype == DT_F16X3 ? DT_F16 : p_dtype, impl = ctx->conv_impl;
  for (int r0 = 0; r0 < n_q; r0 += c.rows) {
    const int rows = std::min(c.rows, n_q - r0);
    HDRVAE_TRY(run_gemm(ctx, ab, q + (size_t)r0 * ldq, ldq, rows, 512 * km, k, ldk, Tp, Tp, c.S, Tp, DT_F32, nullptr, false,
                        alpha, nullptr, impl, s));
    HDRVAE_TRY(launch_softmax_rows(c.S, c.P, p_dtype, c.inv, rows, T, Tp, Tp, (long long)km * Tp, s));
    HDRVAE_TRY(run_gemm(ctx, ab, c.P, (long long)km * Tp, rows, km * Tp, vt, ldv, 512, 512,
                        reinterpret_cast<uint8_t*>(o) + (size_t)r0 * ldo * dt_bytes(o_dtype), ldo, o_dtype, nullptr, false, 1.0f,
                        c.inv, impl, s));
  }
  return 0;
}

// Epilogue phase A on the decoder's features (slab start `feat`, `pad` halo rows above / below each image's H rows).
// fp16 operands: conv_out runs on the tensor cores into `conv8` (dense [B][H][W][8] fp32 scratch), then one streaming
// pass does the MAX-pool and the statistics; otherwise (bf16 operands, validation kernel) the all-in-one CUDA-core kernel.
static int run_phase_a(hdrvae_ctx* ctx, const void* feat, int B, int H, int W, int pad, float* conv8, void* epi, cudaStream_t s) {
  const long long img_stride = (long long)(H + 2 * pad) * W * 128;
  if (ctx->high)     // fp32 features: conv_out in fp32 on the CUDA cores (the 1e-5 parity kernel)
    return launch_epilogue_phase_a(feat, DT_F32, B, H, W, ctx->conv_out_w, ctx->conv_out_b, nullptr, epi, s, 0, img_stride);
  const uint16_t* interior = reinterpret_cast<const uint16_t*>(feat) + (size_t)pad * W * 128;
  if (ctx->op_dtype == DT_F16 && ctx->conv_impl == HDRVAE_CONV_TCGEN05 && ctx->conv_out_tc.w[0] != nullptr) {
    ConvIO io; io.x = feat; io.x_pad = pad; io.y = conv8; io.y_dtype = DT_F32; io.y_channels = 8; io.n_store = 8;
    HDRVAE_TRY(run_conv(ctx, ctx->conv_out_tc, io, B, H, W, HDRVAE_CONV_TCGEN05, s));
    return launch_epilogue_phase_a_pre(interior, ctx->op_dtype, B, H, W, conv8, ctx->conv_out_b, nullptr, epi, s, img_stride);
  }
  return launch_epilogue_phase_a(interior, ctx->op_dtype, B, H, W, ctx->conv_out_w, ctx->conv_out_b, nullptr, epi, s, pad, img_stride);
}

// "precision high" attention of ONE image: every GEMM on K-concatenated fp16 hi / lo operands (activations [hi|lo|hi],
// weight-like operands [hi|hi|lo]), fp32 scores and outputs.  t3: GroupNorm output [T][1536]; o3: [T][1536] operand of
// proj_out.  The projections run in fp32 and are split into the operands of the GEMM-level form (the fused kernel keeps a
// 16-bit Q tile resident and has no room for a second copy), whose fp32 output is split once more for proj_out.
static int run_attention_high(hdrvae_ctx* ctx, const Plan& pl, uint8_t* ws, const uint16_t* t3, uint16_t* o3, cudaStream_t s) {
  const int impl = ctx->conv_impl, T = pl.T, Tp = pl.Tp;
  float* f32 = reinterpret_cast<float*>(ws + pl.off_f32);                 // [Tp][1024] q|k, then [512][Tp] v^T, then [T][512] o
  uint16_t* q3 = reinterpret_cast<uint16_t*>(ws + pl.off_qk);            // [Tp][1536] hi|lo|hi
  uint16_t* k3 = q3 + (size_t)Tp * 1536;                                 // [Tp][1536] hi|hi|lo
  uint16_t* vt3 = reinterpret_cast<uint16_t*>(ws + pl.off_vt);           // [512][3 Tp] hi|hi|lo along the keys
  if (Tp != T) HDRVAE_CUDA_OK(cudaMemsetAsync(f32, 0, (size_t)Tp * 1024 * 4, s));
  HDRVAE_TRY(run_gemm(ctx, DT_F16, t3, 1536, T, 1536, ctx->qk.w[0], 1536, 1024, 1024, f32, 1024, DT_F32, ctx->qk.bias, false, 1.0f,
                      nullptr, impl, s));
  HDRVAE_TRY(launch_split3(f32, 1024, q3, 1536, Tp, 512, 1.f, 0, s));
  HDRVAE_TRY(launch_split3(f32 + 512, 1024, k3, 1536, Tp, 512, 1.f, 1, s));
  // v^T = Wv t^T + bv: the weights are the A operand here ([hi|hi|lo] against the activations' [hi|lo|hi]: same 3 terms)
  HDRVAE_TRY(run_gemm(ctx, DT_F16, ctx->vproj.w[0], 1536, 512, 1536, t3, 1536, T, Tp, f32, Tp, DT_F32, ctx->vproj.bias, true, 1.0f,
                      nullptr, impl, s));
  HDRVAE_TRY(launch_split3(f32, Tp, vt3, 3ll * Tp, 512, Tp, 1.f, 1, s));
  float* of = f32;                                                       // [T][512], v^T fp32 is dead after the split
  HDRVAE_TRY(attention_gemm(ctx, q3, 1536, k3, 1536, vt3, 3ll * Tp, T, T, Tp, DT_F16X3, of, DT_F32, 512, 1.0f, plan_chunk(pl, ws), s));
  return launch_split3(of, 512, o3, 1536, T, 512, 1.f, 0, s);
}

// Attention core of B images: q|k [B][Tp][1024], v^T [B][512][Tp] -> o 16-bit [B][T][512].  The fused kernel takes all
// images in one launch (ksplit: idle memory for its key-split partials); the validation build runs the GEMM-level form one
// image at a time in the scratch chunk c.
static int run_attention_core(hdrvae_ctx* ctx, int B, int T, int Tp, const void* qk, const void* vt, void* o, float qk_alpha,
                              void* ksplit, size_t ksplit_bytes, const AttnChunk& c, cudaStream_t s) {
  const uint16_t* q = reinterpret_cast<const uint16_t*>(qk);
  const uint16_t* v = reinterpret_cast<const uint16_t*>(vt);
  if (attention_fused_enabled(ctx)) {
    ProfScope prof("attention fused kernel", 4.0 * B * (double)T * T * 512, 0.0, s);
    return attention_fused(ctx, q, q + 512, v, B, T, T, Tp, o, qk_alpha, ksplit, ksplit_bytes, s);
  }
  for (int b = 0; b < B; ++b) {
    const uint16_t* qb = q + (size_t)b * Tp * 1024;
    HDRVAE_TRY(attention_gemm(ctx, qb, 1024, qb + 512, 1024, v + (size_t)b * 512 * Tp, Tp, T, T, Tp, ctx->op_dtype,
                              reinterpret_cast<uint16_t*>(o) + (size_t)b * T * 512, ctx->op_dtype, 512, qk_alpha, c, s));
  }
  return 0;
}

static int check_ws(const Plan& pl, void* ws, size_t bytes) {
  HDRVAE_REQUIRE(ws != nullptr && bytes >= pl.total, "hdrvae: workspace too small (%zu < %zu bytes)", bytes, pl.total);
  // every plan offset is a multiple of 1024; TMA and the vector loads need 16 bytes, cudaMalloc gives 256 and torch's
  // caching allocator 512 (a 1024-byte demand made small workspaces fail depending on the allocator's history)
  HDRVAE_REQUIRE((reinterpret_cast<uintptr_t>(ws) & 255) == 0, "hdrvae: workspace must be 256-byte aligned");
  return 0;
}


// =================================================================================================== row tiling
// Step machine of the row-tiled decode (one image, latent rows split over `world` ranks).  Every activation
// lives in a slab with one halo row above and below; conv outputs get their halo rows from the neighbours
// (HALO exchange), GroupNorm sums are all-reduced, attention K/V are all-gathered.  See include/hdrvae.h.
struct RowsPlan {
  int h, w, hl, world, T, Tl, Tp, gn_chunks;
  size_t off_lat, off_x, off_h, off_t, off_xa, off_xb, off_gn, off_qk, off_v, off_vt, off_o, off_epi, off_mail, total;
};

static RowsPlan make_rows_plan(int h, int w, int world) {
  RowsPlan pl;
  pl.h = h; pl.w = w; pl.world = world; pl.hl = h / world;
  pl.T = h * w; pl.Tl = pl.hl * w;
  pl.Tp = (pl.T + 63) / 64 * 64;
  pl.gn_chunks = gn_chunk_capacity(pl.hl, w);
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off += align_up(bytes, 1024); return o; };
  const size_t widest = (size_t)(8 * pl.hl + 2) * 8 * w * 256;           // slab elements incl. halo rows
  size_t xa = std::max((size_t)(pl.hl + 2) * w * 512, std::max((size_t)(2 * pl.hl + 2) * 2 * w * 512,
                                                               (size_t)(4 * pl.hl + 2) * 4 * w * 256));
  pl.off_lat = take((size_t)(pl.hl + 2) * w * 64 * 2);
  pl.off_x = take(widest * 4);
  pl.off_h = take(widest * 4);
  pl.off_t = take(widest * 2);
  pl.off_xa = take(xa * 2);
  pl.off_xb = take(widest * 2);
  pl.off_gn = take(gn_scratch_bytes(1, 512, pl.gn_chunks));
  pl.off_qk = take((size_t)pl.Tp * 1024 * 2);          // gathered [T][q|k]
  pl.off_v = take((size_t)pl.Tp * 512 * 2);            // gathered v [T][512]
  pl.off_vt = take((size_t)512 * pl.Tp * 2);
  pl.off_o = take((size_t)pl.Tl * 512 * 2);
  pl.off_epi = take(epilogue_scratch_bytes(1, 8 * pl.hl, 8 * w));
  pl.off_mail = take(sizeof(RowsMailbox));              // flags / tables of the device-driven exchanges (rows_p2p.cu)
  pl.total = off;
  return pl;
}

}  // namespace hdrvae

struct hdrvae_rows {
  hdrvae_ctx* ctx = nullptr;
  RowsPlan pl;
  int rank = 0, mode = 0;
  float factor = 1.f, ev = 1.f;
  uint8_t* ws = nullptr;
  const float* latent = nullptr;
  float* out = nullptr;
  struct Op { bool exchange; std::function<int(cudaStream_t)> fn; hdrvae_exchange ex; };
  std::vector<Op> ops;
  size_t pc = 0;
  int pending = 0;          // GroupNorm partial chunks of the last conv, written and read while the ops run
  // every rank's workspace as mapped into this process (hdrvae_peer_open; own pointer at [rank]): hdrvae_rows_set_peers
  uint8_t* peers[kRowsMaxRanks] = {};
  bool peers_set = false;
};

namespace hdrvae {

static void rows_exchange(hdrvae_rows* st, const hdrvae_exchange& ex) {
  hdrvae_rows::Op op; op.exchange = true; op.ex = ex;
  st->ops.push_back(std::move(op));
}
static size_t ws_off(hdrvae_rows* st, const void* p) { return reinterpret_cast<const uint8_t*>(p) - st->ws; }

// halo descriptor of a slab [H+2][W][C] with element size eb
static void add_halo(hdrvae_rows* st, hdrvae_exchange* ex, const void* slab, int H, int W, int C, int eb) {
  const int i = ex->n_halo++;
  const size_t row = (size_t)W * C * eb;
  const size_t base = ws_off(st, slab);
  ex->kind |= HDRVAE_EX_HALO;
  ex->halo_row_bytes[i] = row;
  ex->halo_top_off[i] = base;
  ex->halo_first_row_off[i] = base + row;
  ex->halo_last_row_off[i] = base + (size_t)H * row;
  ex->halo_bottom_off[i] = base + (size_t)(H + 1) * row;
}

// zero the halo rows that lie outside the image (true conv padding) of a 16-bit operand slab
static int zero_border_halos(hdrvae_rows* st, void* slab, int H, int W, int C, int eb, cudaStream_t s) {
  const size_t row = (size_t)W * C * eb;
  if (st->rank == 0) HDRVAE_CUDA_OK(cudaMemsetAsync(slab, 0, row, s));
  if (st->rank == st->pl.world - 1) HDRVAE_CUDA_OK(cudaMemsetAsync(reinterpret_cast<uint8_t*>(slab) + (size_t)(H + 1) * row, 0, row, s));
  return 0;
}

// ---- decoder layer program ----------------------------------------------------------------------------------------
// The decoder graph is written once and issued against a Decoder, which says where the tensors live and how a step is
// issued: the single-GPU decode launches each step for B dense images as it is issued; the row-tiled decode (rows set)
// records the steps of one image, stored as slabs with one halo row above and below, into hdrvae_rows::ops together
// with the exchanges between them.  Only step, norm and conv depend on the target; the storage decisions of the numeric
// plan are made here once for both.
struct Decoder {
  hdrvae_ctx* ctx;
  hdrvae_rows* rows;     // null: single-GPU decode
  cudaStream_t s;        // single-GPU decode: the stream the steps are launched on
  int B;                 // images
  int pad;               // halo rows stored above and below each image: 0 dense, 1 slab
  void* lat;             // staged latent: conv_in's operand
  float* x;              // residual stream (stored as x_dt)
  float* hbuf;           // block-internal tensor h (stored as h_dt); also the stream's second buffer
  void* t;               // GroupNorm outputs: 16-bit operand buffer
  void* xa16;            // scaled 16-bit copy of a level's last ResBlock output = operand of the level's upsample conv
  void* xb16;            // scaled 16-bit copy of an upsample conv's output = operand of the next block's nin_shortcut
  void* gn;              // GroupNorm scratch (partials | scale | shift | sums)
  int gn_chunks;         // capacity of the partial area (chunks per image)
  int* pending;          // partial chunks per image valid for the tensor about to be normalised (read when a step runs)
  int x_dt, h_dt;        // element types of x and h: fp32, or the operand type holding the value times x_scale / h_scale
  float x_scale, h_scale;
};

static Decoder make_decoder(hdrvae_ctx* ctx, hdrvae_rows* rows, cudaStream_t s, int B, int* pending) {
  Decoder d;
  memset(&d, 0, sizeof d);
  d.ctx = ctx; d.rows = rows; d.s = s; d.B = B; d.pad = rows != nullptr ? 1 : 0; d.pending = pending;
  const bool x16 = x_is_16bit(ctx), h16 = h_is_16bit(ctx);
  d.x_dt = x16 ? ctx->op_dtype : DT_F32; d.x_scale = x16 ? kRawOperandScale : 1.f;
  d.h_dt = h16 ? ctx->op_dtype : DT_F32; d.h_scale = h16 ? kRawOperandScale : 1.f;
  return d;
}

// Runs fn now (single-GPU) or appends it to the row-tiled program, which runs it from hdrvae_rows_run: steps capture by
// value what they read.
static int step(Decoder& d, std::function<int(cudaStream_t)> fn) {
  if (d.rows == nullptr) return fn(d.s);
  hdrvae_rows::Op op; op.exchange = false; op.fn = std::move(fn); memset(&op.ex, 0, sizeof op.ex);
  d.rows->ops.push_back(std::move(op));
  return 0;
}

// t = [SiLU](GroupNorm(x)), x stored as x_dt holding the value times x_scale; y_dt: element type of t (-1: operand type).
// Single-GPU: the streaming kernel on the producing conv's partials.  Row tiling: from the all-reduced sums, over the whole
// slab (halo rows included: GroupNorm is elementwise once the global statistics are known), then the zero padding at the
// image borders is restored.
static int norm(Decoder& d, const void* x, int x_dt, float x_scale, const NormW& nw, bool silu, int H, int W, int y_dt = -1) {
  const int ydt = y_dt >= 0 ? y_dt : (d.ctx->high ? DT_F16X3 : d.ctx->op_dtype);
  if (d.rows == nullptr) {
    char pname[64];
    snprintf(pname, sizeof pname, "groupnorm%s C=%d @%dx%d", silu ? "+silu" : "", nw.C, d.B, H * W);
    ProfScope prof(pname, 0.0, (double)d.B * H * W * nw.C * (dt_bytes(x_dt) * (*d.pending > 0 ? 1 : 2) + 2.0), d.s);
    const int partials = *d.pending;
    *d.pending = 0;
    return launch_groupnorm(x, x_dt, d.t, ydt, d.B, H * W, nw.C, nw.gamma, nw.beta, silu, d.gn, d.gn_chunks, partials, d.s,
                            1.f / x_scale);
  }
  const NormW n = nw;
  const double count = (double)H * d.rows->pl.world * (double)W * (double)(n.C / 32);
  return step(d, [=](cudaStream_t s) {
    const long long slab = (long long)(H + 2) * W * n.C;
    HDRVAE_TRY(launch_gn_apply_from_sums(x, x_dt, slab, d.t, ydt, slab, 1, (H + 2) * W, n.C, n.gamma, n.beta, silu, d.gn,
                                         d.gn_chunks, count, s, 1.f / x_scale));
    return zero_border_halos(d.rows, d.t, H, W, n.C, 2, s);
  });
}

static float* stats_ptr(const Decoder& d) {
  return d.ctx->conv_impl == HDRVAE_CONV_TCGEN05 ? reinterpret_cast<float*>(d.gn) : nullptr;
}

// conv flags
constexpr int kNoStats = 1;      // no GroupNorm statistics (the separate nin_shortcut: its output is conv2's residual)
constexpr int kZeroHalos = 2;    // row tiling: y is the 16-bit stream, read raw by later 3x3 convs: zero its border halo rows
constexpr int kDenseInput = 4;   // x is dense, not a slab (proj_out reads the attention output)

// Issues run_conv with the target's halo rows and the GroupNorm statistics of y.  xf: GroupNorm + SiLU of io.x applied
// inside the conv (norm_conv), its scale / shift computed right before the conv.  Row tiling, after a conv with
// statistics: fold this rank's partials, then one exchange all-reduces the sums and fills the halo rows of y and of its
// scaled copy in xa16 (the upsample conv's 3x3 operand).
static int conv(Decoder& d, const PackedConv& pc, ConvIO io, int H, int W, int flags = 0, const NormW* xf = nullptr) {
  hdrvae_rows* rows = d.rows;
  io.x_pad = (flags & kDenseInput) ? 0 : d.pad;
  io.y_pad = d.pad;
  if (!(flags & kNoStats)) { io.stats = stats_ptr(d); io.stats_chunks = d.pending; }
  if (xf != nullptr && rows != nullptr) {     // a border rank's outer halo row is padding, not an image row
    io.xf_y_lo = rows->rank == 0 ? 0 : -1;
    io.xf_y_hi = rows->rank == rows->pl.world - 1 ? H : H + 1;
  }
  const int OH = pc.upsample ? 2 * H : H, OW = pc.upsample ? 2 * W : W;
  const PackedConv* p = &pc;
  const bool zero_y = rows != nullptr && (flags & kZeroHalos);
  const bool xa_copy = rows != nullptr && io.y2 != nullptr && io.y2 == d.xa16;
  HDRVAE_TRY(step(d, [=](cudaStream_t s) mutable {
    if (xf != nullptr && rows == nullptr) {
      // only the reduction of the producer's partials runs as a kernel (-> per-(image, channel) scale / shift); the conv's
      // transform warps normalise the scaled fp16 tensor as it lands in shared memory: no normalised copy in HBM
      char pname[64];
      snprintf(pname, sizeof pname, "groupnorm statistics C=%d @%dx%d", xf->C, d.B, H * W);
      ProfScope prof(pname, 0.0, 0.0, s);
      const int partials = *d.pending;
      *d.pending = 0;
      HDRVAE_TRY(launch_gn_scale_shift(d.B, H * W, xf->C, xf->gamma, xf->beta, d.gn, d.gn_chunks, partials, s, &io.xf_scale,
                                       &io.xf_shift));
    } else if (xf != nullptr) {
      HDRVAE_TRY(launch_gn_scale_shift_from_sums(1, xf->C, xf->gamma, xf->beta, d.gn, d.gn_chunks,
                                                 (double)H * rows->pl.world * (double)W * (double)(xf->C / 32), s,
                                                 &io.xf_scale, &io.xf_shift));
    }
    HDRVAE_TRY(run_conv(d.ctx, *p, io, d.B, H, W, d.ctx->conv_impl, s));
    if (zero_y) HDRVAE_TRY(zero_border_halos(rows, io.y, OH, OW, p->cout, 2, s));
    if (xa_copy) HDRVAE_TRY(zero_border_halos(rows, io.y2, OH, OW, p->cout, 2, s));
    return 0;
  }));
  if (rows == nullptr || io.stats == nullptr) return 0;
  HDRVAE_TRY(step(d, [=](cudaStream_t s) { return launch_gn_reduce_partials(d.gn, 1, 512, d.gn_chunks, *d.pending, s); }));
  hdrvae_exchange ex;
  memset(&ex, 0, sizeof ex);
  add_halo(rows, &ex, io.y, OH, OW, pc.cout, dt_bytes(io.y_dtype));
  if (xa_copy) add_halo(rows, &ex, io.y2, OH, OW, pc.cout, 2);
  ex.kind |= HDRVAE_EX_ALLREDUCE_F64;
  ex.allreduce_off = ws_off(rows, gn_sums_ptr(d.gn, 1, 512, d.gn_chunks));
  ex.allreduce_count = 32 * 2;
  rows_exchange(rows, ex);
  return 0;
}

// conv(SiLU(GroupNorm(x))): the GroupNorm is applied inside the conv when gn_is_fused allows it for the conv as issued,
// otherwise by norm into t.
static int norm_conv(Decoder& d, const void* x, int x_dt, float x_scale, const NormW& nw, const PackedConv& pc, ConvIO io,
                     int H, int W, int flags = 0) {
  io.stats = stats_ptr(d);                       // what conv sets: the decision sees the conv as issued
  if (!gn_is_fused(d.ctx, pc, io, x_dt, H, W)) {
    HDRVAE_TRY(norm(d, x, x_dt, x_scale, nw, true, H, W));
    io.x = d.t;
    return conv(d, pc, io, H, W, flags);
  }
  io.x = x; io.xf_in_scale = 1.f / x_scale;
  return conv(d, pc, io, H, W, flags, &nw);
}

static int decode_res(Decoder& d, const ResW& rw, int H, int W) {
  hdrvae_ctx* ctx = d.ctx;
  const bool x16 = d.x_dt != DT_F32;
  const int stream_flags = x16 ? kZeroHalos : 0;
  {
    ConvIO io; io.y = d.hbuf; io.y_dtype = d.h_dt; io.y_scale = d.h_scale;
    HDRVAE_TRY(norm_conv(d, d.x, d.x_dt, d.x_scale, rw.n1, rw.c1, io, H, W));
  }
  ConvIO io;
  if (x16) { io.y_dtype = d.x_dt; io.y_scale = d.x_scale; }
  else if (rw.dual_out) { io.y2 = d.xa16; io.y2_dtype = ctx->op_dtype; io.y2_scale = kRawOperandScale; }
  if (!rw.has_nin) {
    io.y = d.x; io.residual = d.x;                  // x += conv2(t), in place
    io.res_dtype = d.x_dt; io.res_scale = 1.f / d.x_scale;
    return norm_conv(d, d.hbuf, d.h_dt, d.h_scale, rw.n2, rw.c2, io, H, W, stream_flags);
  }
  // norm2 as a separate pass (conv1's output lives in hbuf, which the shortcut is about to overwrite); then the
  // shortcut on the scaled 16-bit copy of x into hbuf, and conv2 accumulates onto it in place
  HDRVAE_TRY(norm(d, d.hbuf, d.h_dt, d.h_scale, rw.n2, true, H, W));
  io.x = d.t;
  if (nin_is_fused(ctx, rw, H, W)) {
    // x_new = conv2(t) + nin(x): ONE launch, written over the old x (whose scaled 16-bit copy is what the shortcut reads)
    io.x2 = d.xb16; io.pc2 = &rw.nin_x16; io.bias = rw.bias_c2_nin; io.y = d.x;
    if (!x16) return conv(d, rw.c2, io, H, W);
    // the shortcut reads the 16-bit stream itself; Cin != Cout, so the new stream goes to the other buffer
    io.x2 = d.x; io.y = d.hbuf;
    HDRVAE_TRY(conv(d, rw.c2, io, H, W, stream_flags));
    std::swap(d.x, d.hbuf);
    return 0;
  }
  HDRVAE_REQUIRE(!x16, "the 16-bit residual stream needs the fused shortcut");
  ConvIO sc; sc.x = d.xb16; sc.y = d.hbuf; sc.alpha = 1.0f / kRawOperandScale;
  HDRVAE_TRY(conv(d, rw.nin, sc, H, W, kNoStats));
  io.y = d.hbuf; io.residual = d.hbuf;
  HDRVAE_TRY(conv(d, rw.c2, io, H, W));
  std::swap(d.x, d.hbuf);
  return 0;
}

// conv_in on the staged latent, mid.block_1 and mid.attn_1's GroupNorm (no SiLU) into t
static int decode_to_attention(Decoder& d, int H, int W) {
  ConvIO io; io.x = d.lat; io.y = d.x; io.y_dtype = d.x_dt; io.y_scale = d.x_scale;
  HDRVAE_TRY(conv(d, d.ctx->conv_in, io, H, W, d.x_dt != DT_F32 ? kZeroHalos : 0));
  HDRVAE_TRY(decode_res(d, d.ctx->mid1, H, W));
  return norm(d, d.x, d.x_dt, d.x_scale, d.ctx->attn_norm, false, H, W);
}

// x += proj_out(o), mid.block_2, the up levels and norm_out (+ SiLU) into t: the tensor the reference's hook captures
// (16-bit operand of conv_out, or fp32 in the high-precision mode)
static int decode_from_attention(Decoder& d, const void* o, int H, int W) {
  hdrvae_ctx* ctx = d.ctx;
  const bool x16 = d.x_dt != DT_F32;
  {
    // proj_out adds in place and writes no halo rows: the stream's border halos stay zero
    ConvIO io; io.x = o; io.y = d.x; io.residual = d.x;
    io.y_dtype = d.x_dt; io.y_scale = d.x_scale; io.res_dtype = d.x_dt; io.res_scale = 1.f / d.x_scale;
    HDRVAE_TRY(conv(d, ctx->proj_out, io, H, W, kDenseInput));
  }
  HDRVAE_TRY(decode_res(d, ctx->mid2, H, W));
  for (int lvl = 3; lvl >= 0; --lvl) {
    for (int i = 0; i < 3; ++i) HDRVAE_TRY(decode_res(d, ctx->up[lvl][i], H, W));
    if (lvl != 0) {
      // operand: the scaled 16-bit copy written by the level's last ResBlock; levels 2 and 1 feed a nin_shortcut
      // one block later, so their output gets a scaled copy too
      ConvIO io; io.x = d.xa16; io.y = d.hbuf; io.alpha = 1.0f / kRawOperandScale;
      if (x16) { io.x = d.x; io.y_dtype = d.x_dt; io.y_scale = d.x_scale; }     // the stream is its own operand copy
      else if (lvl <= 2) { io.y2 = d.xb16; io.y2_dtype = ctx->op_dtype; io.y2_scale = kRawOperandScale; }
      HDRVAE_TRY(conv(d, ctx->upsample[lvl], io, H, W, x16 ? kZeroHalos : 0));
      std::swap(d.x, d.hbuf);
      H *= 2; W *= 2;
    }
  }
  return norm(d, d.x, d.x_dt, d.x_scale, ctx->norm_out, true, H, W, ctx->high ? DT_F32 : -1);
}

// mid.attn_1 between its GroupNorm (t) and proj_out, single-GPU: per-image q|k and v^T projections, then the attention
// core over all images; the high-precision mode takes the GEMM-level form on hi / lo operands.  *o: proj_out's operand.
static int attend_dense(Decoder& d, const Plan& pl, uint8_t* ws, const void** o_out) {
  hdrvae_ctx* ctx = d.ctx;
  const int B = d.B, impl = ctx->conv_impl, dt = ctx->op_dtype;
  cudaStream_t s = d.s;
  void* qk = ws + pl.off_qk;
  void* vt = ws + pl.off_vt;
  void* o = ws + pl.off_o;
  *o_out = o;
  if (ctx->high) {
    ProfScope prof("attention (high precision, GEMM form)", 4.0 * B * (double)pl.T * pl.T * 512 * 3, 0.0, s);
    for (int b = 0; b < B; ++b)
      HDRVAE_TRY(run_attention_high(ctx, pl, ws, reinterpret_cast<const uint16_t*>(d.t) + (size_t)b * pl.T * 1536,
                                    reinterpret_cast<uint16_t*>(o) + (size_t)b * pl.T * 1536, s));
    return 0;
  }
  if (pl.Tp != pl.T) HDRVAE_CUDA_OK(cudaMemsetAsync(qk, 0, (size_t)B * pl.Tp * 1024 * 2, s));
  {
    ProfScope pq("attention q|k and v^T projections", 2.0 * B * (double)pl.T * 512 * 1536, 0.0, s);
    for (int b = 0; b < B; ++b) {
      const uint16_t* tb = reinterpret_cast<const uint16_t*>(d.t) + (size_t)b * pl.T * 512;
      // [q*scale | k] = t Wqk^T + bqk : [T][1024]
      HDRVAE_TRY(run_gemm(ctx, dt, tb, 512, pl.T, 512, ctx->qk.w[0], 512, 1024, 1024,
                          reinterpret_cast<uint16_t*>(qk) + (size_t)b * pl.Tp * 1024, 1024, dt, ctx->qk.bias, false, 1.0f,
                          nullptr, impl, s));
      // v^T = Wv t^T + bv : [512][Tp]  (operand roles swapped so PV sees a K-major B operand)
      HDRVAE_TRY(run_gemm(ctx, dt, ctx->vproj.w[0], 512, 512, 512, tb, 512, pl.T, pl.Tp,
                          reinterpret_cast<uint16_t*>(vt) + (size_t)b * 512 * pl.Tp, pl.Tp, dt, ctx->vproj.bias, true, 1.0f,
                          nullptr, impl, s));
    }
  }
  ProfScope prof("attention core (QK^T, softmax, PV)", 4.0 * B * (double)pl.T * pl.T * 512, 10.0 * B * (double)pl.T * pl.Tp, s);
  // key-split partials borrow the block-internal fp32 buffer: nothing of a ResnetBlock is live across mid.attn_1
  return run_attention_core(ctx, B, pl.T, pl.Tp, qk, vt, o, 1.0f, d.hbuf, (size_t)B * pl.T * 64 * 256 * 4, plan_chunk(pl, ws), s);
}

static int run_decoder(hdrvae_ctx* ctx, const float* latent, const Plan& pl, uint8_t* ws, void** features,
                       cudaStream_t s) {
  HDRVAE_REQUIRE(ctx->loaded, "hdrvae: weights not loaded");
  const int B = pl.B, H = pl.h, W = pl.w;
  int pending = 0;
  Decoder d = make_decoder(ctx, nullptr, s, B, &pending);
  d.lat = ws + pl.off_lat;
  d.x = reinterpret_cast<float*>(ws + pl.off_x);
  d.hbuf = reinterpret_cast<float*>(ws + pl.off_h);
  d.t = ws + pl.off_t;
  d.xa16 = ws + pl.off_x16;
  d.xb16 = ws + pl.off_x16b;
  d.gn = ws + pl.off_gn;
  d.gn_chunks = pl.gn_chunks;
  HDRVAE_TRY(gn_scratch_reset(d.gn, B, pl.gn_chunks, s));
  if (ctx->high) {
    float* latf = reinterpret_cast<float*>(ws + pl.off_f32) + (size_t)pl.Tp * 1536;
    HDRVAE_TRY(launch_latent_to_nhwc(latent, latf, DT_F32, B, ctx->c_z, ctx->c_lat, ctx->pq_w, ctx->pq_b, H * W, 64, s));
    HDRVAE_TRY(launch_split3(latf, 64, d.lat, 192, (long long)B * H * W, 64, 1.f, 0, s));
  } else {
    HDRVAE_TRY(launch_latent_to_nhwc(latent, d.lat, ctx->op_dtype, B, ctx->c_z, ctx->c_lat, ctx->pq_w, ctx->pq_b, H * W, 64, s));
  }
  HDRVAE_TRY(decode_to_attention(d, H, W));
  const void* o = nullptr;
  HDRVAE_TRY(attend_dense(d, pl, ws, &o));
  HDRVAE_TRY(decode_from_attention(d, o, H, W));
  *features = d.t;
  return 0;
}

// mid.attn_1 between its GroupNorm (t) and proj_out, row tiling: q|k and v of this rank's tokens, all-gathered, then this
// rank's queries attend to all keys.  *o: proj_out's operand (dense [Tl][512]).
static void attend_rows(Decoder& d, int W, const void** o_out) {
  hdrvae_rows* st = d.rows;
  hdrvae_ctx* ctx = d.ctx;
  const RowsPlan& pl = st->pl;
  uint8_t* ws = st->ws;
  const int rank = st->rank, dt = ctx->op_dtype;
  uint16_t* qk = reinterpret_cast<uint16_t*>(ws + pl.off_qk);
  uint16_t* vb = reinterpret_cast<uint16_t*>(ws + pl.off_v);
  uint16_t* vt = reinterpret_cast<uint16_t*>(ws + pl.off_vt);
  uint16_t* o = reinterpret_cast<uint16_t*>(ws + pl.off_o);
  *o_out = o;
  const uint16_t* tl = reinterpret_cast<const uint16_t*>(d.t) + (size_t)W * 512;      // interior rows of the slab
  float* hscr = d.hbuf;                                   // idle across the attention: lends its memory to the key-split partials
  const size_t hscr_bytes = (size_t)(8 * pl.hl + 2) * 8 * pl.w * 256 * 4;
  step(d, [=](cudaStream_t s) {
    if (pl.Tp != pl.T) {
      HDRVAE_CUDA_OK(cudaMemsetAsync(qk, 0, (size_t)pl.Tp * 1024 * 2, s));
      HDRVAE_CUDA_OK(cudaMemsetAsync(vt, 0, (size_t)512 * pl.Tp * 2, s));
    }
    HDRVAE_TRY(run_gemm(ctx, dt, tl, 512, pl.Tl, 512, ctx->qk.w[0], 512, 1024, 1024, qk + (size_t)rank * pl.Tl * 1024, 1024, dt,
                        ctx->qk.bias, false, 1.0f, nullptr, HDRVAE_CONV_TCGEN05, s));
    return run_gemm(ctx, dt, tl, 512, pl.Tl, 512, ctx->vproj.w[0], 512, 512, 512, vb + (size_t)rank * pl.Tl * 512, 512, dt,
                    ctx->vproj.bias, false, 1.0f, nullptr, HDRVAE_CONV_TCGEN05, s);
  });
  hdrvae_exchange ex;
  memset(&ex, 0, sizeof ex);
  ex.kind = HDRVAE_EX_ALLGATHER;
  ex.n_gather = 2;
  ex.gather_off[0] = pl.off_qk; ex.gather_bytes_per_rank[0] = (size_t)pl.Tl * 1024 * 2;
  ex.gather_off[1] = pl.off_v;  ex.gather_bytes_per_rank[1] = (size_t)pl.Tl * 512 * 2;
  rows_exchange(st, ex);
  step(d, [=](cudaStream_t s) {
    HDRVAE_TRY(launch_transpose_pad(vb, vt, pl.T, 512, pl.Tp, s));
    return attention_fused(ctx, qk + (size_t)rank * pl.Tl * 1024, qk + 512, vt, 1, pl.Tl, pl.T, pl.Tp, o, 1.0f, hscr, hscr_bytes, s);
  });
}

static int build_rows_program(hdrvae_rows* st) {
  hdrvae_ctx* ctx = st->ctx;
  const RowsPlan& pl = st->pl;
  uint8_t* ws = st->ws;
  const int H = pl.hl, W = pl.w, rank = st->rank;
  Decoder d = make_decoder(ctx, st, nullptr, 1, &st->pending);
  d.lat = ws + pl.off_lat;
  d.x = reinterpret_cast<float*>(ws + pl.off_x);
  d.hbuf = reinterpret_cast<float*>(ws + pl.off_h);
  d.t = ws + pl.off_t;
  d.xa16 = ws + pl.off_xa;
  d.xb16 = ws + pl.off_xb;
  d.gn = ws + pl.off_gn;
  d.gn_chunks = pl.gn_chunks;
  step(d, [=](cudaStream_t s) {
    // latent rows of this rank plus one neighbour row each side (rows outside the image are zero)
    HDRVAE_TRY(launch_latent_rows_to_nhwc(st->latent, d.lat, ctx->op_dtype, ctx->c_z, ctx->c_lat, ctx->pq_w, ctx->pq_b, pl.h,
                                          pl.w, rank * pl.hl - 1, pl.hl + 2, 64, s));
    return gn_scratch_reset(d.gn, 1, pl.gn_chunks, s);
  });
  HDRVAE_TRY(decode_to_attention(d, H, W));
  const void* o = nullptr;
  attend_rows(d, W, &o);
  HDRVAE_TRY(decode_from_attention(d, o, H, W));
  // epilogue: phase A on this rank's rows, the HDR statistics all-reduced, phase B
  void* epi = ws + pl.off_epi;
  // conv_out's scratch: the other stream buffer is free by now
  step(d, [=](cudaStream_t s) { return run_phase_a(ctx, d.t, 1, 8 * H, 8 * W, 1, d.hbuf, epi, s); });
  hdrvae_exchange ex;
  memset(&ex, 0, sizeof ex);
  ex.kind = HDRVAE_EX_RAW_STATS;
  ex.raw_stats_off = ws_off(st, epilogue_raw_stats_ptr(epi, 1, 8 * H, 8 * W));
  rows_exchange(st, ex);
  step(d, [=](cudaStream_t s) {
    return launch_epilogue_phase_b(1, 8 * H, 8 * W, st->mode, st->factor, st->ev, st->out, nullptr, epi, s);
  });
  return 0;
}

}  // namespace hdrvae

// =================================================================================================== C ABI
extern "C" {

const char* hdrvae_last_error(void) { return g_last_error.c_str(); }
int hdrvae_abi_version(void) { return HDRVAE_ABI_VERSION; }

int hdrvae_create(hdrvae_ctx** out, int device) {
  HDRVAE_REQUIRE(out != nullptr, "hdrvae_create: null out pointer");
  int n = 0;
  HDRVAE_CUDA_OK(cudaGetDeviceCount(&n));
  HDRVAE_REQUIRE(device >= 0 && device < n, "hdrvae_create: no CUDA device %d (count %d); there is no CPU path", device, n);
  HDRVAE_CUDA_OK(cudaSetDevice(device));
  cudaDeviceProp prop;
  HDRVAE_CUDA_OK(cudaGetDeviceProperties(&prop, device));
  HDRVAE_REQUIRE(prop.major == 10, "hdrvae_create: device %d is sm_%d%d; this library is sm_100a only", device, prop.major,
                 prop.minor);
  hdrvae_ctx* ctx = new hdrvae_ctx();
  ctx->device = device;
  ctx->num_sms = prop.multiProcessorCount;
  if (switches().conv_direct) ctx->conv_impl = HDRVAE_CONV_DIRECT;
  *out = ctx;
  return 0;
}

int hdrvae_destroy(hdrvae_ctx* ctx) {
  if (ctx == nullptr) return 0;
  cudaSetDevice(ctx->device);
  for (auto& g : ctx->graphs) cudaGraphExecDestroy(g.exec);
  for (void* p : ctx->owned) cudaFree(p);
  delete ctx;
  return 0;
}

static_assert(sizeof(hdrvae_stats) == 200 && sizeof(hdrvae_raw_stats) == 96 && sizeof(hdrvae_exchange) == 152 &&
              sizeof(hdrvae_conv_extra) == 64, "ABI struct layout changed");
static_assert((int)HDRVAE_ACT_NONE == (int)ACT_NONE && (int)HDRVAE_ACT_SILU == (int)ACT_SILU &&
              (int)HDRVAE_ACT_GATE == (int)ACT_GATE,
              "hdrvae_conv_extra::act is GemmParams::act");

long long hdrvae_launch_count(void) { return g_launch_count; }

int hdrvae_profile_begin(void) {
  for (auto& e : g_prof) { cudaEventDestroy(e.e0); cudaEventDestroy(e.e1); }
  g_prof.clear();
  g_prof_on = true;
  return 0;
}

// Synchronises the device, writes "name\tms\tTFLOP/s\tGB/s" lines to `path` (or stderr) and stops profiling.
int hdrvae_profile_end(const char* path) {
  g_prof_on = false;
  HDRVAE_CUDA_OK(cudaDeviceSynchronize());
  FILE* f = path ? fopen(path, "w") : stderr;
  HDRVAE_REQUIRE(f != nullptr, "hdrvae_profile_end: cannot open %s", path);
  double total = 0.0;
  for (auto& e : g_prof) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e.e0, e.e1);
    total += ms;
    fprintf(f, "%-52s\t%9.4f ms\t%8.1f TFLOP/s\t%8.1f GB/s\n", e.name.c_str(), ms, e.flops / ms / 1e9, e.bytes / ms / 1e6);
    cudaEventDestroy(e.e0); cudaEventDestroy(e.e1);
  }
  fprintf(f, "%-52s\t%9.4f ms\n", "TOTAL (sum of scopes)", total);
  if (path) fclose(f);
  g_prof.clear();
  return 0;
}

int hdrvae_set_conv_impl(hdrvae_ctx* ctx, int impl) {
  HDRVAE_REQUIRE(ctx != nullptr && (impl == HDRVAE_CONV_TCGEN05 || impl == HDRVAE_CONV_DIRECT), "bad conv impl");
  ctx->conv_impl = impl;
  return 0;
}

int hdrvae_latent_channels(const hdrvae_ctx* ctx) {
  HDRVAE_REQUIRE(ctx != nullptr && ctx->loaded, "hdrvae_latent_channels: weights not loaded");
  return ctx->c_lat;
}

int hdrvae_operand_dtype(hdrvae_ctx* ctx) { return ctx ? ctx->op_dtype : -1; }
int hdrvae_features_dtype(hdrvae_ctx* ctx) { return ctx ? (ctx->high ? DT_F32 : ctx->op_dtype) : -1; }

int hdrvae_set_cta_group(hdrvae_ctx* ctx, int cta_group) {
  HDRVAE_REQUIRE(ctx != nullptr && cta_group >= 0 && cta_group <= 2, "bad cta_group");
  ctx->cta_group = cta_group;
  return 0;
}

int hdrvae_load_weights(hdrvae_ctx* ctx, const hdrvae_weight_desc* descs, int n, int precision) {
  HDRVAE_REQUIRE(ctx != nullptr && descs != nullptr, "hdrvae_load_weights: null argument");
  HDRVAE_REQUIRE(precision == HDRVAE_PRECISION_BF16 || precision == HDRVAE_PRECISION_F16 || precision == HDRVAE_PRECISION_HIGH,
                 "hdrvae_load_weights: unsupported precision %d", precision);
  HDRVAE_REQUIRE(!ctx->loaded, "hdrvae_load_weights: context already holds weights (create a new one)");
  HDRVAE_CUDA_OK(cudaSetDevice(ctx->device));
  ctx->op_dtype = precision == HDRVAE_PRECISION_BF16 ? DT_BF16 : DT_F16;
  ctx->high = precision == HDRVAE_PRECISION_HIGH;
  const bool high = ctx->high;
  const int op = ctx->op_dtype;
  cudaStream_t s = nullptr;
  std::vector<void*> staging;
  for (int i = 0; i < n; ++i) {
    const hdrvae_weight_desc& d = descs[i];
    HDRVAE_REQUIRE(d.name && d.data && d.ndim >= 1 && d.ndim <= 4, "hdrvae_load_weights: bad descriptor %d", i);
    long long cnt = 1;
    std::vector<int64_t> shp;
    for (int k = 0; k < d.ndim; ++k) { cnt *= d.shape[k]; shp.push_back(d.shape[k]); }
    const size_t esz = d.dtype == HDRVAE_F32 ? 4 : 2;
    void* stage = nullptr;
    HDRVAE_CUDA_OK(cudaMalloc(&stage, cnt * esz));
    staging.push_back(stage);
    HDRVAE_CUDA_OK(cudaMemcpyAsync(stage, d.data, cnt * esz, cudaMemcpyDefault, s));
    float* f = nullptr;
    HDRVAE_TRY(dev_alloc(ctx, cnt * sizeof(float), (void**)&f));
    HDRVAE_TRY(launch_to_f32(stage, d.dtype, f, cnt, s));
    ctx->raw[d.name] = f;
    ctx->shapes[d.name] = shp;
  }
  auto W = [&](const std::string& k) -> float* { auto it = ctx->raw.find(k); return it == ctx->raw.end() ? nullptr : it->second; };
  auto need_conv = [&](const std::string& k, int cout, int cin, int ks) -> int {
    auto it = ctx->shapes.find(k + ".weight");
    HDRVAE_REQUIRE(it != ctx->shapes.end() && W(k + ".bias") != nullptr, "state dict lacks %s.{weight,bias}", k.c_str());
    const auto& sh = it->second;
    HDRVAE_REQUIRE(sh.size() == 4 && sh[0] == cout && sh[1] == cin && sh[2] == ks && sh[3] == ks,
                   "%s.weight has the wrong shape (want [%d,%d,%d,%d])", k.c_str(), cout, cin, ks, ks);
    return 0;
  };
  auto conv = [&](const std::string& k, int cout, int cin, int ks, bool up, int w_dtype, PackedConv* pc) -> int {
    HDRVAE_TRY(need_conv(k, cout, cin, ks));
    return pack_conv(ctx, W(k + ".weight"), W(k + ".bias"), cout, cin, ks, up, 1.f, w_dtype, pc, s, high);
  };
  auto norm = [&](const std::string& k, int C, NormW* nw) -> int {
    HDRVAE_REQUIRE(W(k + ".weight") && W(k + ".bias") && ctx->shapes[k + ".weight"].size() == 1 &&
                       ctx->shapes[k + ".weight"][0] == C, "state dict lacks %s (GroupNorm over %d channels)", k.c_str(), C);
    nw->gamma = W(k + ".weight"); nw->beta = W(k + ".bias"); nw->C = C;
    return 0;
  };
  auto res = [&](const std::string& k, int cin, int cout, ResW* rw) -> int {
    HDRVAE_TRY(norm(k + ".norm1", cin, &rw->n1));
    HDRVAE_TRY(conv(k + ".conv1", cout, cin, 3, false, op, &rw->c1));
    HDRVAE_TRY(norm(k + ".norm2", cout, &rw->n2));
    HDRVAE_TRY(conv(k + ".conv2", cout, cout, 3, false, op, &rw->c2));
    rw->has_nin = cin != cout;
    if (rw->has_nin) {
      HDRVAE_TRY(conv(k + ".nin_shortcut", cout, cin, 1, false, op, &rw->nin));   // reads the scaled 16-bit copy of x
      if (!high) {
        // the form fused into conv2: weights x 2^4 (undoes the operand scale), bias = conv2.bias + nin_shortcut.bias
        HDRVAE_TRY(pack_conv(ctx, W(k + ".nin_shortcut.weight"), nullptr, cout, cin, 1, false, 1.0f / kRawOperandScale, op, &rw->nin_x16, s));
        HDRVAE_TRY(dev_alloc(ctx, rw->c2.cout_pad * sizeof(float), (void**)&rw->bias_c2_nin));
        HDRVAE_TRY(launch_add_vectors(rw->c2.bias, rw->nin.bias, rw->bias_c2_nin, rw->c2.cout_pad, s));
      }
    }
    return 0;
  };

  {
    // latent channels from the weights: conv_in's input (Flux 16, SD1.x / SDXL 4), and post_quant_conv's input when the
    // first-stage model has one (a 1x1 conv with bias that SD-family AutoencoderKL applies to the latent before the decoder)
    auto it = ctx->shapes.find("conv_in.weight");
    const int cz = it != ctx->shapes.end() && it->second.size() == 4 ? (int)it->second[1] : 16;
    HDRVAE_REQUIRE(cz >= 1 && cz <= 64, "conv_in.weight has %d input channels (latent channels must be 1..64)", cz);
    HDRVAE_TRY(conv("conv_in", 512, cz, 3, false, op, &ctx->conv_in));
    ctx->c_z = ctx->c_lat = cz;
    const bool pw = ctx->shapes.count("post_quant_conv.weight") != 0, pb = ctx->shapes.count("post_quant_conv.bias") != 0;
    HDRVAE_REQUIRE(pw == pb, "post_quant_conv needs both weight and bias (got only its %s)", pw ? "weight" : "bias");
    if (pw) {
      const auto& sw = ctx->shapes["post_quant_conv.weight"];
      const auto& sb = ctx->shapes["post_quant_conv.bias"];
      const int cl = sw.size() == 4 ? (int)sw[1] : 0;
      HDRVAE_REQUIRE(sw.size() == 4 && sw[0] == cz && cl >= 1 && cl <= 64 && sw[2] == 1 && sw[3] == 1 && sb.size() == 1 && sb[0] == cz,
                     "post_quant_conv has the wrong shape (want weight [%d,C,1,1] with 1 <= C <= 64 and bias [%d])", cz, cz);
      ctx->c_lat = cl;
      ctx->pq_w = W("post_quant_conv.weight");
      ctx->pq_b = W("post_quant_conv.bias");
    }
  }
  HDRVAE_TRY(res("mid.block_1", 512, 512, &ctx->mid1));
  HDRVAE_TRY(res("mid.block_2", 512, 512, &ctx->mid2));
  HDRVAE_TRY(norm("mid.attn_1.norm", 512, &ctx->attn_norm));
  {
    // fused [q * 1/sqrt(512) ; k] projection: one [1024][512] K-major operand + concatenated bias
    HDRVAE_TRY(need_conv("mid.attn_1.q", 512, 512, 1));
    HDRVAE_TRY(need_conv("mid.attn_1.k", 512, 512, 1));
    const float scale = 1.0f / sqrtf(512.0f);
    PackedConv& qk = ctx->qk;
    qk.cin = qk.cin_pad = 512; qk.cout = 1024; qk.ks = 1; qk.w_dtype = op; qk.kmul = high ? 3 : 1;
    HDRVAE_TRY(dev_alloc(ctx, (size_t)1024 * 512 * 2 * qk.kmul, &qk.w[0]));
    HDRVAE_TRY(dev_alloc(ctx, 1024 * sizeof(float), (void**)&qk.bias));
    int mask1[1] = {1};
    HDRVAE_TRY(launch_pack_weight(W("mid.attn_1.q.weight"), qk.w[0], op, 512, 512, 1, 1, 512, mask1, scale, s, high ? 1 : 0));
    HDRVAE_TRY(launch_pack_weight(W("mid.attn_1.k.weight"), reinterpret_cast<uint16_t*>(qk.w[0]) + 512 * 512 * qk.kmul, op, 512, 512, 1,
                                  1, 512, mask1, 1.f, s, high ? 1 : 0));
    std::vector<float> hb(1024);
    HDRVAE_CUDA_OK(cudaMemcpyAsync(hb.data(), W("mid.attn_1.q.bias"), 512 * 4, cudaMemcpyDeviceToHost, s));
    HDRVAE_CUDA_OK(cudaMemcpyAsync(hb.data() + 512, W("mid.attn_1.k.bias"), 512 * 4, cudaMemcpyDeviceToHost, s));
    HDRVAE_CUDA_OK(cudaStreamSynchronize(s));
    for (int i = 0; i < 512; ++i) hb[i] *= scale;
    HDRVAE_CUDA_OK(cudaMemcpy(qk.bias, hb.data(), 1024 * 4, cudaMemcpyHostToDevice));
  }
  HDRVAE_TRY(conv("mid.attn_1.v", 512, 512, 1, false, op, &ctx->vproj));
  HDRVAE_TRY(conv("mid.attn_1.proj_out", 512, 512, 1, false, op, &ctx->proj_out));
  const int ch[4] = {128, 256, 512, 512};
  int cin = 512;
  for (int lvl = 3; lvl >= 0; --lvl) {
    for (int i = 0; i < 3; ++i) {
      HDRVAE_TRY(res("up." + std::to_string(lvl) + ".block." + std::to_string(i), cin, ch[lvl], &ctx->up[lvl][i]));
      cin = ch[lvl];
    }
    if (lvl != 0) {
      ctx->up[lvl][2].dual_out = true;      // its output is the upsample conv's operand
      HDRVAE_TRY(conv("up." + std::to_string(lvl) + ".upsample.conv", cin, cin, 3, true, op, &ctx->upsample[lvl]));
    }
  }
  HDRVAE_TRY(norm("norm_out", 128, &ctx->norm_out));
  HDRVAE_TRY(need_conv("conv_out", 3, 128, 3));
  ctx->conv_out_w = W("conv_out.weight");
  ctx->conv_out_b = W("conv_out.bias");
  if (op == DT_F16 && !high) {
    // conv_out on the tensor cores for the product path: fp32 weights as fp16 hi + lo rows (exact to ~2^-21)
    float* w8 = nullptr;
    HDRVAE_CUDA_OK(cudaMalloc((void**)&w8, 8 * 1152 * sizeof(float)));
    staging.push_back(w8);
    HDRVAE_TRY(launch_split_hi_lo(ctx->conv_out_w, w8, 1152, s));
    HDRVAE_TRY(pack_conv(ctx, w8, nullptr, 8, 128, 3, false, 1.f, DT_F16, &ctx->conv_out_tc, s));
  }
  HDRVAE_CUDA_OK(cudaStreamSynchronize(s));
  for (void* p : staging) cudaFree(p);
  ctx->loaded = true;
  return 0;
}

int hdrvae_workspace_bytes(hdrvae_ctx* ctx, int B, int h, int w, size_t* bytes) {
  HDRVAE_REQUIRE(ctx != nullptr && bytes != nullptr, "hdrvae_workspace_bytes: null argument");
  HDRVAE_REQUIRE(B >= 1 && h >= 1 && w >= 1, "hdrvae_workspace_bytes: empty latent batch [%d,%d,%d,%d]", B, ctx->c_lat, h, w);
  *bytes = decode_plan(ctx, B, h, w).total;
  return 0;
}

// ---- CUDA-graph segments ------------------------------------------------------------------------------------------
// The decode is captured into two CUDA graphs the second time a (shape, mode, workspace) key is seen and replayed
// afterwards: segment 0 = decoder + epilogue phase A (~160 launches for a batch of 4), segment 1 = epilogue phase B.
// The split sits exactly where batch sharding all-reduces the raw statistics (hdrvae_decode_begin / _finish), so the
// sharded path replays the same graphs as the single-GPU one.  The latent is staged into / the image out of fixed
// workspace buffers so the graphs do not depend on the caller's tensor addresses.  HDRVAE_NO_GRAPH=1 disables it.
static bool graphs_enabled(hdrvae_ctx* ctx, cudaStream_t s) {
  return ctx->use_graphs && switches().graphs && !g_prof_on && s != nullptr;     // capture needs a non-default stream
}

static int run_segment(hdrvae_ctx* ctx, hdrvae_ctx::GraphEntry key, cudaStream_t s, const std::function<int()>& body) {
  auto same = [&](const hdrvae_ctx::GraphEntry& g) {
    return g.seg == key.seg && g.B == key.B && g.h == key.h && g.w == key.w && g.mode == key.mode && g.factor == key.factor &&
           g.ev == key.ev && g.ws == key.ws && g.conv_impl == key.conv_impl && g.cta_group == key.cta_group;
  };
  for (auto& g : ctx->graphs)
    if (same(g)) {
      g_launch_count += g.n_kernels;
      HDRVAE_CUDA_OK(cudaGraphLaunch(g.exec, s));
      return 0;
    }
  bool seen = false;
  for (auto& g : ctx->seen) if (same(g)) seen = true;
  if (!seen) {
    // first use of this key: plain launches (also runs every one-time cudaFuncSetAttribute outside a capture)
    if (ctx->seen.size() > 64) ctx->seen.clear();
    ctx->seen.push_back(key);
    return body();
  }
  const long long n_before = g_launch_count;    // launches recorded by the capture = kernels of every replay
  HDRVAE_CUDA_OK(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
  const int r = body();
  cudaGraph_t graph = nullptr;
  cudaError_t e = cudaStreamEndCapture(s, &graph);
  if (r != 0) { if (graph) cudaGraphDestroy(graph); return r; }
  HDRVAE_REQUIRE(e == cudaSuccess && graph != nullptr, "hdrvae_decode: CUDA graph capture failed: %s", cudaGetErrorString(e));
  cudaGraphExec_t exec = nullptr;
  e = cudaGraphInstantiate(&exec, graph, 0);
  cudaGraphDestroy(graph);
  HDRVAE_REQUIRE(e == cudaSuccess, "hdrvae_decode: cudaGraphInstantiate failed: %s", cudaGetErrorString(e));
  if (ctx->graphs.size() >= 16) { cudaGraphExecDestroy(ctx->graphs.front().exec); ctx->graphs.erase(ctx->graphs.begin()); }
  key.exec = exec;
  key.n_kernels = g_launch_count - n_before;
  ctx->graphs.push_back(key);
  HDRVAE_CUDA_OK(cudaGraphLaunch(exec, s));
  return 0;
}

int hdrvae_decode_begin(hdrvae_ctx* ctx, const float* latent, int B, int h, int w, void* workspace, size_t ws_bytes,
                        void** raw_stats_dev, void* stream) {
  HDRVAE_REQUIRE(ctx != nullptr && latent != nullptr, "hdrvae_decode: null argument");
  HDRVAE_REQUIRE(B >= 1 && h >= 1 && w >= 1, "hdrvae_decode: empty latent batch [%d,%d,%d,%d]", B, ctx->c_lat, h, w);
  HDRVAE_CUDA_OK(cudaSetDevice(ctx->device));
  const Plan pl = decode_plan(ctx, B, h, w);
  HDRVAE_TRY(check_ws(pl, workspace, ws_bytes));
  uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  auto body = [&](const float* lat) -> int {
    void* feat = nullptr;
    HDRVAE_TRY(run_decoder(ctx, lat, pl, ws, &feat, s));
    ProfScope prof("epilogue phase A (conv_out, max-pool, stats)", 2.0 * B * 64.0 * h * w * 3 * 1152, B * 64.0 * h * w * (256 + 24), s);
    return run_phase_a(ctx, feat, B, 8 * h, 8 * w, 0, reinterpret_cast<float*>(ws + pl.off_h), ws + pl.off_epi, s);
  };
  if (graphs_enabled(ctx, s)) {
    float* lat_in = reinterpret_cast<float*>(ws + pl.off_lat_in);
    HDRVAE_CUDA_OK(cudaMemcpyAsync(lat_in, latent, (size_t)B * ctx->c_lat * pl.T * 4, cudaMemcpyDeviceToDevice, s));
    hdrvae_ctx::GraphEntry key{0, B, h, w, 0, ctx->conv_impl, ctx->cta_group, 0.f, 0.f, workspace, nullptr, 0};
    HDRVAE_TRY(run_segment(ctx, key, s, [&]() { return body(lat_in); }));
  } else {
    HDRVAE_TRY(body(latent));
  }
  if (raw_stats_dev != nullptr) *raw_stats_dev = epilogue_raw_stats_ptr(ws + pl.off_epi, B, 8 * h, 8 * w);
  return 0;
}

int hdrvae_decode_finish(hdrvae_ctx* ctx, int B, int h, int w, int mode, float expansion_factor, float ev_multiplier,
                         float* out_bhwc, hdrvae_stats* stats, void* workspace, size_t ws_bytes, void* stream) {
  HDRVAE_REQUIRE(ctx != nullptr && out_bhwc != nullptr, "hdrvae_decode: null argument");
  HDRVAE_REQUIRE(mode >= 0 && mode <= 3, "hdrvae_decode: bad mode %d", mode);
  HDRVAE_CUDA_OK(cudaSetDevice(ctx->device));
  const Plan pl = decode_plan(ctx, B, h, w);
  HDRVAE_TRY(check_ws(pl, workspace, ws_bytes));
  uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  if (!graphs_enabled(ctx, s)) {
    ProfScope prof("epilogue phase B (mode formula)", 0.0, B * 64.0 * h * w * 36, s);
    return launch_epilogue_phase_b(B, 8 * h, 8 * w, mode, expansion_factor, ev_multiplier, out_bhwc, stats, ws + pl.off_epi, s);
  }
  float* img = reinterpret_cast<float*>(ws + pl.off_img);
  hdrvae_ctx::GraphEntry key{1, B, h, w, mode, ctx->conv_impl, ctx->cta_group, expansion_factor, ev_multiplier, workspace, nullptr, 0};
  HDRVAE_TRY(run_segment(ctx, key, s, [&]() {
    return launch_epilogue_phase_b(B, 8 * h, 8 * w, mode, expansion_factor, ev_multiplier, img, nullptr, ws + pl.off_epi, s);
  }));
  HDRVAE_CUDA_OK(cudaMemcpyAsync(out_bhwc, img, (size_t)B * 64 * pl.T * 3 * 4, cudaMemcpyDeviceToDevice, s));
  if (stats != nullptr) {
    HDRVAE_CUDA_OK(cudaMemcpyAsync(stats, epilogue_stats_dev_ptr(ws + pl.off_epi, B, 8 * h, 8 * w), sizeof(hdrvae_stats),
                                   cudaMemcpyDeviceToHost, s));
    HDRVAE_CUDA_OK(cudaStreamSynchronize(s));
  }
  return 0;
}

// One call = the two segments back to back (single GPU: nothing to exchange in between).
int hdrvae_decode(hdrvae_ctx* ctx, const float* latent, int B, int h, int w, int mode, float expansion_factor,
                  float ev_multiplier, float* out_bhwc, hdrvae_stats* stats, void* workspace, size_t ws_bytes,
                  void* stream) {
  HDRVAE_REQUIRE(ctx != nullptr && latent != nullptr && out_bhwc != nullptr, "hdrvae_decode: null argument");
  HDRVAE_REQUIRE(B >= 1 && h >= 1 && w >= 1, "hdrvae_decode: empty latent batch [%d,%d,%d,%d]", B, ctx->c_lat, h, w);
  HDRVAE_REQUIRE(mode >= 0 && mode <= 3, "hdrvae_decode: bad mode %d", mode);
  HDRVAE_TRY(hdrvae_decode_begin(ctx, latent, B, h, w, workspace, ws_bytes, nullptr, stream));
  return hdrvae_decode_finish(ctx, B, h, w, mode, expansion_factor, ev_multiplier, out_bhwc, stats, workspace, ws_bytes, stream);
}

// Merge `n` gathered hdrvae_raw_stats blocks (96 bytes each, rank order) into `dst`: MIN / MAX / SUM in a fixed order,
// so every rank computes bit-identical batch-global statistics from ONE all-gather.
int hdrvae_raw_stats_merge(const void* blocks, int n, void* dst, void* stream) {
  HDRVAE_REQUIRE(blocks != nullptr && dst != nullptr && n >= 1, "hdrvae_raw_stats_merge: bad argument");
  return launch_raw_stats_merge(reinterpret_cast<const hdrvae_raw_stats*>(blocks), n, reinterpret_cast<hdrvae_raw_stats*>(dst),
                                reinterpret_cast<cudaStream_t>(stream));
}

int hdrvae_rows_workspace_bytes(hdrvae_ctx* ctx, int h, int w, int world, size_t* bytes) {
  HDRVAE_REQUIRE(ctx && bytes && h >= 1 && w >= 1 && world >= 1, "hdrvae_rows_workspace_bytes: bad argument");
  HDRVAE_REQUIRE(h % world == 0, "row tiling needs the latent height (%d) to be a multiple of the rank count (%d)", h, world);
  *bytes = make_rows_plan(h, w, world).total;
  return 0;
}

int hdrvae_rows_begin(hdrvae_ctx* ctx, const float* latent_full, int h, int w, int rank, int world, int mode,
                      float expansion_factor, float ev_multiplier, float* out_rows, void* workspace, size_t ws_bytes,
                      hdrvae_rows** state) {
  HDRVAE_REQUIRE(ctx && latent_full && out_rows && workspace && state, "hdrvae_rows_begin: null argument");
  HDRVAE_REQUIRE(ctx->loaded, "hdrvae: weights not loaded");
  HDRVAE_REQUIRE(h >= 1 && w >= 1 && world >= 1 && rank >= 0 && rank < world && h % world == 0,
                 "hdrvae_rows_begin: latent height %d must split evenly over %d ranks (rank %d)", h, world, rank);
  HDRVAE_REQUIRE(mode >= 0 && mode <= 3, "hdrvae_rows_begin: bad mode %d", mode);
  HDRVAE_REQUIRE(ctx->conv_impl == HDRVAE_CONV_TCGEN05, "row tiling runs on the tcgen05 kernels only");
  HDRVAE_REQUIRE(!ctx->high, "row tiling is not available in the high-precision mode");
  hdrvae_rows* st = new hdrvae_rows();
  st->ctx = ctx;
  st->pl = make_rows_plan(h, w, world);
  if (ws_bytes < st->pl.total || (reinterpret_cast<uintptr_t>(workspace) & 1023) != 0) {
    set_error("hdrvae_rows_begin: workspace too small or misaligned (%zu < %zu bytes)", ws_bytes, st->pl.total);
    delete st;
    return -2;
  }
  st->rank = rank; st->mode = mode; st->factor = expansion_factor; st->ev = ev_multiplier;
  st->ws = reinterpret_cast<uint8_t*>(workspace);
  st->latent = latent_full;
  st->out = out_rows;
  int r = build_rows_program(st);
  if (r != 0) { delete st; return r; }
  *state = st;
  return 0;
}

int hdrvae_rows_run(hdrvae_rows* st, hdrvae_exchange* ex, void* stream) {
  HDRVAE_REQUIRE(st && ex, "hdrvae_rows_run: null argument");
  HDRVAE_CUDA_OK(cudaSetDevice(st->ctx->device));
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  memset(ex, 0, sizeof *ex);
  while (st->pc < st->ops.size()) {
    hdrvae_rows::Op& op = st->ops[st->pc++];
    if (op.exchange) {
      *ex = op.ex;
      return 0;
    }
    HDRVAE_TRY(op.fn(s));
  }
  ex->kind = HDRVAE_EX_END;
  return 0;
}

// ---- device-driven transport (rows_p2p.cu): library-owned, IPC-shared workspaces ---------------------------------
int hdrvae_peer_alloc(hdrvae_ctx* ctx, size_t bytes, void** dev_ptr, hdrvae_ipc_handle* handle) {
  HDRVAE_REQUIRE(ctx && dev_ptr && handle && bytes > 0, "hdrvae_peer_alloc: bad argument");
  static_assert(sizeof(hdrvae_ipc_handle) == sizeof(cudaIpcMemHandle_t), "IPC handle size");
  HDRVAE_CUDA_OK(cudaSetDevice(ctx->device));
  void* p = nullptr;
  HDRVAE_CUDA_OK(cudaMalloc(&p, bytes));
  cudaError_t e = cudaMemset(p, 0, bytes);              // the mailbox must start at zero (exchange counter, flags)
  if (e == cudaSuccess) e = cudaIpcGetMemHandle(reinterpret_cast<cudaIpcMemHandle_t*>(handle), p);
  if (e != cudaSuccess) { cudaFree(p); set_error("hdrvae_peer_alloc: %s", cudaGetErrorString(e)); return -1; }
  *dev_ptr = p;
  return 0;
}
int hdrvae_peer_open(hdrvae_ctx* ctx, const hdrvae_ipc_handle* handle, void** mapped) {
  HDRVAE_REQUIRE(ctx && handle && mapped, "hdrvae_peer_open: bad argument");
  HDRVAE_CUDA_OK(cudaSetDevice(ctx->device));
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof h);
  HDRVAE_CUDA_OK(cudaIpcOpenMemHandle(mapped, h, cudaIpcMemLazyEnablePeerAccess));
  return 0;
}
int hdrvae_peer_close(hdrvae_ctx* ctx, void* mapped) {
  if (ctx == nullptr || mapped == nullptr) return 0;
  cudaSetDevice(ctx->device);
  HDRVAE_CUDA_OK(cudaIpcCloseMemHandle(mapped));
  return 0;
}
int hdrvae_peer_free(hdrvae_ctx* ctx, void* dev_ptr) {
  if (ctx == nullptr || dev_ptr == nullptr) return 0;
  cudaSetDevice(ctx->device);
  HDRVAE_CUDA_OK(cudaFree(dev_ptr));
  return 0;
}

int hdrvae_rows_set_peers(hdrvae_rows* st, void* const* workspaces, int world) {
  HDRVAE_REQUIRE(st != nullptr && workspaces != nullptr && world == st->pl.world && world <= kRowsMaxRanks,
                 "hdrvae_rows_set_peers: need the workspaces of all %d ranks (at most %d)", st ? st->pl.world : 0, kRowsMaxRanks);
  for (int r = 0; r < world; ++r) {
    HDRVAE_REQUIRE(workspaces[r] != nullptr, "hdrvae_rows_set_peers: workspace of rank %d is null", r);
    st->peers[r] = reinterpret_cast<uint8_t*>(workspaces[r]);
  }
  HDRVAE_REQUIRE(st->peers[st->rank] == st->ws, "hdrvae_rows_set_peers: entry [rank] must be this rank's own workspace");
  st->peers_set = true;
  return 0;
}

// The whole program in one call: compute steps and exchanges are enqueued on `stream` back to back; nothing returns to
// the host in between.
int hdrvae_rows_run_direct(hdrvae_rows* st, void* stream) {
  HDRVAE_REQUIRE(st != nullptr && st->peers_set, "hdrvae_rows_run_direct: call hdrvae_rows_set_peers first");
  HDRVAE_CUDA_OK(cudaSetDevice(st->ctx->device));
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const int rank = st->rank, world = st->pl.world;
  while (st->pc < st->ops.size()) {
    hdrvae_rows::Op& op = st->ops[st->pc++];
    if (!op.exchange) { HDRVAE_TRY(op.fn(s)); continue; }
    const hdrvae_exchange& ex = op.ex;
    RowsPushArgs a;
    memset(&a, 0, sizeof a);
    a.ws = st->ws; a.off_mail = st->pl.off_mail; a.rank = rank; a.world = world;
    for (int r = 0; r < world; ++r) a.peers[r] = st->peers[r];
    size_t total = 0;
    auto seg = [&](int peer, int kind, size_t dst, size_t src, size_t bytes) -> int {
      HDRVAE_REQUIRE(a.n_seg < 72 && (dst & 15) == 0 && (src & 15) == 0 && (bytes & 15) == 0 && bytes < (1ull << 32),
                     "rows exchange: segment not 16-byte aligned or too many segments");
      RowsSegment& g = a.seg[a.n_seg++];
      g.peer = peer; g.kind = kind; g.dst_off = dst; g.src_off = src; g.bytes = (unsigned int)bytes;
      total += bytes;
      return 0;
    };
    if (ex.kind & HDRVAE_EX_HALO) {
      for (int i = 0; i < ex.n_halo; ++i) {
        if (rank > 0) HDRVAE_TRY(seg(rank - 1, 0, ex.halo_bottom_off[i], ex.halo_first_row_off[i], ex.halo_row_bytes[i]));
        if (rank < world - 1) HDRVAE_TRY(seg(rank + 1, 0, ex.halo_top_off[i], ex.halo_last_row_off[i], ex.halo_row_bytes[i]));
      }
    }
    if (ex.kind & HDRVAE_EX_ALLREDUCE_F64) {
      HDRVAE_REQUIRE(ex.allreduce_count <= 64, "rows exchange: at most 64 sums");
      for (int r = 0; r < world; ++r) HDRVAE_TRY(seg(r, 1, 0, ex.allreduce_off, ex.allreduce_count * 8));
    }
    if (ex.kind & HDRVAE_EX_ALLGATHER) {
      for (int i = 0; i < ex.n_gather; ++i) {
        const size_t n = ex.gather_bytes_per_rank[i], mine = ex.gather_off[i] + (size_t)rank * n;
        for (int r = 0; r < world; ++r)
          if (r != rank) HDRVAE_TRY(seg(r, 0, mine, mine, n));
      }
    }
    if (ex.kind & HDRVAE_EX_RAW_STATS)
      for (int r = 0; r < world; ++r) HDRVAE_TRY(seg(r, 2, 0, ex.raw_stats_off, sizeof(hdrvae_raw_stats)));
    // all blocks of the push kernel wait on flags: the grid must be co-resident (one block per SM at most)
    int blocks = (int)std::min<size_t>(std::max<size_t>(total / 32768, 1), (size_t)st->ctx->num_sms);
    HDRVAE_TRY(launch_rows_push(a, blocks, s));
    HDRVAE_TRY(launch_rows_wait(st->ws, st->pl.off_mail, world, ex.allreduce_off,
                                (ex.kind & HDRVAE_EX_ALLREDUCE_F64) ? (int)ex.allreduce_count : 0, ex.raw_stats_off,
                                (ex.kind & HDRVAE_EX_RAW_STATS) != 0, s));
  }
  return 0;
}

int hdrvae_rows_end(hdrvae_rows* st, hdrvae_stats* stats, void* stream) {
  if (st == nullptr) return 0;
  int r = 0;
  if (stats != nullptr) {
    cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
    cudaError_t e = cudaMemcpyAsync(stats, epilogue_stats_dev_ptr(st->ws + st->pl.off_epi, 1, 8 * st->pl.hl, 8 * st->pl.w),
                                    sizeof(hdrvae_stats), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) { set_error("hdrvae_rows_end: %s", cudaGetErrorString(e)); r = -1; }
  }
  delete st;
  return r;
}

int hdrvae_decode_features(hdrvae_ctx* ctx, const float* latent, int B, int h, int w, void* features, void* workspace,
                           size_t ws_bytes, void* stream) {
  HDRVAE_REQUIRE(ctx != nullptr && latent != nullptr && features != nullptr, "hdrvae_decode_features: null argument");
  HDRVAE_REQUIRE(B >= 1 && h >= 1 && w >= 1, "hdrvae_decode_features: empty latent batch");
  HDRVAE_CUDA_OK(cudaSetDevice(ctx->device));
  const Plan pl = decode_plan(ctx, B, h, w);
  HDRVAE_TRY(check_ws(pl, workspace, ws_bytes));
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  void* feat = nullptr;
  HDRVAE_TRY(run_decoder(ctx, latent, pl, reinterpret_cast<uint8_t*>(workspace), &feat, s));
  HDRVAE_CUDA_OK(cudaMemcpyAsync(features, feat, (size_t)B * 64 * h * w * 128 * (ctx->high ? 4 : 2), cudaMemcpyDeviceToDevice, s));
  return 0;
}

int hdrvae_epilogue_scratch_bytes(int B, int H, int W, size_t* bytes) {
  HDRVAE_REQUIRE(bytes != nullptr && B >= 1 && H >= 1 && W >= 1, "hdrvae_epilogue_scratch_bytes: bad argument");
  *bytes = epilogue_scratch_bytes(B, H, W);
  return 0;
}

int hdrvae_epilogue(hdrvae_ctx* ctx, const void* pre, int dtype, int B, int H, int W, const float* conv_w,
                    const float* conv_b, int mode, float expansion_factor, float ev_multiplier, float* out_bhwc,
                    hdrvae_stats* stats, float* dbg_post3, float* dbg_pre3, int32_t* dbg_argmax3, void* scratch,
                    size_t scratch_bytes, void* stream) {
  HDRVAE_REQUIRE(ctx != nullptr && pre != nullptr && conv_w != nullptr && conv_b != nullptr && out_bhwc != nullptr,
                 "hdrvae_epilogue: null argument");
  HDRVAE_REQUIRE(B >= 1 && H >= 1 && W >= 1, "hdrvae_epilogue: empty image batch");
  HDRVAE_REQUIRE(scratch != nullptr && scratch_bytes >= epilogue_scratch_bytes(B, H, W), "hdrvae_epilogue: scratch too small");
  HDRVAE_CUDA_OK(cudaSetDevice(ctx->device));
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  HDRVAE_TRY(launch_epilogue_phase_a(pre, dtype, B, H, W, conv_w, conv_b, dbg_argmax3, scratch, s));
  const size_t img = (size_t)B * H * W * 3 * sizeof(float);
  if (dbg_post3) HDRVAE_CUDA_OK(cudaMemcpyAsync(dbg_post3, epilogue_post3_ptr(scratch, B, H, W), img, cudaMemcpyDeviceToDevice, s));
  if (dbg_pre3) HDRVAE_CUDA_OK(cudaMemcpyAsync(dbg_pre3, epilogue_pre3_ptr(scratch, B, H, W), img, cudaMemcpyDeviceToDevice, s));
  return launch_epilogue_phase_b(B, H, W, mode, expansion_factor, ev_multiplier, out_bhwc, stats, scratch, s);
}

// ---- kernel-level entry points -------------------------------------------------------------------
int hdrvae_conv2d(hdrvae_ctx* ctx, const void* x, int x_dtype, int B, int H, int W, int Cin, const float* w,
                  const float* bias, int Cout, int ksize, int upsample2x, const void* residual, int res_dtype, void* y,
                  int y_dtype, int round_tf32, float* gn_partials, int* gn_chunks, int impl, void* stream,
                  const hdrvae_conv_extra* extra) {
  HDRVAE_REQUIRE(ctx && x && w && y, "hdrvae_conv2d: null argument");
  HDRVAE_REQUIRE(ksize == 1 || ksize == 3, "hdrvae_conv2d: ksize must be 1 or 3");
  HDRVAE_REQUIRE(x_dtype >= 0 && x_dtype <= 2 && y_dtype >= 0 && y_dtype <= 2 && res_dtype >= 0 && res_dtype <= 2,
                 "hdrvae_conv2d: bad dtype");
  hdrvae_conv_extra e;
  memset(&e, 0, sizeof e);
  if (extra != nullptr) e = *extra;
  if (e.x_channels > 0)
    HDRVAE_REQUIRE(e.x_channels % 8 == 0 && e.x_channels >= Cin, "hdrvae_conv2d: x_channels (%d) must be a multiple of 8 "
                   "(16-byte pixel strides for the TMA) and at least Cin (%d)", e.x_channels, Cin);
  else
    HDRVAE_REQUIRE(Cin % 64 == 0, "hdrvae_conv2d: Cin (%d) must be a multiple of 64 unless x_channels gives x's pixel stride", Cin);
  const int cout4 = (Cout + 3) / 4 * 4;     // the columns a conv with Cout % 32 != 0 stores
  if (e.y_channels > 0)
    HDRVAE_REQUIRE(e.y_chan_off >= 0 && e.y_chan_off % 4 == 0 && e.y_channels % 4 == 0 && e.y_chan_off + cout4 <= e.y_channels,
                   "hdrvae_conv2d: the output slice [%d, %d + round_up(Cout, 4) = %d) must lie in y_channels (%d), "
                   "with the offset and the stride multiples of 4", e.y_chan_off, e.y_chan_off, e.y_chan_off + cout4, e.y_channels);
  else
    HDRVAE_REQUIRE(Cout % 32 == 0 && e.y_chan_off == 0,
                   "hdrvae_conv2d: Cout (%d) must be a multiple of 32 and y_chan_off 0 unless y_channels gives y's pixel stride", Cout);
  if (e.y2 != nullptr) {
    HDRVAE_REQUIRE(e.y2_dtype == HDRVAE_F16 || e.y2_dtype == HDRVAE_BF16, "hdrvae_conv2d: y2 must be fp16 or bf16");
    if (e.y2_channels > 0)
      HDRVAE_REQUIRE(e.y2_chan_off >= 0 && e.y2_chan_off % 4 == 0 && e.y2_channels % 4 == 0 && e.y2_chan_off + cout4 <= e.y2_channels,
                     "hdrvae_conv2d: the y2 slice [%d, %d) must lie in y2_channels (%d), with the offset and the stride "
                     "multiples of 4", e.y2_chan_off, e.y2_chan_off + cout4, e.y2_channels);
    else
      HDRVAE_REQUIRE(e.y2_chan_off == 0, "hdrvae_conv2d: y2_chan_off needs y2_channels");
  }
  HDRVAE_REQUIRE(e.act >= HDRVAE_ACT_NONE && e.act <= HDRVAE_ACT_GATE, "hdrvae_conv2d: bad act (%d)", e.act);
  HDRVAE_CUDA_OK(cudaSetDevice(ctx->device));
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  hdrvae_ctx tmp;                     // owns the temporary packed operands
  tmp.device = ctx->device; tmp.num_sms = ctx->num_sms; tmp.cta_group = ctx->cta_group;
  PackedConv pc;
  int r = pack_conv(&tmp, w, bias, Cout, Cin, ksize, upsample2x != 0, 1.f, x_dtype, &pc, s);
  float* slopes = nullptr;            // the kernels read cout_pad slopes, zero-padded (as the upscaler packs them)
  if (r == 0 && e.act_slope != nullptr) {
    r = dev_alloc(&tmp, pc.cout_pad * sizeof(float), (void**)&slopes);
    if (r == 0 && (cudaMemsetAsync(slopes, 0, pc.cout_pad * sizeof(float), s) != cudaSuccess ||
                   cudaMemcpyAsync(slopes, e.act_slope, Cout * sizeof(float), cudaMemcpyDeviceToDevice, s) != cudaSuccess)) {
      set_error("hdrvae_conv2d: copying the PReLU slopes failed");
      r = -1;
    }
  }
  if (r == 0) {
    ConvIO io; io.x = x; io.y = y; io.y_dtype = y_dtype; io.residual = residual; io.res_dtype = res_dtype;
    io.round_tf32 = round_tf32 != 0; io.stats = gn_partials; io.stats_chunks = gn_chunks;
    io.x_channels = e.x_channels; io.y_channels = e.y_channels; io.y_chan_off = e.y_chan_off;
    io.y2 = e.y2; io.y2_dtype = e.y2 != nullptr ? e.y2_dtype : DT_F16; io.y2_scale = e.y2_scale != 0.f ? e.y2_scale : 1.f;
    io.y2_channels = e.y2_channels; io.y2_chan_off = e.y2_chan_off;
    io.res_scale = e.res_scale != 0.f ? e.res_scale : 1.f; io.residual2 = e.residual2;
    io.lrelu = e.lrelu; io.act_slope = slopes; io.act = e.act;
    r = run_conv(&tmp, pc, io, B, H, W, impl, s);
  }
  cudaStreamSynchronize(s);
  for (void* p : tmp.owned) cudaFree(p);
  if (r == 0) HDRVAE_CUDA_OK(cudaGetLastError());
  return r;
}

int hdrvae_conv2d_stats_chunks(int H, int W, int upsample2x) { return (upsample2x ? 4 : 1) * tiles_for(H, W); }

int hdrvae_groupnorm_silu(hdrvae_ctx* ctx, const void* x, int x_dtype, int B, int HW, int C, const float* gamma,
                          const float* beta, int apply_silu, void* y, int y_dtype, const float* gn_partials,
                          int gn_chunks, void* stream) {
  HDRVAE_REQUIRE(ctx && x && gamma && beta && y, "hdrvae_groupnorm_silu: null argument");
  HDRVAE_CUDA_OK(cudaSetDevice(ctx->device));
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const int max_chunks = std::max(1184, gn_chunks);
  void* scratch = nullptr;
  HDRVAE_CUDA_OK(cudaMalloc(&scratch, gn_scratch_bytes(B, C, max_chunks)));
  int r = gn_scratch_reset(scratch, B, max_chunks, s);
  if (gn_partials != nullptr && gn_chunks > 0)
    HDRVAE_CUDA_OK(cudaMemcpyAsync(scratch, gn_partials, (size_t)B * gn_chunks * 64 * sizeof(float), cudaMemcpyDeviceToDevice, s));
  if (r == 0)
    r = launch_groupnorm(x, x_dtype, y, y_dtype, B, HW, C, gamma, beta, apply_silu != 0, scratch, max_chunks,
                         gn_partials != nullptr ? gn_chunks : 0, s);
  cudaStreamSynchronize(s);
  cudaFree(scratch);
  return r;
}

int hdrvae_attention(hdrvae_ctx* ctx, const void* q, const void* k, const void* v, int dtype, int B, int T, void* o,
                     void* stream) {
  HDRVAE_REQUIRE(ctx && q && k && v && o && B >= 1 && T >= 1, "hdrvae_attention: bad argument");
  HDRVAE_REQUIRE(dtype == HDRVAE_BF16 || dtype == HDRVAE_F16, "hdrvae_attention: q/k/v must be bf16 or fp16");
  HDRVAE_CUDA_OK(cudaSetDevice(ctx->device));
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  // the q|k and v^T operands, then the fused kernel's key-split partials or one GEMM-level scratch chunk
  const int Tp = (T + 63) / 64 * 64;
  size_t total = 0;
  auto take = [&](size_t bytes) { size_t o = total; total += align_up(bytes, 1024); return o; };
  const size_t off_qk = take((size_t)B * Tp * 1024 * 2), off_vt = take((size_t)B * 512 * Tp * 2);
  const bool fused = attention_fused_enabled(ctx);
  const size_t ksp = attention_key_splits(T), ksplit_bytes = fused && ksp > 1 ? (size_t)B * T * (512 + 2) * 4 * ksp : 0;
  const size_t off_ksplit = take(ksplit_bytes);
  const int s_rows = score_chunk_rows(T, Tp);
  const size_t off_s = take(fused ? 0 : (size_t)s_rows * Tp * 4), off_p = take(fused ? 0 : (size_t)s_rows * Tp * 2),
               off_inv = take(fused ? 0 : (size_t)s_rows * 4);
  uint8_t* ws = nullptr;
  HDRVAE_CUDA_OK(cudaMalloc((void**)&ws, total));
  uint16_t* qk = reinterpret_cast<uint16_t*>(ws + off_qk);
  uint16_t* vt = reinterpret_cast<uint16_t*>(ws + off_vt);
  const AttnChunk chunk{reinterpret_cast<float*>(ws + off_s), ws + off_p, reinterpret_cast<float*>(ws + off_inv), s_rows};
  int r = 0;
  const float scale = 1.0f / sqrtf(512.0f);
  cudaMemsetAsync(qk, 0, (size_t)B * Tp * 1024 * 2, s);
  cudaMemsetAsync(vt, 0, (size_t)B * 512 * Tp * 2, s);
  const uint16_t* q16 = reinterpret_cast<const uint16_t*>(q);
  const uint16_t* k16 = reinterpret_cast<const uint16_t*>(k);
  const uint16_t* v16 = reinterpret_cast<const uint16_t*>(v);
  for (int b = 0; b < B && r == 0; ++b) {
    // interleave q and k rows into the [Tp][1024] operand, transpose v
    r = launch_transpose_pad(v16 + (size_t)b * T * 512, vt + (size_t)b * 512 * Tp, T, 512, Tp, s);
    if (r == 0) HDRVAE_CUDA_OK(cudaMemcpy2DAsync(qk + (size_t)b * Tp * 1024, 2048, q16 + (size_t)b * T * 512, 1024, 1024, T, cudaMemcpyDeviceToDevice, s));
    if (r == 0) HDRVAE_CUDA_OK(cudaMemcpy2DAsync(qk + (size_t)b * Tp * 1024 + 512, 2048, k16 + (size_t)b * T * 512, 1024, 1024, T, cudaMemcpyDeviceToDevice, s));
  }
  const int saved = ctx->op_dtype;
  ctx->op_dtype = dtype;
  if (r == 0) r = run_attention_core(ctx, B, T, Tp, qk, vt, o, scale, ws + off_ksplit, ksplit_bytes, chunk, s);
  ctx->op_dtype = saved;
  cudaStreamSynchronize(s);
  cudaFree(ws);
  return r;
}

int hdrvae_quantiles(const float* data, long long n, const double* q, int nq, float* out_host, void* stream) {
  HDRVAE_REQUIRE(data && q && out_host && n >= 1 && nq >= 1 && nq <= 8, "hdrvae_quantiles: bad argument (1..8 quantiles, n >= 1)");
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  unsigned long long ranks[8];
  for (int i = 0; i < nq; ++i) {
    HDRVAE_REQUIRE(q[i] >= 0.0 && q[i] <= 1.0, "hdrvae_quantiles: q must be in [0,1]");
    ranks[i] = (unsigned long long)floor(q[i] * (double)(n - 1));      // torch.quantile(..., interpolation="lower")
  }
  void* scratch = nullptr;
  HDRVAE_CUDA_OK(cudaMalloc(&scratch, quantile_scratch_bytes() + 8 * sizeof(float)));
  float* out_dev = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(scratch) + quantile_scratch_bytes());
  int r = launch_quantiles(data, n, ranks, nq, out_dev, scratch, s);
  if (r == 0) {
    cudaError_t e = cudaMemcpyAsync(out_host, out_dev, nq * sizeof(float), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) { set_error("hdrvae_quantiles: %s", cudaGetErrorString(e)); r = -1; }
  }
  cudaFree(scratch);
  return r;
}

int hdrvae_pack_half(const float* image, int B, int H, int W, int layout, uint16_t* out, void* stream) {
  HDRVAE_REQUIRE(image && out && B >= 0 && H >= 0 && W >= 0 && (layout == 0 || layout == 1), "hdrvae_pack_half: bad argument");
  return launch_pack_half(image, out, B, H, W, layout, reinterpret_cast<cudaStream_t>(stream));
}

}  // extern "C"
