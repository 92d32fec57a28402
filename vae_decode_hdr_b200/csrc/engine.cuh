// Internal declarations shared by api.cu (decoder program, C ABI) and upscaler.cu.
#pragma once
#include <string>
#include <vector>
#include <map>

#include "../../include/hdrvae.h"
#include "common.cuh"

namespace hdrvae {

// ---- kernels implemented in the other translation units -------------------------------------------
int launch_gemm_tc(const GemmParams& p, int num_sms, cudaStream_t stream);
int launch_gemm_direct(const GemmParams& p, cudaStream_t s);
void choose_tile(int H, int W, GemmParams* p);
int launch_to_f32(const void* src, int dtype, float* dst, long long n, cudaStream_t s);
int launch_pack_weight(const float* w, void* out, int out_dtype, int cout, int cin, int ks, int ntaps, int cin_pad,
                       const int* tap_mask, float scale, cudaStream_t s, int split3 = 0);
int launch_add_vectors(const float* a, const float* b, float* c, int n, cudaStream_t s);
int launch_split3(const float* x, long long x_ld, void* out, long long out_ld, long long n, int C, float scale, int order,
                  cudaStream_t s);
// Latent staging: z [B][C_lat][HW] fp32 -> NHWC [B][HW][cpad] holding C channels, with post_quant_conv applied when
// pq_w ([C][C_lat]) and pq_b ([C]) are given (otherwise C_lat == C and z is copied).
int launch_latent_to_nhwc(const float* z, void* out, int out_dtype, int B, int C, int C_lat, const float* pq_w,
                          const float* pq_b, int HW, int cpad, cudaStream_t s);
int launch_latent_rows_to_nhwc(const float* z, void* out, int out_dtype, int C, int C_lat, const float* pq_w,
                               const float* pq_b, int h, int w, int y0, int rows, int cpad, cudaStream_t s);
int launch_softmax_rows(const float* s, void* p, int p_dtype, float* inv_sum, int n_rows, int n_valid, int n_pad,
                        long long s_ld, long long p_ld, cudaStream_t st);
int launch_attn_row_parts(const float* part, int rows, int parts, int mode, float* out, cudaStream_t st);
int launch_transpose_pad(const void* in, void* out, int rows, int cols, int out_ld, cudaStream_t s);
int launch_attn_reduce_splits(const float* part, const float* inv_sum, void* out, int out_dtype, int rows, int cols,
                              int splits, cudaStream_t st);
int launch_pack_half(const float* img, uint16_t* out, int B, int H, int W, int layout, cudaStream_t s);
size_t quantile_scratch_bytes();
int launch_quantiles(const float* x, long long n, const unsigned long long* ranks_host, int nq, float* out, void* scratch,
                     cudaStream_t s);
size_t gn_scratch_bytes(int B, int C, int max_chunks);
int gn_scratch_reset(void* scratch, int B, int max_chunks, cudaStream_t s);
int launch_gn_scale_shift_from_sums(int B, int C, const float* gamma, const float* beta, void* scratch, int max_chunks,
                                    double count, cudaStream_t s, const float** scale_out, const float** shift_out);
int launch_gn_scale_shift(int B, int HW, int C, const float* gamma, const float* beta, void* scratch, int max_chunks,
                          int partial_chunks, cudaStream_t s, const float** scale_out, const float** shift_out);   // once before a scratch buffer's first use
int launch_groupnorm(const void* x, int x_dtype, void* y, int y_dtype, int B, int HW, int C, const float* gamma,
                     const float* beta, bool silu, void* scratch, int max_chunks, int partial_chunks, cudaStream_t s,
                     float in_scale = 1.f);
size_t epilogue_scratch_bytes(int B, int H, int W);
void* epilogue_raw_stats_ptr(void* scratch, int B, int H, int W);
hdrvae_stats* epilogue_stats_dev_ptr(void* scratch, int B, int H, int W);
float* epilogue_post3_ptr(void* scratch, int B, int H, int W);
float* epilogue_pre3_ptr(void* scratch, int B, int H, int W);
int launch_epilogue_phase_a(const void* pre, int dtype, int B, int H, int W, const float* conv_w, const float* conv_b,
                            int* argmax3, void* scratch, cudaStream_t s, int y_pad = 0, long long img_stride = 0);
double* gn_sums_ptr(void* scratch, int B, int C, int max_chunks);
int launch_gn_reduce_partials(void* scratch, int B, int C, int max_chunks, int n_partials, cudaStream_t s);
int launch_gn_apply_from_sums(const void* x, int x_dtype, long long x_img_stride, void* y, int y_dtype, long long y_img_stride,
                              int B, int rows_px, int C, const float* gamma, const float* beta, bool silu, void* scratch,
                              int max_chunks, double count, cudaStream_t s, float in_scale = 1.f);
int launch_epilogue_phase_a_pre(const void* pre, int dtype, int B, int H, int W, const float* conv8, const float* conv_b,
                                int* argmax3, void* scratch, cudaStream_t s, long long img_stride);
int launch_split_hi_lo(const float* w, float* w8, int k, cudaStream_t s);
int launch_epilogue_phase_b(int B, int H, int W, int mode, float factor, float ev, float* out, hdrvae_stats* host_stats,
                            void* scratch, cudaStream_t s);
int attention_key_splits(int n_keys);
int launch_attention_fused(const void* q, long long q_ld, long long q_img_stride, int n_q, const void* k, long long k_ld,
                           long long k_img_stride, int k_rows, const void* vt, long long vt_ld, long long vt_img_stride,
                           int n_keys, void* o, long long o_img_stride, int n_img, int dt, float alpha, int cta_group,
                           int num_sms, float* part, float* ml, long long part_rows, cudaStream_t s);
int launch_raw_stats_merge(const hdrvae_raw_stats* blocks, int n, hdrvae_raw_stats* dst, cudaStream_t s);

// ---- device-driven exchanges of the row-tiled decode (rows_p2p.cu) --------------------------------------------
constexpr int kRowsMaxRanks = 16;
struct RowsRawSlot { hdrvae_raw_stats s; unsigned char pad[32]; };      // 128 bytes
// lives at RowsPlan::off_mail of every rank's workspace; zero-initialised by hdrvae_peer_alloc
struct RowsMailbox {
  unsigned int arrived[64];     // [src rank]: src has reached exchange number ...
  unsigned int data[64];        // [src rank]: src's contribution to exchange number ... has landed here
  unsigned int seq;             // exchanges completed by THIS rank (advanced by the wait kernel)
  unsigned int ticket;          // block counter of the push kernel
  unsigned int pad[2];
  double sums[2][kRowsMaxRanks][64];            // [parity of the exchange number][src rank]: GroupNorm sums
  RowsRawSlot raw[2][kRowsMaxRanks];            // [parity][src rank]: HDR raw statistics blocks
};
struct RowsSegment {
  unsigned long long dst_off, src_off;          // byte offsets into the peer's / this rank's workspace
  unsigned int bytes;                           // multiple of 16
  int peer;                                     // destination rank
  int kind;                                     // 0 plain, 1 GroupNorm sums -> table slot, 2 raw statistics -> table slot
  int pad;
};
struct RowsPushArgs {
  uint8_t* ws;
  uint8_t* peers[kRowsMaxRanks];                // every rank's workspace as mapped into this process (own included)
  unsigned long long off_mail;
  int rank, world, n_seg, pad;
  RowsSegment seg[72];
};
int launch_rows_push(const RowsPushArgs& a, int blocks, cudaStream_t s);
int launch_rows_wait(uint8_t* ws, size_t off_mail, int world, size_t allreduce_off, int allreduce_count, size_t raw_off,
                     bool has_raw, cudaStream_t s);

// ---- per-op device timing (diagnostics; enabled by hdrvae_profile_begin) -----------------------------
struct ProfEntry { std::string name; cudaEvent_t e0, e1; double flops, bytes; };
extern bool g_prof_on;
extern std::vector<ProfEntry> g_prof;
struct ProfScope {
  cudaStream_t s; bool on;
  ProfScope(const char* name, double flops, double bytes, cudaStream_t st) : s(st), on(g_prof_on) {
    if (!on) return;
    ProfEntry e; e.name = name; e.flops = flops; e.bytes = bytes;
    cudaEventCreate(&e.e0); cudaEventCreate(&e.e1);
    cudaEventRecord(e.e0, s);
    g_prof.push_back(e);
    idx = g_prof.size() - 1;
  }
  ~ProfScope() { if (on) cudaEventRecord(g_prof[idx].e1, s); }
  size_t idx = 0;
};

// ---- packed operands --------------------------------------------------------------------------
struct PackedConv {
  void* w[4] = {nullptr, nullptr, nullptr, nullptr};  // [Cout][ntaps*cin_pad] K-major; 4 phase matrices when upsample
  float* bias = nullptr;
  int cin = 0, cin_pad = 0, cout = 0, ks = 0;
  int cout_pad = 0;          // cout rounded up to 32: columns the GEMM computes (bias is allocated to this length)
  int w_dtype = DT_F16;      // operand type of this conv (DT_F32 = tf32 MMA on the raw fp32 stream)
  int kmul = 1;              // 3: "precision high" — every tap's K range is [hi | hi | lo] (3 * cin_pad), the activations
                             //    come as [hi | lo | hi] (DT_F16X3)
  bool upsample = false;
};
struct NormW {
  float* gamma = nullptr;
  float* beta = nullptr;
  int C = 0;
};
struct ResW {
  NormW n1, n2;
  PackedConv c1, c2, nin;
  PackedConv nin_x16;        // nin_shortcut weights x 2^4 (its operand is the 2^-4 scaled 16-bit copy of x): the form that is
                             // fused into conv2 as extra K blocks
  float* bias_c2_nin = nullptr;   // conv2.bias + nin_shortcut.bias
  bool has_nin = false;
  bool dual_out = false;     // the block's output is also the operand of the next (upsample) conv: emit the scaled 16-bit copy
};


}  // namespace hdrvae

using namespace hdrvae;

struct hdrvae_ctx {
  int device = 0;
  int num_sms = 148;
  bool loaded = false;
  int conv_impl = HDRVAE_CONV_TCGEN05;
  int op_dtype = DT_F16;                          // 16-bit tensor-core operand type (HDRVAE_PRECISION_*)
  bool high = false;                              // HDRVAE_PRECISION_HIGH: fp16 hi + lo split operands (3 MMAs per product)
  int cta_group = 0;                              // 0 = default (CTA pairs), 1 / 2 forced
  struct GraphEntry { int seg, B, h, w, mode, conv_impl, cta_group; float factor, ev; void* ws; cudaGraphExec_t exec; long long n_kernels; };
  std::vector<GraphEntry> graphs;                 // captured whole-decode CUDA graphs (hdrvae_decode)
  std::vector<GraphEntry> seen;                   // keys decoded once already (capture happens on the second use)
  bool use_graphs = true;
  std::vector<void*> owned;                       // every device allocation of the context
  std::map<std::string, float*> raw;              // fp32 device copies of the state dict
  std::map<std::string, std::vector<int64_t>> shapes;
  int c_z = 16;                                   // input channels of conv_in (Flux 16, SD1.x / SDXL 4)
  int c_lat = 16;                                 // channels of the caller's latent: post_quant_conv's input, else c_z
  const float* pq_w = nullptr;                    // post_quant_conv (1x1, fp32 [c_z][c_lat] + bias [c_z]) or null
  const float* pq_b = nullptr;
  PackedConv conv_in, qk, vproj, proj_out;
  NormW attn_norm, norm_out;
  ResW mid1, mid2, up[4][3];
  PackedConv upsample[4];
  PackedConv conv_out_tc;                         // conv_out as an 8-row fp16 operand: rows 0-2 hi, 4-6 lo of the fp32 weights
  float* conv_out_w = nullptr;                    // fp32 OIHW [3][128][3][3]
  float* conv_out_b = nullptr;
};

namespace hdrvae {

struct ConvIO {
  const void* x = nullptr;        // [B,H,W,cin_pad], element type = pc.w_dtype
  void* y = nullptr;              // [B,OH,OW,cout]
  int y_dtype = DT_F32;
  float y_scale = 1.f;            // multiplier of a 16-bit y (un-normalised tensors are stored scaled by 2^-4)
  const void* residual = nullptr; // y's layout
  int res_dtype = DT_F32;
  bool round_tf32 = false;
  void* y2 = nullptr;             // optional scaled 16-bit copy of y (operand of a conv that reads y un-normalised)
  int y2_dtype = DT_F16;
  float y2_scale = 1.f;
  float alpha = 1.f;              // accumulator scale (undoes the operand scale of a y2-fed conv)
  float* stats = nullptr;         // GroupNorm partials of y, or null
  int* stats_chunks = nullptr;    // out: partial chunks per image written
  // row tiling: x / y (and residual, y2) are slabs with this many halo rows stored above and below the H / OH rows;
  // the pointers address the slab start
  int x_pad = 0, y_pad = 0;
  // channel-sliced tensors (the upscaler's dense-block concat buffers): pixel strides in elements when they differ
  // from the conv's own channel counts (0: dense), and the first channel written
  int x_channels = 0;             // pixel stride of x; the conv reads the first pc.cin channels
  int y_channels = 0, y_chan_off = 0;     // pixel stride / channel offset of y (residuals share y's addressing)
  int y2_channels = 0, y2_chan_off = 0;   // same for y2
  float res_scale = 1.f;          // y = alpha * conv + bias + res_scale * residual + residual2, then LeakyReLU
  const float* residual2 = nullptr;
  float lrelu = 0.f;              // LeakyReLU slope (0: none)
  int n_store = 0;                // channels of y stored (multiple of 4; 0: all)
  // fused 1x1 conv of a second tensor (slab form): y += conv1x1(x2, *pc2); x2 has x's spatial shape / halo rows and
  // pc2->cin_pad channels per pixel (dense); `bias` replaces the conv's own bias when set
  const void* x2 = nullptr;
  const PackedConv* pc2 = nullptr;
  const float* bias = nullptr;
  // GroupNorm + SiLU of x applied inside the conv (GemmParams::xf_*): per-(image, channel) scale / shift, the scale of a
  // scaled 16-bit x, and which rows of x are image rows (row tiling: a border rank's outer halo row is padding)
  const float* xf_scale = nullptr;
  const float* xf_shift = nullptr;
  float xf_in_scale = 1.f;
  int xf_y_lo = 0, xf_y_hi = -1;  // -1: H
};

// true when run_conv would take the slab form of the tensor-core kernel (needed by the fused nin_shortcut path)
bool conv_takes_slab(const PackedConv& pc, const ConvIO& io, int H, int W, int impl);

int dev_alloc(hdrvae_ctx* ctx, size_t bytes, void** out);
int pack_conv(hdrvae_ctx* ctx, const float* w, const float* bias, int cout, int cin, int ks, bool upsample,
              float scale, int w_dtype, PackedConv* pc, cudaStream_t s, bool split3 = false);
int run_conv(hdrvae_ctx* ctx, const PackedConv& pc, const ConvIO& io, int B, int H, int W, int impl, cudaStream_t s);

}  // namespace hdrvae
