// comic_internal.cuh -- handle, error plumbing and workspace carving shared by
// the translation units of libcomic_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>

#include "../../include/comic_b200.h"
#include "gemm_f32.cuh"
#include "gemm_tc.cuh"

namespace comic {

void set_error(const char* fmt, ...);

#define COMIC_CHECK_CUDA(expr)                                                         \
  do {                                                                                 \
    cudaError_t _e = (expr);                                                           \
    if (_e != cudaSuccess) {                                                           \
      comic::set_error("%s:%d CUDA error %s: %s", __FILE__, __LINE__, #expr,           \
                       cudaGetErrorString(_e));                                        \
      return COMIC_E_CUDA;                                                             \
    }                                                                                  \
  } while (0)

#define COMIC_REQUIRE(cond, code, ...)                                                 \
  do {                                                                                 \
    if (!(cond)) {                                                                     \
      comic::set_error(__VA_ARGS__);                                                   \
      return (code);                                                                   \
    }                                                                                  \
  } while (0)

// One inception block of the encoder plan.
struct BlockDesc {
  int cin, b0, b1a, b1b, b2a, b2b, b3;
  int conv[6];   // indices into the 57-conv table: b0, b1a, b1b, b2a, b2b, b3
};

constexpr int kNumBlocks = 9;

struct Packed {
  float* outq = nullptr;       // [R, LQ]  = [W_o | 0-pad | W_q]
  float* outq_bias = nullptr;  // [LQ]
  float* bn_scale[COMIC_NUM_CONVS];
  float* bn_shift[COMIC_NUM_CONVS];
  float* grp_w[kNumBlocks];      // [cin, b0+b1a+b2a]
  float* grp_scale[kNumBlocks];
  float* grp_shift[kNumBlocks];
  // tensor-core path: B^T hi/lo panels + TMA descriptors
  tc::TcWeight tc_conv[COMIC_NUM_CONVS];
  tc::TcWeight tc_grp[kNumBlocks];
  tc::TcWeight tc_lstm, tc_outq, tc_mem, tc_val, tc_init;
  // GRU cell: [gates/kernel | candidate/kernel x-rows ; 0] panel [W+A+R, 3R] of the gate GEMM, and the tensor-path packs
  // of that panel and of the candidate kernel's h-rows [R, R]
  float* gru_gx = nullptr;
  tc::TcWeight tc_gru_g, tc_gru_c;
  tc::TcWeight tc_stem_s2d;      // Conv2d_1a_7x7 as a 4x4 conv over the space-to-depth image: W2 [4,4,16,64]
};

}  // namespace comic

namespace comic {
enum Tag { T_CONV = 0, T_POOL, T_PROJECT, T_INIT, T_GATES, T_LSTM, T_LQ, T_SCORES, T_CTX, T_BEAM, T_FINAL, T_MISC, T_PERSIST, T_COUNT };
constexpr int kMaxProfEvents = 16384;
}  // namespace comic

struct comic_handle_s {
  comic_cfg_t cfg;
  int dev = 0;
  int num_sms = 148;
  int R, W, H, C, M, E, V, Vp, A, VAL, LQ, KX;
  comic_weights_t w;
  int cell = COMIC_CELL_LSTM;              // comic_set_rnn_cell
  int fm_tap = COMIC_FM_MIXED_4F;          // comic_set_fm_endpoint
  const float* gru_cand_kernel = nullptr;  // GRU candidate/{kernel [W+A+R, R], bias [R]} (comic_bind_gru_candidate);
  const float* gru_cand_bias = nullptr;    // gates/{kernel, bias} travel in w.lstm_kernel / w.lstm_bias
  bool bound = false, cnn_bound = false;
  bool sized = false;                      // a packed / workspace size was handed out (laid out for `cell`)
  int precision = 1;   // 0: fp32 FFMA everywhere; 1: tcgen05 split-precision GEMMs with M >= 128; 2: 1 + tanh.approx
  int fused_min_images = 48;   // fused attention kernel (one CTA per image) from this batch size on
  int attn2_min_images = 12;   // streaming kernel (attention2.cuh) from this batch size on while fused_min_images is at its
                               // default: its slice-granular work split fills the SMs from ~12 images (39 vs 48 us at 12
                               // images x 3 beams, 33 vs 48 at 25, profiles/r08c_attn_small_batch.txt); an explicit
                               // fused_min_images moves both thresholds
  int tma_a = 1;               // bit 0: [logits | query] GEMM, bit 1: gate GEMM read their A operand as bf16 planes through
                               // TMA (no gather / split in the GEMM's loader warps)
  int attn2 = 1;               // streaming attention kernel (attention2.cuh) where it applies: tied values, add_LN, softmax,
                               // R = 512, 8 heads, k <= 3, no attention-map dropout; 0 = always attention.cuh
  int attn2_state = 0;         // 0: score bound of the bound weights not checked yet; 1: within range; -1: too large
  float* attn2_host = nullptr; // pinned [8]: per-head score bound read back once per weight binding
  int persist_trace = 0;       // record per-phase clock stamps of the persistent loop (diagnostics)
  long long* last_trace = nullptr;
  int last_trace_steps = 0;
  int persist_watchdog_ms = 2000;   // grid-barrier watchdog of the persistent loop (0 = disabled)
  int persist_max_rows = 32;   // whole decode loop as one cooperative kernel up to this many rows (0 = off)
  int tc_splitk = 3;           // bit 0: gate GEMM, bit 1: [logits | query] GEMM -- split-K for tensor-path decoder GEMMs of one M tile (tc_ksplit below); COMIC_OPT_TC_SPLITK
  int tc_min_rows = 64;        // GEMMs / convs with at least this many rows take the tensor path (precision >= 1); half-empty
                               // M tiles still beat the FFMA kernel (batch 25-32 beam-3: gate GEMM 37 -> 29 us, r02p)
  int stem_s2d = 2;            // tensor path stem conv: 2 = space-to-depth planes, im2col tile built from a shared-memory
                               // halo patch; 0 = 7x7/2 gather from the fp32 NHWC4 image
  int enc_chunk[3] = {256, 512, 512};  // images per encoder chunk: stem / 28x28 blocks / 14x14 + 7x7 blocks (measured r01p:
                                       // the GEMMs are L2->SM bound, not HBM bound, so fewer, longer launches win over L2 residency)
  comic::Packed pk;
  int64_t launches = 0;
  // optional per-kernel-class device timing (bench.py roofline): CUDA events
  // recorded on the launching stream around every launch of the enabled tags.
  uint32_t prof_mask = 0;
  cudaEvent_t* prof_ev = nullptr;   // 2 * kMaxProfEvents
  int* prof_tag = nullptr;
  int prof_used = 0;
};

namespace comic {
// Counts a launch and, when its tag is enabled, brackets it with events.
struct Prof {
  comic_handle_t h;
  cudaStream_t st;
  int slot;
  Prof(comic_handle_t h_, int tag, cudaStream_t st_, int n = 1) : h(h_), st(st_), slot(-1) {
    h->launches += n;
    if (((h->prof_mask >> tag) & 1u) && h->prof_ev && h->prof_used < kMaxProfEvents) {
      slot = h->prof_used++;
      h->prof_tag[slot] = tag;
      cudaEventRecord(h->prof_ev[2 * slot], st);
    }
  }
  ~Prof() {
    if (slot >= 0) cudaEventRecord(h->prof_ev[2 * slot + 1], st);
  }
};
}  // namespace comic

namespace comic {

// Bump allocator over a caller-provided workspace; with base == nullptr it only
// measures.
struct Carver {
  char* base;
  size_t off = 0;
  explicit Carver(void* b) : base(static_cast<char*>(b)) {}
  template <typename T>
  T* take(size_t n) {
    size_t bytes = (n * sizeof(T) + 255) & ~size_t(255);
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += bytes;
    return p;
  }
};

inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

// Carve + (unless dry) fill one tensor-path weight pack from W[K][N] (row stride ldw).
int pack_tc_weight(comic_handle_t h, Carver& cv, const float* W, int K, int N, int ldw, int cin_src, int cin_dst,
                   tc::TcWeight& out, cudaStream_t st, bool dry);
inline bool use_tc(comic_handle_t h, const tc::TcWeight& w, int M) { return h->precision >= 1 && w.ready && M >= h->tc_min_rows; }
// Split-K factor of a tensor-path decode-step GEMM that is far from filling the chip (33..~400 rows: batch 25 x beam 3 = 75
// rows is the reference's default inference shape, src/infer.py:72).  One 128-row tile per 128 columns leaves 16 of 148
// SMs walking 20 K blocks at ~1.3 us each; cutting K puts (tiles x ranges) CTAs on the chip with >= 2 K blocks each.
inline int tc_ksplit_shape(int num_sms, int M, int N, int K) {
  const int nk = (K + 63) / 64, tiles = ((M + 127) / 128) * ((N + 127) / 128);
  int ks = num_sms / tiles;
  if (ks > nk / 2) ks = nk / 2;
  if (ks > 8) ks = 8;
  return ks < 2 ? 1 : ks;
}
inline int tc_ksplit(comic_handle_t h, int M, int N, int K, int which) {   // which: 1 = gate GEMM, 2 = [logits | query]
  if (!(h->tc_splitk & which)) return 1;
  if (which == 2 && M > 128) return 1;      // [logits | query] (8 K blocks): the extra reduce launch costs more than the split saves
  return tc_ksplit_shape(h->num_sms, M, N, K);
}
// Decode-step GEMMs: with the K split the tensor path also wins from 33 rows on (batch 16 x beam 3: gate GEMM 22.9 -> 14.9 us,
// profiles/r12e_*); 32 rows and fewer belong to the persistent loop / the FFMA kernel.
inline bool use_tc_step(comic_handle_t h, const tc::TcWeight& w, int M, int N, int K, int which) {
  return use_tc(h, w, M) || (h->precision >= 1 && w.ready && M > 32 && tc_ksplit(h, M, N, K, which) > 1);
}

// Attention end points (COMIC_FM_*, in network order): channels and side of each.
constexpr int kNumFmTaps = 9;
constexpr int kFmTapC[kNumFmTaps] = {480, 512, 512, 512, 528, 832, 832, 832, 1024};
constexpr int kFmTapS[kNumFmTaps] = {14, 14, 14, 14, 14, 14, 7, 7, 7};
// Encoder blocks (block_table() order) whose output is an end point: Mixed_4b..4f = blocks 2..6, Mixed_5b / 5c = 7 / 8.
inline int fm_tap_block(int tap) {
  return (tap >= COMIC_FM_MIXED_4B && tap <= COMIC_FM_MIXED_4F) ? tap + 1 : (tap >= COMIC_FM_MIXED_5B ? tap : -1);
}
// The config's feature map (C, M) is the selected end point's.
inline bool fm_tap_matches(comic_handle_t h) {
  return h->C == kFmTapC[h->fm_tap] && h->M == kFmTapS[h->fm_tap] * kFmTapS[h->fm_tap];
}

// encoder.cu
int encoder_workspace_bytes(comic_handle_t h, int B, size_t* bytes);
int encoder_forward(comic_handle_t h, const float* images, int B, float* fm_out, float* im_embed_out,
                    float* mixed5c_out, void* ws, size_t ws_bytes, cudaStream_t st);
int encoder_pack(comic_handle_t h, Carver& cv, cudaStream_t st, bool dry);
const BlockDesc* block_table();
const comic_conv_desc_t* conv_table();
struct EncBufs {
  float *a, *b, *t1, *t2, *p;   // ping, pong, branch temporaries (Branch_1/2 1x1 outputs), pooled input
};
void same_pads(int n, int k, int s, int* out, int* before);
int run_conv(comic_handle_t h, const float* x, int B, int H, int W, int ldx, int ci, float* dst, int ld_dst, int coff,
             int* Ho_out, int* Wo_out, cudaStream_t st);
int run_maxpool(comic_handle_t h, const float* x, float* y, int B, int H, int W, int C, int k, int s, int* Ho_out,
                int* Wo_out, cudaStream_t st);
void run_pad_c3_c4(comic_handle_t h, const float* img, float* dst, size_t npix, cudaStream_t st);
void run_avgpool_global(comic_handle_t h, const float* x, float* y, int B, int HW, int C, cudaStream_t st);
int run_block(comic_handle_t h, int bi, const float* x, float* y, int B, int S, EncBufs& eb, cudaStream_t st);

// decoder.cu
struct StepBufs {
  float* gates;        // [nz1][N][4R]
  float* lq_part;      // [nz2][N][LQ]
  float* lq;           // [N][LQ]
  float* scores;       // [N][H][M]
  float* xdense;       // [N][W+A] (input-dropout path only)
  float* ctxraw;       // [N][VAL] (context-layer path only)
  float* kstats;       // [N * M][2] per key row: mean, centred sum of squares (attention2.cuh; once per decode call)
  float* abound;       // [8] per-head bound of |score|
  float* a2_scratch;   // partial contexts / sums of images split across CTAs (attention2.cuh)
  int* a2_counters;    // [N] arrival counters of split images, zero between launches
  // TMA-staged A operands of the two decoder GEMMs (tensor path, >= 128 rows, no dropout): bf16 (hi, lo) planes of
  // x = [emb(tok) ; ctx[src] ; h[src]] (built once per step) and of h' (written by the LSTM kernel), with their tensor maps
  uint16_t *xp_hi, *xp_lo;   // [N][KX]
  uint16_t *hp_hi, *hp_lo;   // [N][R]
  ATma xmaps, hmaps;
  bool tma_a;
  float* gru;          // GRU cell only: [3][N][R] = r * h[src], u, x . candidate/kernel x-rows
};

struct StepIO {
  const float* keys;       // [B, M, R]
  const float* values;     // [B, M, VAL]
  const int* tok;          // [N]
  const int* src;          // [N] or nullptr
  int src_limit;
  const float* c_prev;     // rows indexed through src
  const float* h_prev;
  const float* ctx_prev;
  float* c_new;            // [N, R]
  float* h_new;            // [N, R]
  float* h_drop;           // [N, R] or nullptr (train): query/logits use this when set
  float* ctx_new;          // [N, A]
  float* hist_t;           // [N, H*M] or nullptr
  float* hist_scale;       // [N, H] or nullptr: streaming attention kernel only -- hist_t stays unnormalised, 1 / sum goes here
  const float* in_mask; const float* out_mask; const float* att_mask;
  float in_keep, out_keep, att_keep;
  const int* fin_count; int t; int n_rows;
  // training tape (train.cu): pre-activation gates [N,4R], pre-dropout alignments [N,H*M];
  // force_dense assembles x = [emb;ctx] into StepBufs::xdense even without an input mask
  float* gates_save; float* alpha_pre; int force_dense;
  // training with signorm attention (train.cu): keep the raw scores of the step in StepBufs::scores (sliced kernels only)
  int no_fused;
  // streaming attention (attention2.cuh): key-row statistics / score bound of `keys`, or nullptr when not prepared
  const float* kstats; const float* abound;
  float* a2_scratch; int* a2_counters;
};

int run_step(comic_handle_t h, const StepIO& io, const StepBufs& sb, int B, int k, cudaStream_t st);
int gru_init_step(comic_handle_t h, const float* x0, int B, float* part, float* gru, float* h0, float* tape, cudaStream_t st);
// Once per decode call (keys fixed): decides whether the streaming attention kernel applies to (B, k) and, if so, fills
// sb.kstats / sb.abound and points io at them.  Returns < 0 on error.
int attn2_prepare(comic_handle_t h, StepIO& io, const StepBufs& sb, int B, int k, bool masks, cudaStream_t st);
void carve_step(comic_handle_t h, Carver& cv, int N, StepBufs& sb, bool train_masks);
int decoder_workspace_bytes(comic_handle_t h, int mode, int B, int k, int T, size_t* bytes);
int decoder_pack(comic_handle_t h, Carver& cv, cudaStream_t st, bool dry);
int decoder_configure();

// persistent.cu: the whole decode loop in one cooperative launch (small row counts)
struct PersistCall {
  const float *keys, *values, *c0, *h0;
  int B, k, max_it, greedy;
  float lpw;
  float *c[2], *h[2], *ctx[2];
  float *lq, *scores, *hist;
  int *tok, *src;
  float* cum;
  uint8_t* fin;
  long long* len;
  int* fin_count;
  int *step_ids, *parents;
  float* sc;
  float* logits_out;
  unsigned* bar;   // [2]: barrier counter, abort flag
  long long* trace;   // [max_it][2][16] phase time stamps or nullptr
  float* part;        // [16][N][4R] partial gate sums (K groups of phase A)
};
bool persist_applicable(comic_handle_t h, int B, int k, bool greedy);
int decode_persistent(comic_handle_t h, const PersistCall& pc, cudaStream_t st);

}  // namespace comic
