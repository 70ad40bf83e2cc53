// attention2.cuh -- streaming multi-head additive-LN attention for one decoder step
// (MultiHeadAddLN.__call__, common/ops_rnn.py:531-565, and the context / alignment
// part of MultiHeadAttentionWrapperV3.call, common/ops_rnn.py:692-716, 741-744).
//
// Second-generation kernel for the large-batch decode loop (tied values, softmax,
// R = 512, 8 heads).  attention.cuh (one warp per key row, channels across lanes) spent
// its time in shuffle-reduction chains and load-to-use stalls (profiles/r01z_ncu_attn_*:
// 34 % short-scoreboard, issue slots 55 % busy).  Here the mapping is turned round:
//
//   * a score-warp LANE owns half a head (32 channels) of two feature-map positions, so the tanh sum is a serial
//     in-thread accumulation -- the hot loop has no shuffles -- and every operand that is not the key itself
//     (gamma-scaled queries, gamma', beta', v') is a conflict-free 128-bit shared-memory read shared by both positions;
//   * the key tensor is streamed ONCE per step: persistent CTAs (one per SM) walk a contiguous range of 4-position key
//     slices (8 KB, contiguous in HBM) staged by TMA bulk copies (cp.async.bulk + mbarrier complete_tx) through a ring
//     of STAGES shared-memory stages;
//   * 16 warps, five roles (table kRoles): NSW score warps (slice -> LN + tanh + head sums -> p = exp(score - bound));
//     kStatWarps statistics warps (per landed slice the 4 x k dot products <k_m, qc_j> that the LN variance needs, with
//     the image's centred queries held in registers -- for ALL score warps together this costs 16 shared loads and 96
//     packed FMAs per slice, where each score warp used to spend a quarter of its time on it); 2 context warps
//     (sum_m p[m] * key[m, :] from the SAME shared-memory slice -- tied values -- unnormalised weights to the history,
//     then they REFILL the stage they have just released: no producer warp, no "empty" barriers); 1 finaliser
//     (query preparation for the segment after next, per-image normalisation, the split-image combination);
//   * softmax without a max pass: |score| <= bound_h = sum_{c in head} |v_c| / |T| (tanh is
//     bounded), so p = exp(score - bound_h) cannot overflow and alpha = p / sum p equals the
//     max-subtracted form up to rounding.  The host only takes this kernel when bound_h is
//     small enough that p cannot underflow either (attn2_prepare / decoder.cu);
//   * inside a decode loop the history stays unnormalised and 1 / sum p goes to a side buffer (Args.hist_scale) that
//     the top-beam gather applies: a rescaling pass over the history costs ~3 k cycles per L2 round trip behind the
//     TMA queue (profiles/r07e) and sat on the tail of every CTA.
//
// Barriers per stage: full (TMA landed) -> statrdy (statistics published) -> scored (weights in the stage's p buffer)
// -> [context warp accumulates, requests the next slice into the stage] -> full ...
// What the clock64 traces showed on the way (profiles/r07*): a producer that also prepared queries stalled ~10 k cycles
// twice per CTA; claim counters / integer divisions per slice cost ~1 k cycles of scalar latency behind the MUFU
// queue; two statistics warps on one sub-partition starve each other; dynamic in-order claims are slower than a fixed
// round-robin share.
//
// Per-row statistics of the keys (mean, centred sum of squares) do not change during a decode
// call and are computed once per call by key_stats_kernel.
//
// Work split: the B * M / 4 key slices of a step are one sequence that is cut into gridDim.x equal contiguous
// ranges, so every SM gets the same number of slices whatever B is.  An image whose slices fall into several
// CTAs is combined by the LAST CTA to finish its part (a per-image counter): partial sum p and partial contexts
// go through a small global scratch and are added in CTA order (deterministic); the alignment history rows are
// written unnormalised and rescaled by the combining CTA.
//
// Numerics are the old kernel's: variance from (skk + sqq + 2 <k, qc>) / R, tanh(y) =
// 1 - 2 / (2^(2 log2e y) + 1) with ex2.approx / one rcp.approx per four elements.
//
// No clamp: the four reciprocals of a chunk share one MUFU.RCP through the product x0 x1 x2 x3, x = 2^y' + 1, which
// attention.cuh keeps finite with fminf(y', 30) -- one instruction per element.  Here the exponent is shifted
// instead: x'' = 2^(y' - s) + 2^-s = 2^-s x with s folded into beta' and 2^-s into v'.  Layer norm bounds the sum of
// any four normalised channels by sqrt(4 R), so sum(y') <= 2 log2e (gmax sqrt(4 R) + 4 bmax) =: Y4; any s with
// Y4 - 4 s <= 126 and 4 s <= 126 keeps the product inside the fp32 range in both directions.  key_stats_kernel
// picks the smallest such s from max |gamma|, max |beta| and reports when none exists (the host then takes the
// round-1 kernel).
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "attention.cuh"

namespace comic {
namespace a2 {

constexpr int kR = 512;             // attention width
constexpr int kH = 8;               // heads
constexpr int kD = 64;              // head width
constexpr int kPos = 4;             // positions per slice
constexpr int kSliceFloats = kPos * kR;
constexpr int kSliceBytes = kSliceFloats * 4;   // 8 KB
constexpr int kCtxWarps = 4;
constexpr float kTwoLog2e = 2.885390081777927f;
constexpr float kLog2e = 1.4426950408889634f;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_n(uint64_t* bar, uint32_t n) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(n) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
#ifndef COMIC_A2_WATCHDOG
#define COMIC_A2_WATCHDOG 0
#endif
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t done;
#if COMIC_A2_WATCHDOG
  long long t0 = clock64();
#endif
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
#if COMIC_A2_WATCHDOG
    if (!done && clock64() - t0 > (1ll << 31)) {
      printf("attn2 watchdog: block %d warp %d bar %u parity %u\n", blockIdx.x, threadIdx.x >> 5, addr, parity);
      __trap();
    }
#endif
  } while (!done);
}
// one non-blocking probe of a phase (lane-local result)
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {
  uint32_t done;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(done)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return done != 0;
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
// TMA bulk copy global -> shared (1-D, contiguous), completion signalled on an mbarrier.
__device__ __forceinline__ void tma_bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// 128-bit shared-memory load at register + immediate (volatile: stays behind the mbarrier waits and keeps the
// hand-made software pipeline order at the front-end level)
template <int IMM>
__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4+%5];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr), "n"(IMM));
  return v;
}
// Prefetch a contiguous global range into L2 (no shared-memory destination, no completion tracking).
__device__ __forceinline__ void tma_prefetch_l2(const void* gsrc, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(gsrc), "r"(bytes) : "memory");
}
__device__ __forceinline__ void named_bar(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ---------------------------------------------------------------------------------------------
// Once per decode call: per key row mean and centred sum of squares; per head score bound.
//   kstats [rows][2];  bound [0..7] = sum_{c in head} |v_c| / |T|, bound[8] = exponent shift s, bound[9] = s feasible
// One warp per row, lane owns 16 contiguous channels (same reduction order as attention.cuh).
// ---------------------------------------------------------------------------------------------
static __global__ void __launch_bounds__(256) key_stats_kernel(const float* __restrict__ keys, long long rows,
                                                               float* __restrict__ kstats, const float* __restrict__ vvec,
                                                               const float* __restrict__ temperature,
                                                               const float* __restrict__ gamma, const float* __restrict__ beta,
                                                               float* __restrict__ bound) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (blockIdx.x == 0 && threadIdx.x < 32 * kH && bound != nullptr) {
    // warp w < 8: head w
    const int hd = threadIdx.x >> 5;
    float s = fabsf(vvec[hd * kD + lane]) + fabsf(vvec[hd * kD + 32 + lane]);
    s = wsum(s);
    if (lane == 0) bound[hd] = s / fabsf(temperature[0]);
    if (hd == 0) {
      // exponent shift of the clamp-free reciprocal product (see top): bound[8] = s, bound[9] = 1 if feasible
      float gmax = 0.f, bmax = 0.f;
      for (int c = lane; c < kR; c += 32) {
        gmax = fmaxf(gmax, fabsf(gamma[c]));
        bmax = fmaxf(bmax, fabsf(beta[c]));
      }
      gmax = wmax(gmax);
      bmax = wmax(bmax);
      const float y4 = kTwoLog2e * (gmax * sqrtf(4.0f * kR) + 4.0f * bmax) * 1.0001f + 1.0f;   // small margin for rounding
      float sh = ceilf(fmaxf(0.f, (y4 - 126.0f) * 0.25f));
      if (lane == 0) {
        bound[9] = (sh <= 31.0f && y4 == y4) ? 1.0f : 0.0f;
        bound[8] = fminf(sh, 31.0f);
      }
    }
  }
  if (row >= rows) return;
  const float* kr = keys + row * kR + lane * 16;
  float4 v[4];
  float s = 0.f;
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    v[g] = ldg4(kr + g * 4);
    s += (v[g].x + v[g].y) + (v[g].z + v[g].w);
  }
  const float mean = wsum(s) * (1.0f / kR);
  float sq = 0.f;
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    float a = v[g].x - mean, b = v[g].y - mean, c = v[g].z - mean, d = v[g].w - mean;
    sq = fmaf(a, a, sq); sq = fmaf(b, b, sq); sq = fmaf(c, c, sq); sq = fmaf(d, d, sq);
  }
  sq = wsum(sq);
  if (lane == 0) {
    kstats[row * 2 + 0] = mean;
    kstats[row * 2 + 1] = sq;
  }
}

struct Args {
  const float* keys;      // [B, M, 512]; values == keys (tied)
  const float* kstats;    // [B * M, 2]
  const float* bound;     // [8]
  const float* lq;        // [N, ld_lq], query at column q_off
  int ld_lq, q_off;
  const float* gamma;
  const float* beta;
  const float* vvec;
  const float* temperature;
  float* ctx_out;         // [N, ld_ctx]
  int ld_ctx;
  float* hist_t;          // [N, 8 * M] or nullptr
  int B, M;               // M % 4 == 0
  const int* fin_count;
  int t, n_rows;
  float* scratch;         // [2 * gridDim.x][K * (512 + 8)]: partial contexts / sums of images split across CTAs
  int* counters;          // [B], zero between launches: parts of an image that have arrived
  float* hist_scale;       // optional [n_rows][8]: when set, hist_t keeps the UNNORMALISED weights and 1 / sum goes here (the
                           // consumer multiplies: attn_top_gather_kernel); when null the history rows are rescaled in place
  long long* trace;       // diagnostics (COMIC_A2_TRACE builds): [grid][warps][kTraceSlices][8] clock64 stamps, or nullptr
};
constexpr int kTraceSlices = 256;
#ifndef COMIC_A2_TRACE
#define COMIC_A2_TRACE 0
#endif
#ifndef COMIC_A2_L2_AHEAD
#define COMIC_A2_L2_AHEAD 0       // key slices prefetched into L2 ahead of the shared-memory ring (0 = off)
#endif
#ifndef COMIC_A2_STREAM_ONLY
#define COMIC_A2_STREAM_ONLY 0    // diagnostics: consumers only wait and release (times the key stream alone; outputs garbage)
#endif
#if COMIC_A2_TRACE
#define A2_STAMP(slot) do { if (trc != nullptr && tn < kTraceSlices && lane == 0) trc[tn * 8 + (slot)] = clock64(); } while (0)
#else
#define A2_STAMP(slot) do { } while (0)
#endif

constexpr int kCtxWarps2 = 2;      // context warps of the kernel below (each takes every 2nd slice)
#ifndef COMIC_A2_NSW
#define COMIC_A2_NSW 10           // score warps
#endif
#ifndef COMIC_A2_STATW
#define COMIC_A2_STATW 3
#endif
static_assert(COMIC_A2_STATW == 2 || COMIC_A2_STATW == 3, "two or three statistics warps");
constexpr int kStatWarps = COMIC_A2_STATW;      // LN-statistics warps (warp i takes slices i, i + kStatWarps, ...)

template <int K, int NSW, int STAGES>
struct Layout {
  // warps: NSW score | 2 context | 1 finaliser | 1 TMA producer + query preparation
  static constexpr int kWarps = NSW + kCtxWarps2 + 1 + kStatWarps;
  static constexpr int kThreads = kWarps * 32;
  // byte offsets into dynamic shared memory (base 1024-aligned)
  static constexpr int ring = 0;
  static constexpr int consts = ring + STAGES * kSliceBytes;       // gamma' | beta' | v' (pair order)   [3][512]
  static constexpr int qbuf = consts + 3 * kR * 4;                 // [2][ qc [K][512] | qg [K][512] ]
  static constexpr int qstat = qbuf + 2 * 2 * K * kR * 4;          // [2][K][2]  sqq, sum qc
  static constexpr int ssum = qstat + 2 * K * 2 * 4;               // [K][8] 1 / sum p of the image being finalised
  static constexpr int part = (ssum + 2 * K * kH * 4 + 15) & ~15;      // [2][K * 520]: the context warps' partial sums of one image segment
  static constexpr int bars = part + kCtxWarps2 * K * (kR + kH) * 4;   // per context warp: [K][512] context partials | [K][8] sum p      // full[S] scored[S] empty[S] qfull[2] qempty[2] pempty[2] imgdone partfree | next slice
  static constexpr int pbuf = (bars + (4 * STAGES + 8) * 8 + 8 + 15) & ~15;   // [STAGES][K][8][4]: unnormalised weights of the slice in each stage
  static constexpr int sbuf = pbuf + STAGES * K * kH * kPos * 4;             // [STAGES][4 positions] x {var_0 + eps, var_1 + eps, var_2 + eps, -mean}
  static constexpr int kStatBytes = 4 * 16;
  static __host__ __device__ size_t bytes(int) { return (size_t)sbuf + (size_t)STAGES * kStatBytes; }
};

// Pass 2 works on chunks of four channels, software-pipelined by hand: `front4` turns staged operands into 2^y' for
// the K beams of ONE position (FMA + MUFU.EX2), `back4` folds them into the head sums (FMA + one MUFU.RCP per beam).
// The caller alternates the two positions of a lane so that the exponentials of one are in flight while the other's
// are consumed.
// ea[j] = (2^y0, 2^y2), eb[j] = (2^y1, 2^y3)
// Timing experiments (harness builds only; results are wrong): COMIC_A2_KNOCK bit 0: no MUFU in pass 2 (cheap FP
// stand-ins), bit 1: pass 1 dot products skipped, bit 2: pass 2 skipped.
#ifndef COMIC_A2_KNOCK
#define COMIC_A2_KNOCK 0
#endif
#if COMIC_A2_KNOCK & 1
#define A2_EX2(x) ((x) * 1.0001f)
#define A2_RCP(x) ((x) * 0.5f)
#else
#define A2_EX2(x) ex2_approx(x)
#define A2_RCP(x) rcp_approx(x)
#endif
template <int K>
__device__ __forceinline__ void front4(const float4 k, const float4 g, const float4 b, const float4 (&q)[K], const float2 nmu,
                                       const float (&rstd)[K], float2 (&ea)[K], float2 (&eb)[K]) {
  const float2 kg01 = __fmul2_rn(__fadd2_rn(make_float2(k.x, k.y), nmu), make_float2(g.x, g.y));
  const float2 kg23 = __fmul2_rn(__fadd2_rn(make_float2(k.z, k.w), nmu), make_float2(g.z, g.w));
  float2 y01[K], y23[K];
#pragma unroll
  for (int j = 0; j < K; ++j) {
    const float2 r2 = make_float2(rstd[j], rstd[j]);
    y01[j] = __ffma2_rn(__fadd2_rn(kg01, make_float2(q[j].x, q[j].y)), r2, make_float2(b.x, b.y));
    y23[j] = __ffma2_rn(__fadd2_rn(kg23, make_float2(q[j].z, q[j].w)), r2, make_float2(b.z, b.w));
  }
#pragma unroll
  for (int j = 0; j < K; ++j) {
    ea[j] = make_float2(A2_EX2(y01[j].x), A2_EX2(y23[j].x));
    eb[j] = make_float2(A2_EX2(y01[j].y), A2_EX2(y23[j].y));
  }
}
template <int K>
__device__ __forceinline__ void back4(const float4 vv, const float2 (&ea)[K], const float2 (&eb)[K], float (&out)[K], const float c0) {
  const float2 one2 = make_float2(c0, c0);                   // 2^-s (1 when no exponent shift is needed)
#pragma unroll
  for (int j = 0; j < K; ++j) {
    const float2 xa = __fadd2_rn(ea[j], one2), xb = __fadd2_rn(eb[j], one2);
    const float2 p = __fmul2_rn(xa, xb);                     // (x0 x1, x2 x3)
    // vv is stored as (v1, v3, v0, v2) * -2:  n = (x0 v1 + x1 v0, x2 v3 + x3 v2)
    const float2 n = __ffma2_rn(xa, make_float2(vv.x, vv.y), __fmul2_rn(xb, make_float2(vv.z, vv.w)));
    const float rp = A2_RCP(p.x * p.y);
    out[j] = fmaf(rp, fmaf(p.x, n.y, p.y * n.x), out[j]);
  }
}
// Operands of one chunk for the two positions of a lane: keys of row A / row A + 2 (4 KB apart in the slice), gamma',
// beta', v' and the K gamma-scaled queries.
template <int K>
struct Chunk2 {
  float4 ka, kb, g, b, v;
  float4 q[K];
};
template <int K>
__device__ __forceinline__ void chunk2_load(Chunk2<K>& c, uint32_t ka, uint32_t ca, uint32_t qa) {
  c.ka = lds128<0>(ka);
  c.kb = lds128<2 * kR * 4>(ka);
  c.g = lds128<0>(ca);
  c.b = lds128<kR * 4>(ca);
  c.q[0] = lds128<0>(qa);
  if (K > 1) c.q[K > 1 ? 1 : 0] = lds128<kR * 4>(qa);
  if (K > 2) c.q[K > 2 ? 2 : 0] = lds128<2 * kR * 4>(qa);
  c.v = lds128<2 * kR * 4>(ca);
}

// role << 4 | index, per warp (see "Warp roles" in the kernel)
#ifndef COMIC_A2_LAYOUT
#define COMIC_A2_LAYOUT 1
#endif
#define A2S(i) (0x00 | (i))
#define A2C(i) (0x10 | (i))
#define A2F 0x20
#define A2T(i) (0x30 | (i))
#if COMIC_A2_STATW == 2 && COMIC_A2_NSW == 11
#if COMIC_A2_LAYOUT == 0
// sub-partitions: 0: s s s ctx1 | 1: s s s fin | 2: s s s stat0 | 3: s s ctx0 stat1
__device__ constexpr unsigned char kRoles[16] = {A2S(0), A2S(1), A2S(2), A2S(3), A2S(4), A2S(5), A2S(6), A2S(7),
                                                 A2S(8), A2S(9), A2S(10), A2C(0), A2C(1), A2F, A2T(0), A2T(1)};
#else
// sub-partitions: 0: s s s ctx0 | 1: s s s ctx1 | 2: s s s stat0 | 3: s s stat1 fin
__device__ constexpr unsigned char kRoles[16] = {A2S(0), A2S(1), A2S(2), A2S(3), A2S(4), A2S(5), A2S(6), A2S(7),
                                                 A2S(8), A2S(9), A2S(10), A2T(1), A2C(0), A2C(1), A2T(0), A2F};
#endif
#elif COMIC_A2_STATW == 3 && COMIC_A2_NSW == 10
#if COMIC_A2_LAYOUT == 0
// sub-partitions: 0: s s s fin | 1: s s s stat0 | 2: s s ctx0 stat1 | 3: s s ctx1 stat2
__device__ constexpr unsigned char kRoles[16] = {A2S(0), A2S(1), A2S(2), A2S(3), A2S(4), A2S(5), A2S(6), A2S(7),
                                                 A2S(8), A2S(9), A2C(0), A2C(1), A2F, A2T(0), A2T(1), A2T(2)};
#else
// sub-partitions: 0: s s s stat0 | 1: s s s stat1 | 2: s s stat2 ctx0 | 3: s s ctx1 fin
__device__ constexpr unsigned char kRoles[16] = {A2S(0), A2S(1), A2S(2), A2S(3), A2S(4), A2S(5), A2S(6), A2S(7),
                                                 A2S(8), A2S(9), A2T(2), A2C(1), A2T(0), A2T(1), A2C(0), A2F};
#endif
#else
#error "attention2: no warp-role table for this COMIC_A2_NSW / COMIC_A2_STATW"
#endif
#undef A2S
#undef A2C
#undef A2F
#undef A2T

template <int K, int NSW, int STAGES>
__global__ void __launch_bounds__((NSW + kCtxWarps2 + 1 + kStatWarps) * 32, 1) attn2_kernel(const Args a) {
#if COMIC_A2_TRACE
  const long long t_entry = clock64();
  unsigned long long g_entry;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g_entry));
#endif
  using L = Layout<K, NSW, STAGES>;
  extern __shared__ __align__(1024) unsigned char smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int M = a.M;
  const int spi = M / kPos;                                   // slices per image
  float* sm_c = reinterpret_cast<float*>(smem + L::consts);
  float* sm_q = reinterpret_cast<float*>(smem + L::qbuf);
  float* sm_qs = reinterpret_cast<float*>(smem + L::qstat);
  float* sm_inv = reinterpret_cast<float*>(smem + L::ssum);
  float* sm_part = reinterpret_cast<float*>(smem + L::part);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + L::bars);
  uint64_t* scored = full + STAGES;
  uint64_t* empty = scored + STAGES;
  uint64_t* qfull = empty + STAGES;
  uint64_t* qempty = qfull + 2;
  uint64_t* pempty = qempty + 2;
  uint64_t* imgdone = pempty + 2;
  uint64_t* partfree = imgdone + 1;
  unsigned char* sm_st = smem + L::sbuf;
  uint64_t* statrdy = partfree + 1;                           // [STAGES] (after the 8 single barriers)
  float* sm_p = reinterpret_cast<float*>(smem + L::pbuf);     // [STAGES][K][8][4]
  constexpr int kPStage = K * kH * kPos;                      // floats per stage in sm_p

  // this CTA's contiguous range of the step's slice sequence; (b0, sl0) = image / slice of its first slice
  const long long T_all = (long long)a.B * spi;
  const int G = (int)gridDim.x;
  const long long g_lo = T_all * blockIdx.x / G, g_hi = T_all * (blockIdx.x + 1) / G;
  const int n_g = (int)(g_hi - g_lo);
  const int b0 = (int)(g_lo / spi), sl0 = (int)(g_lo - (long long)b0 * spi);
  const int n_seg = (sl0 + n_g + spi - 1) / spi;             // image segments in the range (only the first / last can be partial)
  auto seg_lo = [&](int ii) { return ii == 0 ? sl0 : 0; };
  auto seg_hi = [&](int ii) { const int r = sl0 + n_g - ii * spi; return r < spi ? r : spi; };
  // Processing order: the LAST segment first, then segments 0, 1, ...  The two segments that can be parts of images
  // shared with the neighbouring CTAs are thus finished (and combined) early, behind the whole images that follow.
  const int len_last = (n_seg >= 2) ? seg_hi(n_seg - 1) : 0;       // slices of the segment processed first (it starts at slice 0)
  auto seg_of = [&](int pos) { return len_last > 0 ? (pos == 0 ? n_seg - 1 : pos - 1) : pos; };

  // request slice sl of image b0 + ii into stage s (one TMA bulk copy of the 4 key rows)
  auto request_slice = [&](int s, int ii, int sl) {
    const size_t row0 = ((size_t)(b0 + ii) * spi + sl) * kPos;
    mbar_arrive_expect_tx(&full[s], kSliceBytes);
    tma_bulk_g2s(smem + L::ring + s * kSliceBytes, a.keys + row0 * kR, kSliceBytes, &full[s]);
  };

  if (tid == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&scored[s], 1);
      mbar_init(&empty[s], 1);
      mbar_init(&statrdy[s], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&qfull[i], 1);
      mbar_init(&qempty[i], spi);          // one arrival per scored slice of the image
      mbar_init(&pempty[i], 1);
    }
    mbar_init(imgdone, kCtxWarps2);
    mbar_init(partfree, 1);
    fence_barrier_init();
  }
  // LN constants: gamma' = gamma * 2 log2 e, beta' = beta * 2 log2 e - s, v' = -2 v 2^-s in pair order (v1, v3, v0, v2)
  const float eshift = a.bound[8];                            // exponent shift s (integer valued, 0 for ordinary weights)
  const float escale = exp2f(-eshift);                        // 2^-s, exact
  for (int c4 = tid; c4 < kR / 4; c4 += L::kThreads) {
    const float4 g4 = ldg4(a.gamma + c4 * 4), b4 = ldg4(a.beta + c4 * 4), v4 = ldg4(a.vvec + c4 * 4);
    *reinterpret_cast<float4*>(sm_c + c4 * 4) = make_float4(g4.x * kTwoLog2e, g4.y * kTwoLog2e, g4.z * kTwoLog2e, g4.w * kTwoLog2e);
    *reinterpret_cast<float4*>(sm_c + kR + c4 * 4) = make_float4(b4.x * kTwoLog2e - eshift, b4.y * kTwoLog2e - eshift,
                                                                 b4.z * kTwoLog2e - eshift, b4.w * kTwoLog2e - eshift);
    const float vs = -2.0f * escale;
    *reinterpret_cast<float4*>(sm_c + 2 * kR + c4 * 4) = make_float4(vs * v4.y, vs * v4.w, vs * v4.x, vs * v4.z);
  }
  __syncthreads();
  if (a.fin_count != nullptr && a.t > 0 && a.fin_count[a.t - 1] >= a.n_rows) return;
  if (n_g == 0) return;
#if COMIC_A2_TRACE
  long long* trc = a.trace ? a.trace + ((size_t)blockIdx.x * L::kWarps + warp) * kTraceSlices * 8 : nullptr;
  int tn = 0;
  const long long t_prologue = clock64();
#endif

  // Warp roles.  Warp w issues on sub-partition w & 3, and where the helpers sit matters (+-10 %, profiles/r07l, r07m):
  // two statistics warps on one sub-partition starve each other, and every score warp waits for their output.
  // role: 0 score (index = rank among the score warps), 1 context, 2 finaliser, 3 statistics.
  const int role = (int)(kRoles[warp] >> 4), ridx = (int)(kRoles[warp] & 15);
  if (role == 0) {
    // =========================== score warps ===========================
    // lane = (row pair rp, half head hf, head hp): the lane scores positions rp and rp + 2 of the slice over 32
    // channels of head hp.  Per-channel operands (gamma', beta', v', queries) are loaded once for both positions,
    // which is what keeps the shared-memory pipe (4 wavefronts per 128-bit load) off the critical path.
    const int rp = lane >> 4, hf = (lane >> 3) & 1, hp = lane & 7;
    // swizzled chunk order: at step u the lane reads 16-byte chunk (u ^ hp) of its half head, so the 8 lanes of a
    // quarter warp hit 8 different bank groups (keys: row-major slice; queries / constants: plain [512] rows).  All
    // region bases are multiples of 128 bytes, so the chunk address is one lane register XOR (u << 4) -- a single
    // LOP3 per chunk instead of 16 pinned address registers (which pushed the loop into local-memory spills).
    uint32_t kofs0, cadr0;
    {
      const uint32_t o = (uint32_t)(hp * kD * 4 + hf * 128 + (hp << 4));
      asm volatile("mov.b32 %0, %1;" : "=r"(cadr0) : "r"(smem_u32(sm_c) + o));
      asm volatile("mov.b32 %0, %1;" : "=r"(kofs0) : "r"(smem_u32(smem + L::ring) + (uint32_t)(rp * kR * 4) + o));
    }
    auto kofs = [&](int u) { return kofs0 ^ (uint32_t)(u << 4); };
    auto cadr = [&](int u) { return cadr0 ^ (uint32_t)(u << 4); };
    const uint32_t q_minus_c = smem_u32(sm_q) - smem_u32(sm_c);
    float sv = 0.f;                                           // sum of v over this lane's 32 channels
    for (int c = 0; c < kD / 2; ++c) sv += a.vvec[hp * kD + hf * 32 + c];
    const float inv_T = kLog2e / a.temperature[0];            // p = 2^((score / T - bound) log2 e)
    const float shift = a.bound[hp] * kLog2e;
    int last_img = -1;
    // Score warp w takes slices w, w + NSW, ... of the CTA's sequence.  At most NSW < STAGES slices are in work, so a
    // warp never waits on a stage whose previous use is still pending (the parity waits would alias).  The LN
    // statistics of the slice (1 / std per position and beam, -mean per position) come from the statistics warp.
    for (int g = ridx; g < n_g; g += NSW) {
      A2_STAMP(0);
      int pos, ii, sl;
      if (g < len_last) { pos = 0; ii = n_seg - 1; sl = g; }
      else {
        int v = g - len_last + sl0;                             // v / spi by subtraction (at most n_seg rounds; an integer
        ii = 0;                                                 // or float division would queue behind the MUFU work)
        while (v >= spi) { v -= spi; ++ii; }
        sl = v;
        pos = ii + (len_last > 0 ? 1 : 0);
      }
      const int par = pos & 1;
      if (pos != last_img) {
        mbar_wait(&qfull[par], (uint32_t)((pos >> 1) & 1));
        last_img = pos;
      }
      const int s = g % STAGES;
      A2_STAMP(1);
      mbar_wait(&statrdy[s], (uint32_t)((g / STAGES) & 1));
      mbar_wait(&full[s], (uint32_t)((g / STAGES) & 1));     // completed long ago: makes the TMA writes visible to this warp
      A2_STAMP(2);
      const uint32_t kst = (uint32_t)(s * kSliceBytes);                         // stage offset (uniform)
      const uint32_t qcb = q_minus_c + (uint32_t)(par * 2 * K * kR * 4);        // centred queries of this image, relative to the constants
      const uint32_t qgb = qcb + (uint32_t)(K * kR * 4);                        // * gamma'
      // first chunk of pass 2 is staged behind the statistics loads
      const float4 stA = *reinterpret_cast<const float4*>(sm_st + s * L::kStatBytes + rp * 16);
      const float4 stB = *reinterpret_cast<const float4*>(sm_st + s * L::kStatBytes + (rp + 2) * 16);
      Chunk2<K> c;
      chunk2_load<K>(c, kofs(0) + kst, cadr(0), cadr(0) + qgb);
      float rsA[K], rsB[K], outA[K], outB[K];
#pragma unroll
      for (int j = 0; j < K; ++j) {
        asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(rsA[j]) : "f"(j == 0 ? stA.x : (j == 1 ? stA.y : stA.z)));
        asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(rsB[j]) : "f"(j == 0 ? stB.x : (j == 1 ? stB.y : stB.z)));
        outA[j] = sv;
        outB[j] = sv;
      }
      A2_STAMP(3);
      // ---- pass 2: LN + tanh + v-weighted head sum; per chunk: back A(u-1) | front A(u) | back B(u-1) | front B(u) ----
      const float2 nmuA = make_float2(stA.w, stA.w), nmuB = make_float2(stB.w, stB.w);
      float2 eaA[K], ebA[K], eaB[K], ebB[K];
      front4<K>(c.ka, c.g, c.b, c.q, nmuA, rsA, eaA, ebA);
      front4<K>(c.kb, c.g, c.b, c.q, nmuB, rsB, eaB, ebB);
      float4 vprev = c.v;
#pragma unroll
      for (int u = 1; u < ((COMIC_A2_KNOCK & 4) ? 1 : 8); ++u) {
        chunk2_load<K>(c, kofs(u) + kst, cadr(u), cadr(u) + qgb);
        back4<K>(vprev, eaA, ebA, outA, escale);
        front4<K>(c.ka, c.g, c.b, c.q, nmuA, rsA, eaA, ebA);
        back4<K>(vprev, eaB, ebB, outB, escale);
        front4<K>(c.kb, c.g, c.b, c.q, nmuB, rsB, eaB, ebB);
        vprev = c.v;
      }
      back4<K>(vprev, eaA, ebA, outA, escale);
      back4<K>(vprev, eaB, ebB, outB, escale);
      A2_STAMP(4);
      float* pdst = sm_p + s * kPStage + hp * kPos + rp;
#pragma unroll
      for (int j = 0; j < K; ++j) {
        const float oa = outA[j] + __shfl_xor_sync(0xffffffffu, outA[j], 8);   // two half heads
        const float ob = outB[j] + __shfl_xor_sync(0xffffffffu, outB[j], 8);
        if (hf == 0) {
          pdst[j * kH * kPos] = ex2_approx(fmaf(oa, inv_T, -shift));
          pdst[j * kH * kPos + 2] = ex2_approx(fmaf(ob, inv_T, -shift));
        }
      }
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(&scored[s]);
        mbar_arrive(&qempty[par]);
      }
      A2_STAMP(5);
#if COMIC_A2_TRACE
      if (trc != nullptr && tn < kTraceSlices && lane == 0) trc[tn * 8 + 6] = g;
      ++tn;
#endif
    }
  } else if (role == 1) {
    // =========================== context warps ===========================
    // Context warp cw takes every 2nd slice of the CTA's sequence and accumulates sum_m p[m] * key[m, :] over all 512
    // channels of it from the shared-memory slice (two independent release chains); at the end of an image it hands
    // its partial sums to the finaliser warp and goes straight on to the next image.
    const int cw = ridx;
    const int hd0 = lane >> 4;                                // quad i of this lane: channels 4 (lane + 32 i) .., head hd0 + 2 i
    float4 acc[K][4];
    float S[K][4];                                            // sum of p over this warp's slices, heads hd0 + 2 i
#pragma unroll
    for (int j = 0; j < K; ++j)
#pragma unroll
      for (int i = 0; i < 4; ++i) { acc[j][i] = make_float4(0.f, 0.f, 0.f, 0.f); S[j][i] = 0.f; }
    // The context warps are also the TMA producers: a stage is refilled by the warp that releases it (no "empty"
    // barrier, no producer warp); each first requests its share of the first STAGES slices.
    // r_*: the next slice this warp will request (up front: the slices < STAGES with the parity of cw + STAGES; then
    // slice g + STAGES when it releases slice g), tracked incrementally -- the request sits on the release path
    int r_g = 0, r_pos = 0, r_sl = seg_lo(seg_of(0)), r_hi = seg_hi(seg_of(0));
    auto r_adv = [&](int n) {
      r_g += n; r_sl += n;
      while (r_pos < n_seg && r_sl >= r_hi) {
        const int over = r_sl - r_hi;
        if (++r_pos < n_seg) { r_sl = seg_lo(seg_of(r_pos)) + over; r_hi = seg_hi(seg_of(r_pos)); }
      }
    };
    static_assert(kCtxWarps2 == 2, "request sequence below assumes two context warps");
    r_adv((cw + STAGES) % kCtxWarps2);                        // so that the up-front sequence runs straight into cw + STAGES
    while (r_g < STAGES && r_g < n_g) {
      if (lane == 0) request_slice(r_g % STAGES, seg_of(r_pos), r_sl);
      r_adv(kCtxWarps2);
    }
    int g = 0;
    for (int pos = 0; pos < n_seg; ++pos) {
      const int ii = seg_of(pos);
      const int s_hi = seg_hi(ii);
      // unnormalised weights go straight to the history rows of the image ([K][8][M], contiguous); the finaliser
      // rescales them in place once the image's sums are known
      float* hrow = a.hist_t ? a.hist_t + ((size_t)(b0 + ii) * K * kH + lane) * M : nullptr;
      for (int sl = seg_lo(ii); sl < s_hi; ++sl, ++g) {
        if ((g & (kCtxWarps2 - 1)) != cw) continue;
        const int s = g % STAGES;
        A2_STAMP(0);
        mbar_wait(&scored[s], (uint32_t)((g / STAGES) & 1));
        A2_STAMP(1);
        if (hrow != nullptr && lane < K * kH)
          *reinterpret_cast<float4*>(hrow + sl * kPos) = *reinterpret_cast<const float4*>(sm_p + s * kPStage + lane * kPos);
        const float* tile = reinterpret_cast<const float*>(smem + L::ring + s * kSliceBytes) + lane * 4;
        const float* pp = sm_p + s * kPStage + hd0 * kPos;
        float4 kr[2][kPos], p4[2][K];
#pragma unroll
        for (int r = 0; r < kPos; ++r) kr[0][r] = *reinterpret_cast<const float4*>(tile + r * kR);
#pragma unroll
        for (int j = 0; j < K; ++j) p4[0][j] = *reinterpret_cast<const float4*>(pp + (j * kH) * kPos);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          if (i + 1 < 4) {
#pragma unroll
            for (int r = 0; r < kPos; ++r) kr[(i + 1) & 1][r] = *reinterpret_cast<const float4*>(tile + r * kR + (i + 1) * 128);
#pragma unroll
            for (int j = 0; j < K; ++j) p4[(i + 1) & 1][j] = *reinterpret_cast<const float4*>(pp + (j * kH + 2 * (i + 1)) * kPos);
          }
#pragma unroll
          for (int j = 0; j < K; ++j) {
            const float4 p = p4[i & 1][j];
            S[j][i] += (p.x + p.y) + (p.z + p.w);
            float2 lo = make_float2(acc[j][i].x, acc[j][i].y), hi = make_float2(acc[j][i].z, acc[j][i].w);
            lo = __ffma2_rn(make_float2(p.x, p.x), make_float2(kr[i & 1][0].x, kr[i & 1][0].y), lo);
            hi = __ffma2_rn(make_float2(p.x, p.x), make_float2(kr[i & 1][0].z, kr[i & 1][0].w), hi);
            lo = __ffma2_rn(make_float2(p.y, p.y), make_float2(kr[i & 1][1].x, kr[i & 1][1].y), lo);
            hi = __ffma2_rn(make_float2(p.y, p.y), make_float2(kr[i & 1][1].z, kr[i & 1][1].w), hi);
            lo = __ffma2_rn(make_float2(p.z, p.z), make_float2(kr[i & 1][2].x, kr[i & 1][2].y), lo);
            hi = __ffma2_rn(make_float2(p.z, p.z), make_float2(kr[i & 1][2].z, kr[i & 1][2].w), hi);
            lo = __ffma2_rn(make_float2(p.w, p.w), make_float2(kr[i & 1][3].x, kr[i & 1][3].y), lo);
            hi = __ffma2_rn(make_float2(p.w, p.w), make_float2(kr[i & 1][3].z, kr[i & 1][3].w), hi);
            acc[j][i] = make_float4(lo.x, lo.y, hi.x, hi.y);
          }
        }
        __syncwarp();
        if (r_g < n_g) {                                      // every reader of the stage is done: refill it (r_g == g + STAGES)
          if (lane == 0) request_slice(s, seg_of(r_pos), r_sl);
          r_adv(kCtxWarps2);
        }
        A2_STAMP(2);
#if COMIC_A2_TRACE
        if (tn < kTraceSlices - 1) ++tn;
#endif
      }
      // ---- image complete for this warp: hand the partial sums to the finaliser ----
      mbar_wait(partfree, (uint32_t)((pos & 1) ^ 1));         // the finaliser has read the previous segment's partials
      float* pw = sm_part + (size_t)cw * K * (kR + kH);
#pragma unroll
      for (int j = 0; j < K; ++j)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          *reinterpret_cast<float4*>(pw + j * kR + (lane + 32 * i) * 4) = acc[j][i];
          if ((lane & 15) == 0) pw[K * kR + j * kH + hd0 + 2 * i] = S[j][i];
          acc[j][i] = make_float4(0.f, 0.f, 0.f, 0.f);
          S[j][i] = 0.f;
        }
      if (!(seg_lo(ii) == 0 && s_hi == spi) && hrow != nullptr && a.hist_scale == nullptr)
        __threadfence();                                      // part of an image: its history rows are rescaled by another CTA
      __syncwarp();
      if (lane == 0) mbar_arrive(imgdone);
      A2_STAMP(3);
#if COMIC_A2_TRACE
      if (tn < kTraceSlices - 1) ++tn;
#endif
    }
  } else if (role == 2) {
    // =========================== finaliser ===========================
    // Per image segment: sum p over its positions (fixed order), add the two context partials (warp 0 + warp 1); a
    // whole image is normalised and written at once, a partial one goes through the global scratch (see top).
    constexpr int kPartFloats = K * (kR + kH);
    const int hd0 = lane >> 4;
    const int m4 = M / 4;
    auto cta_of = [&](long long x) { return (int)(((x + 1) * G + T_all - 1) / T_all) - 1; };   // CTA that owns slice x
    // Query preparation (centred queries, their gamma'-scaled copies, sum of squares) for segment pos into buffer
    // pos & 1: segments 0 and 1 up front, segment pos + 2 as soon as segment pos is complete (its buffer is then free
    // and the score warps need the new contents only after all of segment pos + 1).
    auto prep_queries = [&](int pos) {
      const int ii = seg_of(pos);
      const int par = pos & 1;
      mbar_wait(&qempty[par], (uint32_t)(((pos >> 1) & 1) ^ 1));   // buffer last used by the segment before the previous one
      float* qc = sm_q + (size_t)par * 2 * K * kR;
      float* qg = qc + K * kR;
      float4 v[K][4];
#pragma unroll
      for (int j = 0; j < K; ++j) {
        const float* q = a.lq + (size_t)((b0 + ii) * K + j) * a.ld_lq + a.q_off + lane * 16;
#pragma unroll
        for (int g = 0; g < 4; ++g) v[j][g] = ldg4(q + g * 4);
      }
#pragma unroll
      for (int j = 0; j < K; ++j) {
        float s = 0.f;
#pragma unroll
        for (int g = 0; g < 4; ++g) s += (v[j][g].x + v[j][g].y) + (v[j][g].z + v[j][g].w);
        const float mean = wsum(s) * (1.0f / kR);
        float sq = 0.f, sc = 0.f;
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          const float4 c = make_float4(v[j][g].x - mean, v[j][g].y - mean, v[j][g].z - mean, v[j][g].w - mean);
          const float4 g4 = *reinterpret_cast<const float4*>(sm_c + lane * 16 + g * 4);
          *reinterpret_cast<float4*>(qc + j * kR + lane * 16 + g * 4) = c;
          *reinterpret_cast<float4*>(qg + j * kR + lane * 16 + g * 4) = make_float4(c.x * g4.x, c.y * g4.y, c.z * g4.z, c.w * g4.w);
          sq = fmaf(c.x, c.x, sq); sq = fmaf(c.y, c.y, sq); sq = fmaf(c.z, c.z, sq); sq = fmaf(c.w, c.w, sq);
          sc += (c.x + c.y) + (c.z + c.w);
        }
        sq = wsum(sq);
        sc = wsum(sc);
        if (lane == 0) {
          sm_qs[(par * K + j) * 2 + 0] = sq;
          sm_qs[(par * K + j) * 2 + 1] = sc;
        }
      }
      __syncwarp();
      if (lane == 0) {
        // a partial segment scores fewer than spi slices: make up the difference on the buffer's release barrier
        const int missing = spi - (seg_hi(ii) - seg_lo(ii));
        if (missing > 0) mbar_arrive_n(&qempty[par], (uint32_t)missing);
        mbar_arrive(&qfull[par]);
      }
    };
    prep_queries(0);
    if (n_seg > 1) prep_queries(1);
    for (int pos = 0; pos < n_seg; ++pos) {
      const int ii = seg_of(pos);
      const int b = b0 + ii;
      const int lo = seg_lo(ii), hi = seg_hi(ii);
      A2_STAMP(0);
      mbar_wait(imgdone, (uint32_t)(pos & 1));
      A2_STAMP(1);
      if (pos + 2 < n_seg) prep_queries(pos + 2);
      float4 tot[K][4];
#pragma unroll
      for (int j = 0; j < K; ++j)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float4 x = *reinterpret_cast<const float4*>(sm_part + j * kR + (lane + 32 * i) * 4);
          const float4 y = *reinterpret_cast<const float4*>(sm_part + K * (kR + kH) + j * kR + (lane + 32 * i) * 4);
          tot[j][i] = make_float4(x.x + y.x, x.y + y.y, x.z + y.z, x.w + y.w);
        }
      if (lane < K * kH) sm_inv[lane] = sm_part[K * kR + lane] + sm_part[K * (kR + kH) + K * kR + lane];   // sum p of the segment
      __syncwarp();
      if (lane == 0) mbar_arrive(partfree);
      float* hdst = a.hist_t ? a.hist_t + (size_t)b * K * kH * M : nullptr;   // rows b*K + j, each [8][M]: contiguous
      // rescale the unnormalised history rows of the whole image in place (written by the context warps of this CTA, or,
      // for a split image, of all its CTAs), 8 independent 16-byte loads in flight per lane
      auto rescale_history = [&]() {
        const int n4 = K * kH * m4;
        for (int i0 = lane; i0 < n4; i0 += 256) {
          float4 v[8];
#pragma unroll
          for (int r = 0; r < 8; ++r)
            if (i0 + 32 * r < n4) v[r] = __ldcg(reinterpret_cast<const float4*>(hdst) + i0 + 32 * r);
#pragma unroll
          for (int r = 0; r < 8; ++r) {
            const int idx = i0 + 32 * r;
            if (idx < n4) {
              const float inv = sm_inv[K * kH + idx / m4];
              reinterpret_cast<float4*>(hdst)[idx] = make_float4(v[r].x * inv, v[r].y * inv, v[r].z * inv, v[r].w * inv);
            }
          }
        }
      };
      if (lo == 0 && hi == spi) {
#pragma unroll
        for (int j = 0; j < K; ++j)
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float inv = 1.0f / sm_inv[j * kH + hd0 + 2 * i];
            *reinterpret_cast<float4*>(a.ctx_out + (size_t)(b * K + j) * a.ld_ctx + (lane + 32 * i) * 4) =
                make_float4(tot[j][i].x * inv, tot[j][i].y * inv, tot[j][i].z * inv, tot[j][i].w * inv);
          }
        if (hdst != nullptr) {
          if (a.hist_scale != nullptr) {
            if (lane < K * kH) a.hist_scale[(size_t)b * K * kH + lane] = 1.0f / sm_inv[lane];
          } else {
            if (lane < K * kH) sm_inv[K * kH + lane] = 1.0f / sm_inv[lane];
            __syncwarp();
            rescale_history();
          }
        }
      } else {
        // part of an image: park the partial results, the last part to arrive combines them
        const int c_first = cta_of((long long)b * spi), c_last = cta_of((long long)(b + 1) * spi - 1);
        auto slot_of = [&](int c) { return 2 * c + (((int)((T_all * c / G) / spi) == b) ? 0 : 1); };
        float* sc = a.scratch + (size_t)slot_of((int)blockIdx.x) * kPartFloats;
#pragma unroll
        for (int j = 0; j < K; ++j)
#pragma unroll
          for (int i = 0; i < 4; ++i) *reinterpret_cast<float4*>(sc + j * kR + (lane + 32 * i) * 4) = tot[j][i];
        if (lane < K * kH) sc[K * kR + lane] = sm_inv[lane];
        __syncwarp();
        A2_STAMP(6);
        int old = 0;
        if (lane == 0) {
          __threadfence();
          old = atomicAdd(a.counters + b, 1);
        }
        old = __shfl_sync(0xffffffffu, old, 0);
        A2_STAMP(3);
        if (old == c_last - c_first) {
          __threadfence();
          // Parts are added in CTA order.  At small batches an image is cut into many parts (25 images: 6) and this
          // combine is the tail of the launch: with two parts in flight per round and the slot arithmetic (64-bit
          // divisions) inside the loop it took 32 k of the launch's 64 k cycles (profiles/r12g_attn2_combine_trace.txt).
          // Now: the slot of part l is computed once by lane l, and four parts x four quads of loads are in flight.
          const int nparts = c_last - c_first + 1;
          const int slot_l = slot_of(c_first + (lane < nparts ? lane : 0));
          auto slot_at = [&](int idx) {                                  // whole warp, idx uniform
            return nparts <= 32 ? __shfl_sync(0xffffffffu, slot_l, idx & 31) : slot_of(c_first + idx);
          };
          {
            float s = 0.f;
            for (int p0 = 0; p0 < nparts; p0 += 4) {
              float v[4];
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                const int sl = slot_at(p0 + q < nparts ? p0 + q : p0);
                v[q] = (p0 + q < nparts && lane < K * kH) ? __ldcg(a.scratch + (size_t)sl * kPartFloats + K * kR + lane) : 0.f;
              }
#pragma unroll
              for (int q = 0; q < 4; ++q) if (p0 + q < nparts) s += v[q];
            }
            if (lane < K * kH) sm_inv[lane] = s;
          }
          __syncwarp();
#pragma unroll 1
          for (int j = 0; j < K; ++j) {
            float4 t[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) t[i] = make_float4(0.f, 0.f, 0.f, 0.f);
            for (int p0 = 0; p0 < nparts; p0 += 4) {
              float4 x[4][4];
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                const int sl = slot_at(p0 + q < nparts ? p0 + q : p0);
                const float* sp = a.scratch + (size_t)sl * kPartFloats + j * kR;
#pragma unroll
                for (int i = 0; i < 4; ++i)
                  x[q][i] = (p0 + q < nparts) ? __ldcg(reinterpret_cast<const float4*>(sp + (lane + 32 * i) * 4))
                                              : make_float4(0.f, 0.f, 0.f, 0.f);
              }
#pragma unroll
              for (int q = 0; q < 4; ++q)
                if (p0 + q < nparts) {
#pragma unroll
                  for (int i = 0; i < 4; ++i) { t[i].x += x[q][i].x; t[i].y += x[q][i].y; t[i].z += x[q][i].z; t[i].w += x[q][i].w; }
                }
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float inv = 1.0f / sm_inv[j * kH + hd0 + 2 * i];
              *reinterpret_cast<float4*>(a.ctx_out + (size_t)(b * K + j) * a.ld_ctx + (lane + 32 * i) * 4) =
                  make_float4(t[i].x * inv, t[i].y * inv, t[i].z * inv, t[i].w * inv);
            }
          }
          A2_STAMP(4);
          if (hdst != nullptr) {
            if (a.hist_scale != nullptr) {
              if (lane < K * kH) a.hist_scale[(size_t)b * K * kH + lane] = 1.0f / sm_inv[lane];
            } else {
              if (lane < K * kH) sm_inv[K * kH + lane] = 1.0f / sm_inv[lane];
              __syncwarp();
              rescale_history();
            }
          }
          A2_STAMP(5);
          if (lane == 0) a.counters[b] = 0;
        }
      }
      __syncwarp();
      A2_STAMP(2);
#if COMIC_A2_TRACE
      if (tn < kTraceSlices - 1) ++tn;
#endif
    }
  } else {
    // =========================== LN statistics ===========================
    // Statistics warp sw takes every 2nd landed slice and computes <k_m - mean, qc_j> for the 4 positions x K beams -- the centred queries of the image
    // live in registers, lane owns float4 chunks lane + 32 i, so a slice costs 16 shared loads and 96 packed FMAs for
    // all score warps together (they used to spend a quarter of their time on it, 40 loads + 96 FMAs + 48 shuffle /
    // add steps EACH per slice) -- and publishes 1 / std per (position, beam) and -mean per position.
    static_assert(K <= 3, "statistics record: {rstd_0, rstd_1, rstd_2, -mean}");
    const int sw = ridx;
    float4 qreg[K][4];
    float sqq[K], sumq[K];
    const int r_own = lane >> 3, j_own = lane & 7;             // after the reduction: lane group r_own holds position r_own
    int g = 0;
    for (int pos = 0; pos < n_seg; ++pos) {
      const int ii = seg_of(pos);
      const int par = pos & 1;
      const int lo = seg_lo(ii), hi = seg_hi(ii);
      {
        // no slice of this segment for this warp (1-slice segment): skip it without touching its barriers (a warp
        // that waits for a query buffer two preparations late would wait on an aliased parity)
        const int first = g + (sw - g % kStatWarps + kStatWarps) % kStatWarps;
        if (first >= g + (hi - lo)) { g += hi - lo; continue; }
      }
      mbar_wait(&qfull[par], (uint32_t)((pos >> 1) & 1));
      {
        const float* qc = sm_q + (size_t)par * 2 * K * kR;
#pragma unroll
        for (int j = 0; j < K; ++j) {
#pragma unroll
          for (int i = 0; i < 4; ++i) qreg[j][i] = *reinterpret_cast<const float4*>(qc + j * kR + (lane + 32 * i) * 4);
          sqq[j] = sm_qs[(par * K + j) * 2 + 0];
          sumq[j] = sm_qs[(par * K + j) * 2 + 1];
        }
      }
      for (int sl = lo; sl < hi; ++sl, ++g) {
        if (g % kStatWarps != sw) continue;
        const int s = g % STAGES;
        A2_STAMP(0);
        // mean, centred sum of squares of key row r_own of the slice: needed last, fetched first
        const float2 ks = __ldg(reinterpret_cast<const float2*>(a.kstats) + ((size_t)(b0 + ii) * M + sl * kPos + r_own));
        mbar_wait(&full[s], (uint32_t)((g / STAGES) & 1));
        A2_STAMP(1);
        const float* tile = reinterpret_cast<const float*>(smem + L::ring + s * kSliceBytes) + lane * 4;
        float v[kPos * K];
        {
          float4 kr[2][4];
#pragma unroll
          for (int i = 0; i < 4; ++i) kr[0][i] = *reinterpret_cast<const float4*>(tile + i * 128);
#pragma unroll
          for (int r = 0; r < kPos; ++r) {
            if (r + 1 < kPos) {
#pragma unroll
              for (int i = 0; i < 4; ++i) kr[(r + 1) & 1][i] = *reinterpret_cast<const float4*>(tile + (r + 1) * kR + i * 128);
            }
#pragma unroll
            for (int j = 0; j < K; ++j) {
              float2 acc = make_float2(0.f, 0.f);
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                acc = __ffma2_rn(make_float2(kr[r & 1][i].x, kr[r & 1][i].y), make_float2(qreg[j][i].x, qreg[j][i].y), acc);
                acc = __ffma2_rn(make_float2(kr[r & 1][i].z, kr[r & 1][i].w), make_float2(qreg[j][i].z, qreg[j][i].w), acc);
              }
              v[r * K + j] = acc.x + acc.y;
            }
          }
        }
        // reduce-scatter over the 32 lanes: xor 16 halves the positions {0,1 | 2,3}, xor 8 again, then a butterfly
        float w[2 * K], x[K];
        {
          const bool up = (lane & 16) != 0;
#pragma unroll
          for (int t = 0; t < 2 * K; ++t) {
            const float send = up ? v[t] : v[t + 2 * K], keep = up ? v[t + 2 * K] : v[t];
            w[t] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
          }
          const bool up8 = (lane & 8) != 0;
#pragma unroll
          for (int t = 0; t < K; ++t) {
            const float send = up8 ? w[t] : w[t + K], keep = up8 ? w[t + K] : w[t];
            x[t] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
          }
#pragma unroll
          for (int o = 4; o >= 1; o >>= 1)
#pragma unroll
            for (int t = 0; t < K; ++t) x[t] += __shfl_xor_sync(0xffffffffu, x[t], o);
        }
        {
          float* rec = reinterpret_cast<float*>(sm_st + s * L::kStatBytes + r_own * 16);
          if (j_own < K) {
            const float xd = j_own == 0 ? x[0] : (j_own == 1 ? x[K > 1 ? 1 : 0] : x[K > 2 ? 2 : 0]);
            const float sq = j_own == 0 ? sqq[0] : (j_own == 1 ? sqq[K > 1 ? 1 : 0] : sqq[K > 2 ? 2 : 0]);
            const float sm = j_own == 0 ? sumq[0] : (j_own == 1 ? sumq[K > 1 ? 1 : 0] : sumq[K > 2 ? 2 : 0]);
            const float d = fmaf(-ks.x, sm, xd);                // <k - mean, qc> (sum qc is ~0, not exactly 0)
            const float sa = fmaxf(fmaf(2.0f, d, ks.y + sq), 0.f);
            rec[j_own] = sa * (1.0f / kR) + 1e-12f;        // variance + eps: the score warps take the rsqrt (no MUFU queue here)
          } else if (j_own == 3) {
            rec[3] = -ks.x;
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&statrdy[s]);
        A2_STAMP(2);
#if COMIC_A2_TRACE
        if (tn < kTraceSlices - 1) ++tn;
#endif
      }
    }
  }
#if COMIC_A2_TRACE
  // whole-warp residency: entry / end of prologue / exit (SM clock) and entry / exit on the global timer (ns), last record
  if (trc != nullptr && lane == 0) {
    unsigned long long g_exit;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g_exit));
    long long* e = trc + (kTraceSlices - 1) * 8;
    e[0] = t_entry; e[1] = t_prologue; e[2] = clock64(); e[3] = (long long)g_entry; e[4] = (long long)g_exit;
  }
#endif
}

}  // namespace a2
}  // namespace comic

namespace comic {
namespace a2 {

#ifndef COMIC_A2_STAGES
#define COMIC_A2_STAGES 21
#endif

// Launch for k beams per image (instantiated: 1, 2, 3).  Returns cudaErrorInvalidValue for shapes the kernel
// does not cover (the caller falls back to attention.cuh).
template <int K, int NSW = COMIC_A2_NSW, int STAGES = COMIC_A2_STAGES>
inline cudaError_t launch_k(const Args& a, int num_sms, int dev, cudaStream_t st) {
  using L = Layout<K, NSW, STAGES>;
  static_assert(STAGES > NSW, "the ring needs more stages than score warps");
  if (a.M % kPos != 0 || a.M > 256) return cudaErrorInvalidValue;
  const size_t smem = L::bytes(a.M);
  if (smem > 227 * 1024) return cudaErrorInvalidValue;
  (void)dev;
  static PerDeviceOnce once;
  {
    cudaError_t e = once([&] { return cudaFuncSetAttribute(attn2_kernel<K, NSW, STAGES>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); });
    if (e != cudaSuccess) return e;
  }
  const long long total = (long long)a.B * (a.M / kPos);
  const int grid = total < num_sms ? (int)total : num_sms;
  if (a.scratch == nullptr || a.counters == nullptr) return cudaErrorInvalidValue;
  attn2_kernel<K, NSW, STAGES><<<grid, L::kThreads, smem, st>>>(a);
  return cudaGetLastError();
}

inline cudaError_t launch(const Args& a, int k, int num_sms, int dev, cudaStream_t st) {
  switch (k) {
    case 1: return launch_k<1>(a, num_sms, dev, st);
    case 2: return launch_k<2>(a, num_sms, dev, st);
    case 3: return launch_k<3>(a, num_sms, dev, st);
    default: return cudaErrorInvalidValue;
  }
}

// Global scratch of one launch: floats for up to `num_sms` CTAs (two partial-image slots each) and k <= 3 beams.
inline size_t scratch_floats(int num_sms) { return (size_t)2 * num_sms * 3 * (kR + kH); }

constexpr int kBoundFloats = 12;   // [0..7] per-head score bound, [8] exponent shift, [9] shift feasible
inline cudaError_t launch_key_stats(const float* keys, long long rows, float* kstats, const float* vvec,
                                    const float* temperature, const float* gamma, const float* beta, float* bound,
                                    cudaStream_t st) {
  key_stats_kernel<<<(unsigned)((rows + 7) / 8), 256, 0, st>>>(keys, rows, kstats, vvec, temperature, gamma, beta, bound);
  return cudaGetLastError();
}

}  // namespace a2
}  // namespace comic
