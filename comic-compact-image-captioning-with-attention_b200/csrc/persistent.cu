// persistent.cu -- the whole beam / greedy decode loop as ONE cooperative kernel
// for small row counts (N = batch x beam <= 32), sm_100a.
//
// Replaces, for one decode call, the while_loop that TF builds for
//   rnn_decoder_beam_search / rnn_decoder_search   common/ops_rnn.py:49-180
// around MultiHeadAttentionWrapperV3.call           common/ops_rnn.py:660-755
// (~150 TF ops per step; 8 kernel launches per step on the per-step path of
// decoder.cu).  At N = 24 rows a step moves ~16 MB and is pure latency, so the
// loop runs inside one launch with the operands that do not change between
// steps resident in shared memory, and the CTAs meet at five grid barriers per
// step:
//
//   phase A1 gates: the [W+A+R, 4R] LSTM kernel is cut into (K group x 128-column) blocks, one per
//            CTA, RESIDENT in smem for the whole loop (8 x 16 blocks of 160 x 128 = 80 KB at
//            COMIC-256).  A CTA reads only its K slice of x = [emb(tok) ; ctx[src] ; h[src]] (15 KB;
//            every CTA reading all of x measured 15-19 us per step on L2 hot lines) and writes
//            its partial sums.
//   phase A2 fixed-order sum over the K groups + bias, LSTM cell -> c', h'  (4 units per CTA).
//   phase B  [logits | query] = h' . [W_o | W_q] + b: 8-column blocks per CTA.
//   phase C1 attention scores: CTA (image, position slice) keeps its CENTRED key
//            rows resident in smem (keys never re-read from HBM after step 0) and
//            scores them against the k beam queries (ln_tanh_scores, attention.cuh);
//            meanwhile B other CTAs run the beam step (log-softmax, top-k,
//            backpointers: beam_step_block, search_steps.cuh) on the logits.
//   phase C2 softmax over the 196 positions + context: CTA (image, channel slice)
//            with its value columns resident in smem; alignment history write.
//
// Cross-CTA data inside the launch is read with ld.global.cg / cp.async.cg (L2)
// and published with __threadfence() before the barrier arrive.  The barrier is a
// monotonic counter; a spin that exceeds ~2 s sets an abort flag that every CTA
// honours (T_out becomes -1 and the host raises), so a bug cannot hang the GPU.
#include "attention.cuh"
#include "comic_internal.cuh"
#include "search_steps.cuh"

namespace comic {

constexpr int kPT = 512;            // threads per CTA
constexpr int kPW = kPT / 32;       // warps
constexpr int kPMaxRPL = 4;         // rows per lane group: N <= 8 * 4
constexpr int kPCS = 128;           // phase-A column block (16 warps x 8 columns)
constexpr int kPMaxHeads = 4;       // heads a CTA may need in phase C2

struct PersistArgs {
  // weights
  const float* lstm_kernel;   // [KX][4R]
  const float* lstm_bias;     // [4R]
  const float* outq;          // [R][LQ] = [W_o | pad | W_q]
  const float* outq_bias;     // [LQ]
  const float* emb;           // [V][W]
  const float *gamma, *beta, *vvec, *temperature;
  // per-call inputs
  const float* keys;          // [B][M][R]
  const float* values;        // [B][M][VAL]
  const float* c0;            // [B][R]
  const float* h0;
  // dims
  int B, k, N, W, A, KX, V, LQ, q_off, M, VAL, prob_fn, eos, max_it, greedy;
  float lpw;
  // state (global, caller workspace)
  float* c[2];
  float* h[2];
  float* ctx[2];
  float* lq;                  // [N][LQ]
  float* scores;              // [N][H][M]
  float* hist;                // [T][N][H*M] or nullptr
  int* tok;
  int* src;
  float* cum;
  uint8_t* fin;
  long long* len;
  int* fin_count;
  int* step_ids;              // beam: [T][N] words; greedy: ids_out [T][N]
  int* parents;               // beam
  float* sc;                  // beam: [T][N] scores
  float* logits_out;          // greedy: [T][N][V] or nullptr
  unsigned* bar;              // [0] barrier counter, [1] abort flag
  long long spin_limit;       // grid-barrier watchdog in clock cycles (0 = none)
  long long* trace;           // [max_it][2][16] clock64 stamps of CTA 0 and the first selection CTA, or nullptr
  // partition / smem plan (floats)
  int KG, KS, CB, nB, S, rps, cps, nh_max, keys_res, vals_res, n_sel;
  float* part;                // [KG][N][4R] partial gate sums
  int off_wA, off_c, off_keys, off_skk, off_vals, off_tr, tr_floats;
};

__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// All CTAs of the (cooperative) grid meet here.  Returns false when the launch was aborted.
// spin_limit: clock64 cycles a CTA may wait before it declares the launch dead (0 = wait for ever: time-sliced GPUs,
// debuggers); COMIC_OPT_PERSISTENT_WATCHDOG_MS.
__device__ __forceinline__ bool grid_barrier(unsigned* bar, unsigned& target, unsigned nblocks, int* s_abort,
                                             long long spin_limit) {
  __syncthreads();
  if (threadIdx.x == 0) {
    target += nblocks;
    __threadfence();
    atomicAdd(bar, 1u);
    const long long t0 = clock64();
    int ab = 0;
    while (ld_acquire_u32(bar) < target) {
      if (ld_acquire_u32(bar + 1) != 0u) { ab = 1; break; }
      if (spin_limit > 0 && clock64() - t0 > spin_limit) {   // default ~2 s at 1.9 GHz: publish the abort and leave
        atomicExch(bar + 1, 1u);
        ab = 1;
        break;
      }
    }
    __threadfence();
    *s_abort = ab;
  }
  __syncthreads();
  return *s_abort == 0;
}

// Arrive without waiting: for a CTA that neither produced anything the next phase consumes nor
// consumes anything the previous phase produced (the selection CTAs between phases C1 and C2).
__device__ __forceinline__ void grid_arrive(unsigned* bar, unsigned& target, unsigned nblocks) {
  __syncthreads();
  if (threadIdx.x == 0) {
    target += nblocks;
    __threadfence();
    atomicAdd(bar, 1u);
  }
}

__device__ __forceinline__ void cp_async16_zfill(void* smem_dst, const void* gsrc, bool valid) {
  const int sz = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)),
               "l"(gsrc), "r"(sz)
               : "memory");
}

__device__ __forceinline__ float4 ldcg4(const float* p) { return __ldcg(reinterpret_cast<const float4*>(p)); }

// Phase-A1 inner product of one lane: RP row groups x 2 columns over KS k's, with the packed
// fp32 pipe (FFMA2: two FMAs per lane per issue slot; the plain FFMA issues every other cycle
// per scheduler on sm_100).  The k dimension is packed: acc.x sums even k, acc.y odd k.
//   wl: this lane's slice of the k-pair-interleaved weight block, [KS/2][kPCS][2]
template <int RP>
__device__ __forceinline__ void gemm_a1(const float* __restrict__ xs, int XLD, int N, int ng, const float* __restrict__ wl,
                                        int KS, float (&out)[kPMaxRPL][2]) {
  float2 acc[RP][2];
  const float* xrow[RP];
#pragma unroll
  for (int r = 0; r < RP; ++r) {
    acc[r][0] = acc[r][1] = make_float2(0.f, 0.f);
    xrow[r] = xs + (size_t)min(ng + 8 * r, N - 1) * XLD;   // rows beyond N recompute row N-1 (never stored)
  }
#pragma unroll 4
  for (int k4 = 0; k4 < KS; k4 += 4) {
    const float4 wv0 = *reinterpret_cast<const float4*>(wl + (size_t)(k4 >> 1) * kPCS * 2);
    const float4 wv1 = *reinterpret_cast<const float4*>(wl + (size_t)((k4 >> 1) + 1) * kPCS * 2);
#pragma unroll
    for (int r = 0; r < RP; ++r) {
      const float4 x = *reinterpret_cast<const float4*>(xrow[r] + k4);
      acc[r][0] = __ffma2_rn(make_float2(x.x, x.y), make_float2(wv0.x, wv0.y), acc[r][0]);
      acc[r][1] = __ffma2_rn(make_float2(x.x, x.y), make_float2(wv0.z, wv0.w), acc[r][1]);
      acc[r][0] = __ffma2_rn(make_float2(x.z, x.w), make_float2(wv1.x, wv1.y), acc[r][0]);
      acc[r][1] = __ffma2_rn(make_float2(x.z, x.w), make_float2(wv1.z, wv1.w), acc[r][1]);
    }
  }
#pragma unroll
  for (int r = 0; r < RP; ++r) {
    out[r][0] = acc[r][0].x + acc[r][0].y;
    out[r][1] = acc[r][1].x + acc[r][1].y;
  }
}

template <int H, int KB>
__global__ void __launch_bounds__(kPT, 1)
decode_loop_kernel(const PersistArgs a) {
  constexpr int R = 512;
  constexpr int CPL = R / 32, G4 = CPL / 4;
  constexpr int D = R / H;
  constexpr int LPH = (D >= CPL) ? D / CPL : 1;
  constexpr float kTwoLog2e = 2.885390081777927f;
  extern __shared__ __align__(16) float sm[];
  __shared__ BeamStepSmem s_beam;
  __shared__ GreedyStepSmem s_greedy;
  __shared__ const float* s_xp[3][32];   // x segment row pointers (nullptr = zero row)
  __shared__ int s_abort;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int cta = blockIdx.x;
  const unsigned G = gridDim.x;
  const int N = a.N, k = a.k, M = a.M, KX = a.KX, LQ = a.LQ, VAL = a.VAL;
  const int ng = lane >> 2, cg = lane & 3;
  const int rpl = (N + 7) >> 3;
  unsigned bar_target = 0;

  float* wA = sm + a.off_wA;          // [KS/2][kPCS][2] block of the LSTM kernel (k pairs interleaved)
  float* sm_c = sm + a.off_c;         // [3][R] lane-permuted gamma', beta', vv
  float* sm_keys = sm + a.off_keys;   // [rps][R] centred key rows, lane-permuted
  float* sm_skk = sm + a.off_skk;     // [rps]
  float* sm_vals = sm + a.off_vals;   // [M][cps]
  float* tr = sm + a.off_tr;          // transient region (per-phase layouts)

  const int n_colgrp = 4 * R / kPCS;   // column groups of the [KX, 4R] LSTM kernel
  const bool has_A = cta < a.KG * n_colgrp;
  const int kgp = cta / n_colgrp, cgp = cta % n_colgrp;
  const bool has_B = cta < a.nB;
  const bool has_C = cta < a.B * a.S;
  const int img = has_C ? cta / a.S : 0, slc = has_C ? cta % a.S : 0;
  const int m0 = slc * a.rps, m1 = min(M, m0 + a.rps);
  const int ch0 = slc * a.cps, ch1 = min(VAL, ch0 + a.cps);
  const bool sel_cta = cta >= a.B * a.S && cta < a.B * a.S + a.n_sel;
  const int c0l = lane * CPL;

  // ------------------------------------------------------------------ setup
  if (has_A) {
    // rows [kgp*KS, +KS) x columns [cgp*128, +128) of the LSTM kernel, resident for the whole loop
    // smem layout [KS/2][128][2]: the two k's of a pair adjacent (operand pairs of the packed FMA)
    const int tot4 = a.KS * (kPCS / 4);
    for (int i = tid; i < tot4; i += kPT) {
      const int kk = i / (kPCS / 4), j4 = i - kk * (kPCS / 4);
      const float4 w4 = ldg4(a.lstm_kernel + (size_t)(kgp * a.KS + kk) * 4 * R + cgp * kPCS + j4 * 4);
      float* dst = wA + ((size_t)(kk >> 1) * kPCS + j4 * 4) * 2 + (kk & 1);
      dst[0] = w4.x; dst[2] = w4.y; dst[4] = w4.z; dst[6] = w4.w;
    }
  }
  float sv = 0.f;
  {
    if (warp == 0) {
#pragma unroll
      for (int g = 0; g < G4; ++g) {
        float4 g4 = ldg4(a.gamma + c0l + g * 4), b4 = ldg4(a.beta + c0l + g * 4), v4 = ldg4(a.vvec + c0l + g * 4);
        *reinterpret_cast<float4*>(sm_c + (g * 32 + lane) * 4) =
            make_float4(g4.x * kTwoLog2e, g4.y * kTwoLog2e, g4.z * kTwoLog2e, g4.w * kTwoLog2e);
        *reinterpret_cast<float4*>(sm_c + R + (g * 32 + lane) * 4) =
            make_float4(b4.x * kTwoLog2e, b4.y * kTwoLog2e, b4.z * kTwoLog2e, b4.w * kTwoLog2e);
        // pair order (v1, v3 | v0, v2): the layout ln_tanh_scores<.., FAST = false> consumes (attention.cuh)
        *reinterpret_cast<float4*>(sm_c + 2 * R + (g * 32 + lane) * 4) =
            make_float4(v4.y * -2.0f, v4.w * -2.0f, v4.x * -2.0f, v4.z * -2.0f);
      }
    }
#pragma unroll
    for (int g = 0; g < G4; ++g) {
      float4 v4 = ldg4(a.vvec + c0l + g * 4);
      sv += (v4.x + v4.y) + (v4.z + v4.w);
    }
  }
  if (has_C && a.keys_res) {
    for (int r = warp; r < m1 - m0; r += kPW) {
      const float* kr = a.keys + ((size_t)img * M + m0 + r) * R + c0l;
      float4 v[G4];
      float s = 0.f;
#pragma unroll
      for (int g = 0; g < G4; ++g) {
        v[g] = ldg4(kr + g * 4);
        s += (v[g].x + v[g].y) + (v[g].z + v[g].w);
      }
      const float mean = wsum(s) * (1.0f / R);
      float sq = 0.f;
#pragma unroll
      for (int g = 0; g < G4; ++g) {
        float4 c = make_float4(v[g].x - mean, v[g].y - mean, v[g].z - mean, v[g].w - mean);
        sq = fmaf(c.x, c.x, sq); sq = fmaf(c.y, c.y, sq); sq = fmaf(c.z, c.z, sq); sq = fmaf(c.w, c.w, sq);
        *reinterpret_cast<float4*>(sm_keys + (size_t)r * R + (g * 32 + lane) * 4) = c;
      }
      sq = wsum(sq);
      if (lane == 0) sm_skk[r] = sq;
    }
  }
  if (has_C && a.vals_res && ch0 < VAL) {
    const int nc4 = (ch1 - ch0) >> 2;
    for (int i = tid; i < M * nc4; i += kPT) {
      int m = i / nc4, c4 = i - m * nc4;
      *reinterpret_cast<float4*>(sm_vals + (size_t)m * a.cps + c4 * 4) =
          ldg4(a.values + ((size_t)img * M + m) * VAL + ch0 + c4 * 4);
    }
  }
  const float out_scale = 1.0f / __ldg(a.temperature);
  __syncthreads();

  // ------------------------------------------------------------------ step loop
  const int trace_slot = (cta == 0) ? 0 : ((cta == a.B * a.S) ? 1 : -1);
  auto stamp = [&](int t, int i) {
    if (a.trace != nullptr && trace_slot >= 0 && tid == 0) a.trace[((size_t)t * 2 + trace_slot) * 16 + i] = clock64();
  };
  for (int t = 0; t < a.max_it; ++t) {
    const int cur = t & 1;
    stamp(t, 0);
    const float* c_prev = (t == 0) ? a.c0 : a.c[cur];
    const float* h_prev = (t == 0) ? a.h0 : a.h[cur];
    const float* ctx_prev = a.ctx[cur];
    float* c_new = a.c[cur ^ 1];
    float* h_new = a.h[cur ^ 1];
    float* ctx_new = a.ctx[cur ^ 1];

    // ============================ phase A1: partial gate sums of this CTA's (K group, column group) block
    if (has_A) {
      if (tid < N) {
        const int n = tid;
        const int tk = __ldcg(a.tok + n);
        int sr;
        if (a.greedy) sr = n;
        else sr = (t == 0) ? n / k : __ldcg(a.src + n);
        const int lim = (t == 0 && !a.greedy) ? a.B : N;
        const bool ok = sr >= 0 && sr < lim;
        s_xp[0][n] = (tk >= 0 && tk < a.V) ? a.emb + (size_t)tk * a.W : nullptr;
        s_xp[1][n] = ok ? ctx_prev + (size_t)sr * a.A : nullptr;
        s_xp[2][n] = ok ? h_prev + (size_t)sr * R : nullptr;
      }
      __syncthreads();
      stamp(t, 9);
      const int KS = a.KS, XLD = KS + 4;               // padded row stride: one float4 of bank shift per row
      const int kbase = kgp * KS;
      float* xs = tr;                                  // [N][KS + 4]: this K group's slice of x = [emb ; ctx ; h]
      for (int p = tid; p < N * (KS / 4); p += kPT) {
        const int n = p / (KS / 4), q = p - n * (KS / 4);
        const int kg = kbase + q * 4;
        const float* srcp;
        if (kg < a.W) { const float* b0 = s_xp[0][n]; srcp = b0 ? b0 + kg : nullptr; }
        else if (kg < a.W + a.A) { const float* b1 = s_xp[1][n]; srcp = b1 ? b1 + (kg - a.W) : nullptr; }
        else { const float* b2 = s_xp[2][n]; srcp = b2 ? b2 + (kg - a.W - a.A) : nullptr; }
        cp_async16_zfill(xs + (size_t)n * XLD + q * 4, srcp ? (const void*)srcp : (const void*)a.emb, srcp != nullptr);
      }
      cp_async_commit();
      cp_async_wait<0>();
      __syncthreads();
      stamp(t, 10);
      // warp w owns columns [8w, 8w+8) of the block for ALL KS k's (no cross-warp reduction);
      // a lane owns rows {ng, ng+8, ...} x 2 columns
      float acc[kPMaxRPL][2];
      {
        const float* wl = wA + (size_t)(warp * 8 + cg * 2) * 2;
        switch (rpl) {
          case 1: gemm_a1<1>(xs, XLD, N, ng, wl, KS, acc); break;
          case 2: gemm_a1<2>(xs, XLD, N, ng, wl, KS, acc); break;
          case 3: gemm_a1<3>(xs, XLD, N, ng, wl, KS, acc); break;
          default: gemm_a1<4>(xs, XLD, N, ng, wl, KS, acc); break;
        }
      }
#pragma unroll
      for (int r = 0; r < kPMaxRPL; ++r) {
        const int n = ng + 8 * r;
        if (r < rpl && n < N)
          *reinterpret_cast<float2*>(a.part + ((size_t)kgp * N + n) * 4 * R + cgp * kPCS + warp * 8 + cg * 2) =
              make_float2(acc[r][0], acc[r][1]);
      }
    }
    stamp(t, 11);
    if (!grid_barrier(a.bar, bar_target, G, &s_abort, a.spin_limit)) return;
    stamp(t, 12);

    // ============================ phase A2: fixed-order sum over the K groups + bias, LSTM cell -> c', h'
    if (cta < R / 4 && tid < ((N * 16 + 31) & ~31)) {   // whole warps (full-mask shuffles below)
      // thread = (row n, unit u, gate q): the 4 gate sums of a unit sit in 4 adjacent lanes
      const bool row_ok = (tid >> 4) < N;
      const int n = row_ok ? (tid >> 4) : N - 1, u = (tid >> 2) & 3, q = tid & 3;
      const int unit = cta * 4 + u;
      const float* pp = a.part + (size_t)n * 4 * R + q * R + unit;
      const size_t kstride = (size_t)N * 4 * R;
      float v[16];
#pragma unroll
      for (int kg2 = 0; kg2 < 16; ++kg2) v[kg2] = (kg2 < a.KG) ? __ldcg(pp + kg2 * kstride) : 0.f;
      float sacc = 0.f;
#pragma unroll
      for (int kg2 = 0; kg2 < 16; ++kg2) sacc += v[kg2];          // fixed order; + 0 for unused groups
      sacc += __ldg(a.lstm_bias + q * R + unit);
      const int l0 = lane & ~3;
      const float g0 = __shfl_sync(0xffffffffu, sacc, l0), g1 = __shfl_sync(0xffffffffu, sacc, l0 + 1);
      const float g2 = __shfl_sync(0xffffffffu, sacc, l0 + 2), g3 = __shfl_sync(0xffffffffu, sacc, l0 + 3);
      if (q == 0 && row_ok) {
        int sr;
        if (a.greedy) sr = n;
        else sr = (t == 0) ? n / k : __ldcg(a.src + n);
        const int lim = (t == 0 && !a.greedy) ? a.B : N;
        const float cp = (sr >= 0 && sr < lim) ? __ldcg(c_prev + (size_t)sr * R + unit) : 0.f;
        float cn, hn;
        lstm_cell(g0, g1, g2, g3, cp, &cn, &hn);
        c_new[(size_t)n * R + unit] = cn;
        h_new[(size_t)n * R + unit] = hn;
      }
    }
    stamp(t, 1);
    if (!grid_barrier(a.bar, bar_target, G, &s_abort, a.spin_limit)) return;
    stamp(t, 2);

    // ============================ phase B: [logits | q] = h' . [W_o | W_q] + bias
    if (has_B) {
      const int HLD = R + 4;
      float* hs = tr;                                  // [N][R+4]
      float* wB = tr + (size_t)N * HLD;                // [R][8]
      float* red = wB + (size_t)R * 8;                 // [kPW][N][8]
      for (int p = tid; p < N * (R / 4); p += kPT) {
        const int n = p / (R / 4), q = p - n * (R / 4);
        cp_async16(hs + (size_t)n * HLD + q * 4, h_new + (size_t)n * R + q * 4);
      }
      cp_async_commit();
      const int nblk = a.CB / 8;
      for (int blk = 0; blk < nblk; ++blk) {
        const int col0 = cta * a.CB + blk * 8;
        if (col0 >= LQ) break;
        for (int p = tid; p < R * 2; p += kPT) {
          const int kk = p >> 1, hlf = p & 1;
          const int col = col0 + hlf * 4;
          cp_async16_zfill(wB + (size_t)kk * 8 + hlf * 4, col < LQ ? a.outq + (size_t)kk * LQ + col : a.outq, col < LQ);
        }
        cp_async_commit();
        cp_async_wait<0>();
        __syncthreads();
        float acc2[kPMaxRPL][2];
        const float* hrow[kPMaxRPL];
#pragma unroll
        for (int r = 0; r < kPMaxRPL; ++r) {
          acc2[r][0] = acc2[r][1] = 0.f;
          hrow[r] = hs + (size_t)min(ng + 8 * r, N - 1) * HLD;
        }
#pragma unroll
        for (int j = 0; j < R / kPW / 4; ++j) {
          const int kk = warp * (R / kPW) + j * 4;
          float2 w2[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) w2[q] = *reinterpret_cast<const float2*>(wB + (size_t)(kk + q) * 8 + cg * 2);
#pragma unroll
          for (int r = 0; r < kPMaxRPL; ++r) {
            const float4 x = *reinterpret_cast<const float4*>(hrow[r] + kk);
            acc2[r][0] = fmaf(x.x, w2[0].x, acc2[r][0]); acc2[r][1] = fmaf(x.x, w2[0].y, acc2[r][1]);
            acc2[r][0] = fmaf(x.y, w2[1].x, acc2[r][0]); acc2[r][1] = fmaf(x.y, w2[1].y, acc2[r][1]);
            acc2[r][0] = fmaf(x.z, w2[2].x, acc2[r][0]); acc2[r][1] = fmaf(x.z, w2[2].y, acc2[r][1]);
            acc2[r][0] = fmaf(x.w, w2[3].x, acc2[r][0]); acc2[r][1] = fmaf(x.w, w2[3].y, acc2[r][1]);
          }
        }
#pragma unroll
        for (int r = 0; r < kPMaxRPL; ++r) {
          const int n = ng + 8 * r;
          if (r < rpl && n < N)
            *reinterpret_cast<float2*>(red + ((size_t)warp * N + n) * 8 + cg * 2) = make_float2(acc2[r][0], acc2[r][1]);
        }
        __syncthreads();
        if (tid < N * 8) {
          const int n = tid >> 3, cc = tid & 7;
          const int col = col0 + cc;
          if (col < LQ) {
            float s = 0.f;
            for (int w = 0; w < kPW; ++w) s += red[((size_t)w * N + n) * 8 + cc];
            a.lq[(size_t)n * LQ + col] = s + __ldg(a.outq_bias + col);
          }
        }
        __syncthreads();
      }
      cp_async_wait<0>();
    }
    stamp(t, 3);
    if (!grid_barrier(a.bar, bar_target, G, &s_abort, a.spin_limit)) return;
    stamp(t, 4);

    // ============================ phase C1: attention scores  ||  beam / greedy selection
    if (has_C) {
      float* sm_q = tr;                         // [k][R] centred queries (lane-permuted)
      float* sm_qg = tr + (size_t)k * R;        // [k][R] * gamma'
      float* sm_sqq = tr + 2 * (size_t)k * R;   // [k]
      for (int beam = warp; beam < k; beam += kPW) {
        const float* q = a.lq + (size_t)(img * k + beam) * LQ + a.q_off + c0l;
        float4 v[G4];
        float s = 0.f;
#pragma unroll
        for (int g = 0; g < G4; ++g) {
          v[g] = ldcg4(q + g * 4);
          s += (v[g].x + v[g].y) + (v[g].z + v[g].w);
        }
        const float mean = wsum(s) * (1.0f / R);
        float sq = 0.f;
#pragma unroll
        for (int g = 0; g < G4; ++g) {
          float4 c = make_float4(v[g].x - mean, v[g].y - mean, v[g].z - mean, v[g].w - mean);
          *reinterpret_cast<float4*>(sm_q + (size_t)beam * R + (g * 32 + lane) * 4) = c;
          sq = fmaf(c.x, c.x, sq); sq = fmaf(c.y, c.y, sq); sq = fmaf(c.z, c.z, sq); sq = fmaf(c.w, c.w, sq);
          const float4 gm = *reinterpret_cast<const float4*>(sm_c + (g * 32 + lane) * 4);
          *reinterpret_cast<float4*>(sm_qg + (size_t)beam * R + (g * 32 + lane) * 4) =
              make_float4(c.x * gm.x, c.y * gm.y, c.z * gm.z, c.w * gm.w);
        }
        sq = wsum(sq);
        if (lane == 0) sm_sqq[beam] = sq;
      }
      __syncthreads();
      for (int r = warp; r < m1 - m0; r += kPW) {
        const int m = m0 + r;
        float kc[CPL], kg[CPL];
        float skk;
        if (a.keys_res) {
#pragma unroll
          for (int g = 0; g < G4; ++g) {
            const float4 tq = *reinterpret_cast<const float4*>(sm_keys + (size_t)r * R + (g * 32 + lane) * 4);
            kc[g * 4 + 0] = tq.x; kc[g * 4 + 1] = tq.y; kc[g * 4 + 2] = tq.z; kc[g * 4 + 3] = tq.w;
          }
          skk = sm_skk[r];
        } else {
          const float* kr = a.keys + ((size_t)img * M + m) * R + c0l;
          float s = 0.f;
#pragma unroll
          for (int g = 0; g < G4; ++g) {
            const float4 tq = ldg4(kr + g * 4);
            kc[g * 4 + 0] = tq.x; kc[g * 4 + 1] = tq.y; kc[g * 4 + 2] = tq.z; kc[g * 4 + 3] = tq.w;
            s += (tq.x + tq.y) + (tq.z + tq.w);
          }
          const float mean = wsum(s) * (1.0f / R);
          float sq = 0.f;
#pragma unroll
          for (int c = 0; c < CPL; ++c) {
            kc[c] -= mean;
            sq = fmaf(kc[c], kc[c], sq);
          }
          skk = wsum(sq);
        }
#pragma unroll
        for (int g = 0; g < G4; ++g) {
          const float4 gm = *reinterpret_cast<const float4*>(sm_c + (g * 32 + lane) * 4);
          kg[g * 4 + 0] = kc[g * 4 + 0] * gm.x; kg[g * 4 + 1] = kc[g * 4 + 1] * gm.y;
          kg[g * 4 + 2] = kc[g * 4 + 2] * gm.z; kg[g * 4 + 3] = kc[g * 4 + 3] * gm.w;
        }
        for (int beam0 = 0; beam0 < k; beam0 += KB) {
          const int bs = min(beam0, k - KB);
          float part[KB];
          ln_tanh_scores<CPL, KB, false>(kc, kg, sm_q + (size_t)bs * R, sm_qg + (size_t)bs * R, sm_c, sm_sqq + bs, skk,
                                         R, lane, sv, 1.0f / R, part);
#pragma unroll
          for (int o = LPH / 2; o; o >>= 1) {
#pragma unroll
            for (int j = 0; j < KB; ++j) part[j] += __shfl_xor_sync(0xffffffffu, part[j], o);
          }
          if ((lane % LPH) == 0) {
            const int hh = lane / LPH;
#pragma unroll
            for (int j = 0; j < KB; ++j)
              a.scores[((size_t)(img * k + bs + j) * H + hh) * M + m] = part[j] * out_scale;
          }
        }
      }
    }
    stamp(t, 5);
    // The selection CTAs only ARRIVE at this barrier and run the beam / greedy step while the others do
    // phase C2: the step's outputs (tokens, parents, finished counts) are first read after the next barrier.
    if (sel_cta) {
      grid_arrive(a.bar, bar_target, G);
      const int si = cta - a.B * a.S;
      if (!a.greedy) {
        if (tid < 256)
          beam_step_block<true>(s_beam, tr, a.tr_floats, tid, si, a.lq, LQ, k, a.V, a.eos, a.lpw, a.cum, a.fin,
                                a.len, a.sc + (size_t)t * N, a.step_ids + (size_t)t * N, a.parents + (size_t)t * N,
                                a.tok, a.src, a.fin_count, t);
      } else {
        if (tid < 128)
          greedy_step_block<true>(s_greedy, tid, si, a.lq, LQ, a.V, a.eos, a.step_ids + (size_t)t * N,
                                  a.logits_out ? a.logits_out + (size_t)t * N * a.V : nullptr, a.tok, a.fin,
                                  a.fin_count, t);
      }
    } else if (!grid_barrier(a.bar, bar_target, G, &s_abort, a.spin_limit)) {
      return;
    }
    stamp(t, 6);

    // ============================ phase C2: softmax over positions, history, context
    if (has_C) {
      const int dv = VAL / H;
      const bool active = ch0 < VAL;
      // heads this CTA needs: those its channel slice touches + those whose history it writes (h % S == slc)
      int heads[kPMaxHeads];
      int nh = 0;
      if (active)
        for (int hh = ch0 / dv; hh <= (ch1 - 1) / dv && nh < kPMaxHeads; ++hh) heads[nh++] = hh;
      const int n_touched = nh;
      if (a.hist)
        for (int hh = slc; hh < H && nh < kPMaxHeads; hh += a.S) {
          bool dup = false;
          for (int i = 0; i < n_touched; ++i) dup |= (heads[i] == hh);
          if (!dup) heads[nh++] = hh;
        }
      float* sm_al = tr;                                   // [k][nh_max][M]
      float* redc = tr + (size_t)k * a.nh_max * M;          // [groups][tasks] float4
      redc = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(redc) + 15) & ~uintptr_t(15));
      for (int pr = warp; pr < k * nh; pr += kPW) {
        const int beam = pr / nh, hs_ = pr - beam * nh;
        const int hh = heads[hs_];
        const size_t grow = ((size_t)(img * k + beam) * H + hh) * M;
        float* s = sm_al + ((size_t)beam * a.nh_max + hs_) * M;
        float sum = 0.f;
        if (a.prob_fn == 0) {
          float mx = -INFINITY;
          for (int m = lane; m < M; m += 32) {
            const float x = __ldcg(a.scores + grow + m);
            s[m] = x;
            mx = fmaxf(mx, x);
          }
          mx = wmax(mx);
          for (int m = lane; m < M; m += 32) {
            float e = expf(s[m] - mx);
            s[m] = e;
            sum += e;
          }
        } else {
          for (int m = lane; m < M; m += 32) {
            float e = 1.0f / (1.0f + expf(-__ldcg(a.scores + grow + m)));
            s[m] = e;
            sum += e;
          }
        }
        sum = wsum(sum);
        const bool writes_hist = a.hist != nullptr && (hh % a.S) == slc;
        float* hrow = writes_hist ? a.hist + (size_t)t * N * H * M + grow : nullptr;
        for (int m = lane; m < M; m += 32) {
          const float al = s[m] / sum;
          s[m] = al;
          if (hrow) hrow[m] = al;
        }
      }
      __syncthreads();
      if (active) {
        const int nc4 = (ch1 - ch0) >> 2;
        const int ntask = k * nc4;                          // (beam, 4 channels)
        const int ngrp = kPT / ntask;                       // position groups
        const int task = tid % ntask, grp = tid / ntask;
        const int beam = task / nc4, c4 = task - beam * nc4;
        float4 acc4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (grp < ngrp) {
          const int hh = (ch0 + c4 * 4) / dv;
          int hs_ = 0;
          for (int i = 0; i < n_touched; ++i)
            if (heads[i] == hh) hs_ = i;
          const float* al = sm_al + ((size_t)beam * a.nh_max + hs_) * M;
          const int ma = (int)(((long long)M * grp) / ngrp), mb = (int)(((long long)M * (grp + 1)) / ngrp);
          for (int m = ma; m < mb; ++m) {
            const float4 v = a.vals_res ? *reinterpret_cast<const float4*>(sm_vals + (size_t)m * a.cps + c4 * 4)
                                        : ldg4(a.values + ((size_t)img * M + m) * VAL + ch0 + c4 * 4);
            const float w = al[m];
            acc4.x = fmaf(w, v.x, acc4.x); acc4.y = fmaf(w, v.y, acc4.y);
            acc4.z = fmaf(w, v.z, acc4.z); acc4.w = fmaf(w, v.w, acc4.w);
          }
          *reinterpret_cast<float4*>(redc + ((size_t)grp * ntask + task) * 4) = acc4;
        }
        __syncthreads();
        if (tid < ntask) {
          float4 s4 = make_float4(0.f, 0.f, 0.f, 0.f);
          for (int g2 = 0; g2 < ngrp; ++g2) {
            const float4 p = *reinterpret_cast<const float4*>(redc + ((size_t)g2 * ntask + tid) * 4);
            s4.x += p.x; s4.y += p.y; s4.z += p.z; s4.w += p.w;
          }
          const int bm = tid / nc4, cc4 = tid - bm * nc4;
          *reinterpret_cast<float4*>(ctx_new + (size_t)(img * k + bm) * a.A + ch0 + cc4 * 4) = s4;
        }
      }
    }
    stamp(t, 7);
    if (!grid_barrier(a.bar, bar_target, G, &s_abort, a.spin_limit)) return;
    stamp(t, 8);

    // every row finished in this step -> the loop ends (dynamic_decode's all(finished))
    if (__ldcg(a.fin_count + t) >= N) break;
  }
}

// ---------------------------------------------------------------------------
// Host side: applicability, partition and shared-memory plan, cooperative launch.
// ---------------------------------------------------------------------------
struct PersistPlan {
  bool ok = false;
  int G, KG, KS, CB, nB, S, rps, cps, nh_max, keys_res, vals_res;
  int off_wA, off_c, off_keys, off_skk, off_vals, off_tr, tr_floats;
  size_t smem_bytes;
};

static PersistPlan persist_plan(comic_handle_t h, int B, int k, bool greedy) {
  PersistPlan p;
  const int N = B * k, R = h->R, M = h->M, VAL = h->VAL, H = h->H;
  if (h->persist_max_rows <= 0 || N > h->persist_max_rows || N > 8 * kPMaxRPL) return p;
  if (h->cell != COMIC_CELL_LSTM) return p;   // the loop's phase A is the LSTM cell; GRU decodes take the per-step path
  if (R != 512 || h->cfg.alignment != 0 || h->cfg.context_layer || k > 16) return p;
  if (!(H == 1 || H == 2 || H == 4 || H == 8 || H == 16) || VAL % (4 * H) != 0 || h->KX % 4 != 0 || h->W % 4 != 0 ||
      h->A % 4 != 0 || h->LQ % 4 != 0 || h->Vp % 4 != 0 || h->A != VAL)
    return p;
  p.G = h->num_sms;
  const int n_sel = B;   // beam: one CTA per image; greedy: one per row (k == 1)
  if (2 * B > p.G || p.G - n_sel < B) return p;
  // phase A: (K group, 128-column group) blocks of the LSTM kernel, one per CTA
  const int n_colgrp = 4 * R / kPCS;
  p.KG = p.G / n_colgrp;
  while (p.KG > 1 && h->KX % (4 * p.KG) != 0) --p.KG;
  if (p.KG < 1 || R / 4 > p.G) return p;
  p.KS = h->KX / p.KG;
  p.CB = round_up((h->LQ + p.G - 1) / p.G, 8);
  p.nB = (h->LQ + p.CB - 1) / p.CB;
  p.S = (p.G - n_sel) / B;
  if (p.S > M) p.S = M;
  p.rps = (M + p.S - 1) / p.S;
  p.S = (M + p.rps - 1) / p.rps;
  p.cps = round_up((VAL + p.S - 1) / p.S, 4);
  const int dv = VAL / H;
  p.nh_max = 1;
  for (int s = 0; s < p.S; ++s) {
    int ch0 = s * p.cps, ch1 = ch0 + p.cps < VAL ? ch0 + p.cps : VAL;
    int nh = 0;
    if (ch0 < VAL) nh = (ch1 - 1) / dv - ch0 / dv + 1;
    for (int hh = s; hh < H; hh += p.S)
      if (!(ch0 < VAL && hh >= ch0 / dv && hh <= (ch1 - 1) / dv)) ++nh;
    if (nh > p.nh_max) p.nh_max = nh;
  }
  if (p.nh_max > kPMaxHeads) return p;
  if (k * (p.cps / 4) > kPT) return p;
  // transient region: max over the phase layouts (floats)
  size_t trA = (size_t)N * (p.KS + 4), trAr = 0;
  size_t trB = (size_t)N * (R + 4) + (size_t)R * 8 + (size_t)kPW * N * 8;
  size_t trC1 = (size_t)2 * k * R + 32;
  size_t trC2 = (size_t)k * p.nh_max * M + 4 + (size_t)kPT * 4;
  size_t tr = trA;
  if (trAr > tr) tr = trAr;
  if (trB > tr) tr = trB;
  if (trC1 > tr) tr = trC1;
  if (trC2 > tr) tr = trC2;
  const size_t budget = (size_t)(220 * 1024) / sizeof(float);
  for (int attempt = 0; attempt < 3; ++attempt) {
    p.keys_res = attempt < 2;
    p.vals_res = attempt < 1;
    size_t off = 0;
    p.off_wA = (int)off; off += (size_t)p.KS * kPCS;
    p.off_c = (int)off; off += 3 * (size_t)R;
    p.off_keys = (int)off; off += p.keys_res ? (size_t)p.rps * R : 0;
    p.off_skk = (int)off; off += p.keys_res ? (size_t)round_up(p.rps, 4) : 0;
    p.off_vals = (int)off; off += p.vals_res ? (size_t)M * p.cps : 0;
    p.off_tr = (int)off; off += tr;
    p.tr_floats = (int)tr;
    if (off <= budget) {
      p.smem_bytes = off * sizeof(float);
      p.ok = true;
      return p;
    }
  }
  return p;
}

template <int H, int KB>
static cudaError_t launch_persist(const PersistArgs& pa, int G, size_t smem, cudaStream_t st) {
  static PerDeviceOnce once;
  {
    cudaError_t e = once([&] { return cudaFuncSetAttribute(decode_loop_kernel<H, KB>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         222 * 1024); });
    if (e != cudaSuccess) return e;
  }
  void* args[] = {const_cast<PersistArgs*>(&pa)};
  return cudaLaunchCooperativeKernel((const void*)decode_loop_kernel<H, KB>, dim3(G), dim3(kPT), args, smem, st);
}

template <int H>
static cudaError_t launch_persist_h(const PersistArgs& pa, int G, size_t smem, cudaStream_t st) {
  if (pa.k == 1) return launch_persist<H, 1>(pa, G, smem, st);
  if (pa.k == 2 || pa.k == 4) return launch_persist<H, 2>(pa, G, smem, st);
  return launch_persist<H, 3>(pa, G, smem, st);
}

bool persist_applicable(comic_handle_t h, int B, int k, bool greedy) { return persist_plan(h, B, k, greedy).ok; }

// Returns 1 when the loop was enqueued as one cooperative launch, 0 when the configuration is
// not covered (the caller runs the per-step path), < 0 on error.
int decode_persistent(comic_handle_t h, const PersistCall& pc, cudaStream_t st) {
  PersistPlan p = persist_plan(h, pc.B, pc.k, pc.greedy != 0);
  if (!p.ok) return 0;
  PersistArgs a{};
  a.lstm_kernel = h->w.lstm_kernel; a.lstm_bias = h->w.lstm_bias;
  a.outq = h->pk.outq; a.outq_bias = h->pk.outq_bias; a.emb = h->w.embedding_map;
  a.gamma = h->w.ln_gamma; a.beta = h->w.ln_beta; a.vvec = h->w.attention_v; a.temperature = h->w.temperature;
  a.keys = pc.keys; a.values = pc.values; a.c0 = pc.c0; a.h0 = pc.h0;
  a.B = pc.B; a.k = pc.k; a.N = pc.B * pc.k; a.W = h->W; a.A = h->A; a.KX = h->KX; a.V = h->V; a.LQ = h->LQ;
  a.q_off = h->Vp; a.M = h->M; a.VAL = h->VAL; a.prob_fn = h->cfg.prob_fn; a.eos = h->cfg.eos_id;
  a.max_it = pc.max_it; a.greedy = pc.greedy; a.lpw = pc.lpw;
  for (int i = 0; i < 2; ++i) { a.c[i] = pc.c[i]; a.h[i] = pc.h[i]; a.ctx[i] = pc.ctx[i]; }
  a.lq = pc.lq; a.scores = pc.scores; a.hist = pc.hist; a.tok = pc.tok; a.src = pc.src; a.cum = pc.cum;
  a.fin = pc.fin; a.len = pc.len; a.fin_count = pc.fin_count; a.step_ids = pc.step_ids; a.parents = pc.parents;
  a.sc = pc.sc; a.logits_out = pc.logits_out; a.bar = pc.bar; a.trace = pc.trace;
  a.spin_limit = (long long)h->persist_watchdog_ms * 1900000ll;           // ms -> cycles at ~1.9 GHz
  h->last_trace = pc.trace; h->last_trace_steps = pc.trace ? pc.max_it : 0;
  a.KG = p.KG; a.KS = p.KS; a.part = pc.part; a.CB = p.CB; a.nB = p.nB; a.S = p.S; a.rps = p.rps; a.cps = p.cps;
  a.nh_max = p.nh_max; a.keys_res = p.keys_res; a.vals_res = p.vals_res; a.n_sel = pc.B;
  a.off_wA = p.off_wA; a.off_c = p.off_c; a.off_keys = p.off_keys; a.off_skk = p.off_skk; a.off_vals = p.off_vals;
  a.off_tr = p.off_tr; a.tr_floats = p.tr_floats;
  COMIC_CHECK_CUDA(cudaMemsetAsync(pc.bar, 0, 2 * sizeof(unsigned), st));
  cudaError_t e = cudaErrorInvalidValue;
  {
    Prof pf(h, T_PERSIST, st);
    switch (h->H) {
      case 1: e = launch_persist_h<1>(a, p.G, p.smem_bytes, st); break;
      case 2: e = launch_persist_h<2>(a, p.G, p.smem_bytes, st); break;
      case 4: e = launch_persist_h<4>(a, p.G, p.smem_bytes, st); break;
      case 8: e = launch_persist_h<8>(a, p.G, p.smem_bytes, st); break;
      case 16: e = launch_persist_h<16>(a, p.G, p.smem_bytes, st); break;
      default: break;
    }
  }
  COMIC_CHECK_CUDA(e);
  return 1;
}

}  // namespace comic
