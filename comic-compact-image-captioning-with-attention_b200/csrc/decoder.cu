// decoder.cu -- attention-LSTM decoder step, beam / greedy search loops and
// finalisation for sm_100a.
//
// Replaces the TF graph built by
//   MultiHeadAttentionWrapperV3.call      common/ops_rnn.py:660-755
//   MultiHeadAddLN.__call__ / MultiHeadDot common/ops_rnn.py:531-565, 603-632
//   rnn_decoder_beam_search / _search     common/ops_rnn.py:49-180
//   (TF r1.9 BeamSearchDecoder, dynamic_decode, gather_tree underneath)
//   ModelBase._get_rnn_init               src/model_base.py:651-689
//   ModelBase._decoder_post_process       src/model_base.py:272-314
//
// One decode call enqueues the whole T-step loop on the caller's stream with no
// host synchronisation: "all beams finished" is a device-side counter that turns
// the remaining steps into no-ops, and the executed step count is returned in a
// device int.  Beam-search state is never gathered: every consumer reads
// c/h/ctx through the `src` row indirection written by the beam kernel, and the
// keys/values of an image are shared by its k beams (the reference tiles them k
// times, src/model_base.py:130-131).
#include <float.h>
#include <math.h>

#include <algorithm>

#include "attention.cuh"
#include "beam_warp.cuh"
#include "attention2.cuh"
#include "comic_internal.cuh"
#include "search_steps.cuh"

namespace comic {

// ---------------------------------------------------------------------------
// D3: BasicLSTMCell pointwise part.  gates = sum of split-K partials [nz][N][4R]
// (+bias), order i,j,f,o, forget_bias 1.0.  c_prev is read through `src`.
// Optional output dropout (DropoutWrapper): h_drop = h / keep * mask.
// ---------------------------------------------------------------------------
__global__ void lstm_pointwise_kernel(const float* __restrict__ gp, int nz, size_t zstride,
                                      const float* __restrict__ bias, const float* __restrict__ c_prev,
                                      const int* __restrict__ src, int src_limit, float* __restrict__ c_new,
                                      float* __restrict__ h_new, float* __restrict__ h_drop,
                                      const float* __restrict__ out_mask, float out_keep, int N, int R,
                                      const int* fin_count, int t, int n_rows, float* __restrict__ gates_save) {
  if (step_stopped(fin_count, t, n_rows)) return;
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N * R) return;
  int n = i / R, j = i - n * R;
  float g[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    float s = 0.f;
    for (int z = 0; z < nz; ++z) s += gp[z * zstride + (size_t)n * 4 * R + q * R + j];
    g[q] = s + bias[q * R + j];
    if (gates_save) gates_save[(size_t)n * 4 * R + q * R + j] = g[q];
  }
  float cp = 0.f;
  if (c_prev) {
    int r = src ? src[n] : n;
    if (r >= 0 && r < src_limit) cp = c_prev[(size_t)r * R + j];
  }
  float cn, hn;
  lstm_cell(g[0], g[1], g[2], g[3], cp, &cn, &hn);
  c_new[i] = cn;
  h_new[i] = hn;
  if (h_drop) h_drop[i] = out_mask ? (hn / out_keep) * out_mask[i] : hn;
}

// Vectorised variant for the big-batch decode loop (R % 4 == 0, one split-K partial, no dropout / tape): four
// units per thread with 128-bit accesses.  FAST (engine precision >= 1, the tensor path): sigmoid / tanh through
// ex2.approx + rcp.approx (relative error ~1e-6 against expf / tanhf, same budget as the bf16x3 GEMM feeding it).
template <bool FAST, bool PART = false>
__global__ void __launch_bounds__(256)
lstm_pointwise4_kernel(const float* __restrict__ gates, const float* __restrict__ bias, const float* __restrict__ c_prev,
                       const int* __restrict__ src, int src_limit, float* __restrict__ c_new, float* __restrict__ h_new,
                       int N, int R, const int* fin_count, int t, int n_rows, uint16_t* __restrict__ h_hi = nullptr,
                       uint16_t* __restrict__ h_lo = nullptr, int nz = 1, size_t zstride = 0) {
  if (step_stopped(fin_count, t, n_rows)) return;
  const int R4 = R >> 2;
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N * R4) return;
  const int n = i / R4, j = (i - n * R4) * 4;
  const float* gr = gates + (size_t)n * 4 * R + j;
  float4 g[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    float4 v = ldg4(gr + q * R);
    const float4 b = ldg4(bias + q * R + j);
    if (PART) {
      for (int z = 1; z < nz; ++z) {                     // split-K partials of the gate GEMM, fixed order
        const float4 p = ldg4(gr + z * zstride + q * R);
        v.x += p.x; v.y += p.y; v.z += p.z; v.w += p.w;
      }
    }
    g[q] = make_float4(v.x + b.x, v.y + b.y, v.z + b.z, v.w + b.w);
  }
  float4 cp = make_float4(0.f, 0.f, 0.f, 0.f);
  if (c_prev) {
    const int r = src ? src[n] : n;
    if (r >= 0 && r < src_limit) cp = ldg4(c_prev + (size_t)r * R + j);
  }
  const float gi[4] = {g[0].x, g[0].y, g[0].z, g[0].w}, gj[4] = {g[1].x, g[1].y, g[1].z, g[1].w};
  const float gf[4] = {g[2].x, g[2].y, g[2].z, g[2].w}, go[4] = {g[3].x, g[3].y, g[3].z, g[3].w};
  const float cpv[4] = {cp.x, cp.y, cp.z, cp.w};
  float cn[4], hn[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    cn[q] = cpv[q] * sig_<FAST>(gf[q] + 1.0f) + sig_<FAST>(gi[q]) * tanh_<FAST>(gj[q]);
    hn[q] = tanh_<FAST>(cn[q]) * sig_<FAST>(go[q]);
  }
  *reinterpret_cast<float4*>(c_new + (size_t)n * R + j) = make_float4(cn[0], cn[1], cn[2], cn[3]);
  *reinterpret_cast<float4*>(h_new + (size_t)n * R + j) = make_float4(hn[0], hn[1], hn[2], hn[3]);
  if (h_hi != nullptr) {
    // the [logits | q] GEMM reads h' as bf16 (hi, lo) planes through TMA: same split as its fp32 loader would do
    uint2 hi, lo;
    tc::split4(make_float4(hn[0], hn[1], hn[2], hn[3]), hi, lo);
    *reinterpret_cast<uint2*>(h_hi + (size_t)n * R + j) = hi;
    *reinterpret_cast<uint2*>(h_lo + (size_t)n * R + j) = lo;
  }
}

// ---------------------------------------------------------------------------
// D3, GRU cell (TF r1.9 GRUCell, src/model_base.py:622-629):
//   [r, u] = sigmoid([x, h] . gates/kernel + gates/bias)
//   c      = tanh([x, r*h] . candidate/kernel + candidate/bias)
//   h'     = u*h + (1-u)*c
// The gate GEMM multiplies [x, h] by the panel [gates/kernel | candidate/kernel x-rows ; 0] into split-K partials
// [nz][N][3R] (r, u pre-activations, then x . Kc_x).  gru_gate_kernel sums them in a fixed order, takes the sigmoids and
// writes r * h[src] (the A operand of the candidate GEMM), u and x . Kc_x to [3][N][R]; the candidate GEMM adds
// (r*h) . Kc_h and gru_update_kernel forms c and h'.  h_prev == nullptr is the zero state (first_input init step).
// FAST (tensor path): sigmoid / tanh through ex2.approx + rcp.approx, as lstm_pointwise4_kernel<true>.
// ---------------------------------------------------------------------------
template <bool FAST>
__global__ void __launch_bounds__(256)
gru_gate_kernel(const float* __restrict__ gp, int nz, size_t zstride, const float* __restrict__ bias,
                const float* __restrict__ h_prev, const int* __restrict__ src, int src_limit, int N, int R,
                float* __restrict__ gru, const int* fin_count, int t, int n_rows, float* __restrict__ tape = nullptr) {
  if (step_stopped(fin_count, t, n_rows)) return;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N * R) return;
  const int n = i / R, j = i - n * R;
  const float* g = gp + (size_t)n * 3 * R + j;
  float s[3];
#pragma unroll
  for (int q = 0; q < 3; ++q) {
    float v = 0.f;
    for (int z = 0; z < nz; ++z) v += g[z * zstride + q * R];
    s[q] = v;
  }
  const float r = sig_<FAST>(s[0] + bias[j]);
  const float u = sig_<FAST>(s[1] + bias[R + j]);
  float hp = 0.f;
  if (h_prev) {
    const int row = src ? src[n] : n;
    if (row >= 0 && row < src_limit) hp = h_prev[(size_t)row * R + j];
  }
  const size_t NR = (size_t)N * R;
  gru[i] = r * hp;
  gru[NR + i] = u;
  gru[2 * NR + i] = s[2];
  if (tape) {   // training tape, row [r | u | r*h | c] (c: gru_update_kernel)
    float* tr = tape + (size_t)n * 4 * R + j;
    tr[0] = r; tr[R] = u; tr[2 * R] = r * hp;
  }
}

// cp: split-K partials [nz][N][R] of (r*h) . Kc_h (nz = 0: r*h is zero).  Output dropout as lstm_pointwise_kernel.
template <bool FAST>
__global__ void __launch_bounds__(256)
gru_update_kernel(const float* __restrict__ cp, int nz, size_t zstride, const float* __restrict__ gru,
                  const float* __restrict__ bias, const float* __restrict__ h_prev, const int* __restrict__ src, int src_limit,
                  float* __restrict__ h_new, float* __restrict__ h_drop, const float* __restrict__ out_mask, float out_keep,
                  int N, int R, const int* fin_count, int t, int n_rows, float* __restrict__ tape = nullptr) {
  if (step_stopped(fin_count, t, n_rows)) return;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N * R) return;
  const int n = i / R, j = i - n * R;
  const size_t NR = (size_t)N * R;
  float s = gru[2 * NR + i];
  for (int z = 0; z < nz; ++z) s += cp[z * zstride + i];
  const float c = tanh_<FAST>(s + bias[j]);
  if (tape) tape[(size_t)n * 4 * R + 3 * R + j] = c;
  const float u = gru[NR + i];
  float hp = 0.f;
  if (h_prev) {
    const int row = src ? src[n] : n;
    if (row >= 0 && row < src_limit) hp = h_prev[(size_t)row * R + j];
  }
  const float hn = u * hp + (1.f - u) * c;
  h_new[i] = hn;
  if (h_drop) h_drop[i] = out_mask ? (hn / out_keep) * out_mask[i] : hn;
}

// [gates/kernel | candidate/kernel x-rows ; 0]: the [W+A+R, 3R] B operand of the GRU gate GEMM.
__global__ void pack_gru_gates_kernel(const float* __restrict__ kg, const float* __restrict__ kc, float* __restrict__ out,
                                      int KX, int XA, int R) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)KX * 3 * R) return;
  const int row = (int)(i / (3 * R)), col = (int)(i % (3 * R));
  float v;
  if (col < 2 * R) v = kg[(size_t)row * 2 * R + col];
  else v = row < XA ? kc[(size_t)row * R + (col - 2 * R)] : 0.f;
  out[i] = v;
}

// x = [emb(tok) ; ctx[src] ; h[src]] of one decode step as bf16 (hi, lo) planes [N][W + A + R] for the gate GEMM's TMA-staged A
// operand: the gather (token / parent-beam indirection, zero rows for ids out of range) and the split happen ONCE per step
// here instead of once per N tile inside the GEMM (8 N tiles at 4R = 2048: 8 x the loads and conversions).
__global__ void __launch_bounds__(256)
build_x_planes_kernel(const float* __restrict__ emb, const int* __restrict__ tok, int V, const float* __restrict__ ctx_prev,
                      const float* __restrict__ h_prev, const int* __restrict__ src, int src_limit, int N, int W, int A, int R,
                      uint16_t* __restrict__ x_hi, uint16_t* __restrict__ x_lo, const int* fin_count, int t, int n_rows) {
  if (step_stopped(fin_count, t, n_rows)) return;
  const int KX4 = (W + A + R) >> 2;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N * KX4) return;
  const int n = i / KX4, k = (i - n * KX4) * 4;
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  if (k < W) {
    const int tk = tok[n];
    if (tk >= 0 && tk < V) v = ldg4(emb + (size_t)tk * W + k);
  } else {
    const int r = src ? src[n] : n;
    if (r >= 0 && r < src_limit) v = (k < W + A) ? ldg4(ctx_prev + (size_t)r * A + (k - W)) : ldg4(h_prev + (size_t)r * R + (k - W - A));
  }
  uint2 hi, lo;
  tc::split4(v, hi, lo);
  *reinterpret_cast<uint2*>(x_hi + (size_t)n * (W + A + R) + k) = hi;
  *reinterpret_cast<uint2*>(x_lo + (size_t)n * (W + A + R) + k) = lo;
}

// Generic split-K reduction: out[m, n] = sum_z part[z][m][n] + bias[n].
__global__ void splitk_reduce_kernel(const float* __restrict__ part, int nz, size_t zstride,
                                     const float* __restrict__ bias, float* __restrict__ out, int M, int ld,
                                     const int* fin_count, int t, int n_rows) {
  if (step_stopped(fin_count, t, n_rows)) return;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)M * ld) return;
  int n = (int)(i % ld);
  float s = 0.f;
  for (int z = 0; z < nz; ++z) s += part[z * zstride + i];
  out[i] = s + (bias ? bias[n] : 0.f);
}

// x = x / keep * mask (input dropout of the DropoutWrapper) for a [N, ncols] slice.
__global__ void dropout_rows_kernel(float* __restrict__ x, const float* __restrict__ mask, float keep, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) x[i] = (x[i] / keep) * mask[i];
}

// Assemble x = [emb(tok) ; ctx[src]] densely (only needed when input dropout is on).
__global__ void assemble_x_kernel(const float* __restrict__ emb, const int* __restrict__ tok, int V,
                                  int lookup, const float* __restrict__ ctx, float* __restrict__ x, int N,
                                  int W, int A) {
  int n = blockIdx.x;
  int id = tok[n];
  bool ok = id >= 0 && id < V;
  for (int j = threadIdx.x; j < W + A; j += blockDim.x) {
    float v;
    if (j < W) v = ok ? emb[(size_t)id * W + j] : 0.f;
    else v = ctx[(size_t)n * A + (j - W)];
    x[(size_t)n * (W + A) + j] = v;
  }
  (void)lookup; (void)N;
}

// ---------------------------------------------------------------------------
// D4: attention scores.  One CTA per (image, position slice); a warp owns one
// feature-map position at a time, keeps the key row in registers and scores it
// against the k beam queries of the image.
//   add_LN: s[h,m] = sum_{j in head h} tanh(LN(key[m]+q)[j]) * v[j] / T
//   dot   : s[h,m] = sum_{j in head h} key[m][j] * q[j] / sqrt(R/H)
// Two-pass moments in registers (mean, then sum (u-mean)^2), eps 1e-12, as
// tf.contrib.layers.layer_norm does.
// ---------------------------------------------------------------------------
template <int R, int H, int MODE>
__global__ void __launch_bounds__(256)
attn_scores_kernel(const float* __restrict__ keys, const float* __restrict__ lq, int ld_lq, int q_off,
                   const float* __restrict__ gamma, const float* __restrict__ beta,
                   const float* __restrict__ vvec, const float* __restrict__ temperature,
                   float* __restrict__ scores, int k, int M, int pos_per_cta, const int* fin_count, int t,
                   int n_rows) {
  if (step_stopped(fin_count, t, n_rows)) return;
  constexpr int G = R / 128;        // float4 groups per lane
  constexpr int D = R / H;          // head size
  extern __shared__ __align__(16) float sm_q[];   // [k][R]
  const int b = blockIdx.x;
  const int p0 = blockIdx.y * pos_per_cta;
  const int p1 = min(M, p0 + pos_per_cta);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int i = threadIdx.x; i < k * R; i += blockDim.x) {
    int beam = i / R, j = i - beam * R;
    sm_q[i] = lq[(size_t)(b * k + beam) * ld_lq + q_off + j];
  }
  float4 g4[G], b4[G], v4[G];
#pragma unroll
  for (int g = 0; g < G; ++g) {
    int c = g * 128 + lane * 4;
    if (MODE == 0) {
      g4[g] = ldg4(gamma + c);
      b4[g] = ldg4(beta + c);
      v4[g] = ldg4(vvec + c);
    }
  }
  const float inv_scale = (MODE == 0) ? (1.0f / temperature[0]) : 0.f;
  const float dot_div = sqrtf((float)D);
  (void)inv_scale;
  __syncthreads();
  for (int m = p0 + warp; m < p1; m += 8) {
    float4 key[G];
    const float* kr = keys + ((size_t)b * M + m) * R;
#pragma unroll
    for (int g = 0; g < G; ++g) key[g] = ldg4(kr + g * 128 + lane * 4);
    for (int beam = 0; beam < k; ++beam) {
      const float* q = sm_q + beam * R;
      float4 u[G];
      float part[G];
      if (MODE == 0) {
        float s = 0.f;
#pragma unroll
        for (int g = 0; g < G; ++g) {
          float4 qq = *reinterpret_cast<const float4*>(q + g * 128 + lane * 4);
          u[g].x = key[g].x + qq.x; u[g].y = key[g].y + qq.y;
          u[g].z = key[g].z + qq.z; u[g].w = key[g].w + qq.w;
          s += (u[g].x + u[g].y) + (u[g].z + u[g].w);
        }
        float mean = warp_sum(s) * (1.0f / R);
        float vs = 0.f;
#pragma unroll
        for (int g = 0; g < G; ++g) {
          float dx = u[g].x - mean, dy = u[g].y - mean, dz = u[g].z - mean, dw = u[g].w - mean;
          vs += (dx * dx + dy * dy) + (dz * dz + dw * dw);
        }
        float var = warp_sum(vs) * (1.0f / R);
        float rstd = 1.0f / sqrtf(var + 1e-12f);
#pragma unroll
        for (int g = 0; g < G; ++g) {
          // x*inv + (beta - mean*inv), inv = rstd*gamma  (tf.nn.batch_normalization)
          float ix = rstd * g4[g].x, iy = rstd * g4[g].y, iz = rstd * g4[g].z, iw = rstd * g4[g].w;
          float tx = tanhf(u[g].x * ix + (b4[g].x - mean * ix));
          float ty = tanhf(u[g].y * iy + (b4[g].y - mean * iy));
          float tz = tanhf(u[g].z * iz + (b4[g].z - mean * iz));
          float tw = tanhf(u[g].w * iw + (b4[g].w - mean * iw));
          part[g] = (tx * v4[g].x + ty * v4[g].y) + (tz * v4[g].z + tw * v4[g].w);
        }
      } else {
#pragma unroll
        for (int g = 0; g < G; ++g) {
          float4 qq = *reinterpret_cast<const float4*>(q + g * 128 + lane * 4);
          part[g] = (key[g].x * qq.x + key[g].y * qq.y) + (key[g].z * qq.z + key[g].w * qq.w);
        }
      }
      float* srow = scores + ((size_t)(b * k + beam) * H) * M + m;
      if (D >= 128) {
        // a 128-channel group lies inside one head
        float hs[H];
#pragma unroll
        for (int hh = 0; hh < H; ++hh) hs[hh] = 0.f;
#pragma unroll
        for (int g = 0; g < G; ++g) {
          float tsum = warp_sum(part[g]);
          hs[(g * 128) / D] += tsum;
        }
        if (lane == 0) {
#pragma unroll
          for (int hh = 0; hh < H; ++hh)
            srow[(size_t)hh * M] = (MODE == 0) ? hs[hh] * inv_scale : hs[hh] / dot_div;
        }
      } else {
        constexpr int LPH = D / 4;   // lanes per head inside a group
#pragma unroll
        for (int g = 0; g < G; ++g) {
          float v = part[g];
#pragma unroll
          for (int o = LPH / 2; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
          if ((lane % LPH) == 0) {
            int hh = (g * 128 + lane * 4) / D;
            srow[(size_t)hh * M] = (MODE == 0) ? v * inv_scale : v / dot_div;
          }
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------
// D4 (probability fn) + D5 + D6: softmax / signorm over the M positions of each
// (beam, head), optional attention-map dropout, alignment-history write and
// context ctx[n, c] = sum_m alpha[n, head(c), m] * values[b, m, c].
// Grid (B, ceil(VAL/128)); 512 threads = 128 value channels x 4 position slices (fixed-order sum of the four
// partials, deterministic): a single thread walking all M positions of its channel left the kernel latency-bound at
// small batches (42 us at 32 images, profiles/r02e).  CTA y==0 writes the history.
// ---------------------------------------------------------------------------
constexpr int kCtxSlices = 4;
__global__ void __launch_bounds__(128 * kCtxSlices)
attn_ctx_kernel(const float* __restrict__ scores, const float* __restrict__ values, int VAL,
                float* __restrict__ ctx_out, int ld_ctx, float* __restrict__ hist_t,
                const float* __restrict__ att_mask, float att_keep, int k, int H, int M, int prob_fn,
                const int* fin_count, int t, int n_rows, float* __restrict__ hist_pre) {
  if (step_stopped(fin_count, t, n_rows)) return;
  extern __shared__ __align__(16) float sm_alpha[];   // [k][H][M] | partial contexts [kCtxSlices][4][128]
  const int b = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int npair = k * H;
  float* sm_part = sm_alpha + (((size_t)npair * M + 3) & ~(size_t)3);
  for (int pr = warp; pr < npair; pr += 4 * kCtxSlices) {
    const float* s = scores + ((size_t)b * npair + pr) * M;
    float* a = sm_alpha + (size_t)pr * M;
    float sum = 0.f;
    if (M <= 256) {
      // up to 8 positions per lane: the row's scores and its dropout mask are fetched in ONE round of independent loads
      // (the generic loops below walk them one L2 round trip at a time: long-scoreboard stall 20 per issued
      // instruction, 28 us per launch at batch 32, profiles/r13b_*); same arithmetic in the same order
      const float* mk8 = att_mask ? att_mask + ((size_t)b * npair + pr) * M : nullptr;
      float sv[8], mv[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int m = lane + 32 * i;
        sv[i] = (m < M) ? s[m] : 0.f;
        mv[i] = (mk8 != nullptr && m < M) ? mk8[m] : 1.0f;
      }
      if (prob_fn == 0) {
        float mx = -INFINITY;
#pragma unroll
        for (int i = 0; i < 8; ++i) if (lane + 32 * i < M) mx = fmaxf(mx, sv[i]);
        mx = warp_max(mx);
#pragma unroll
        for (int i = 0; i < 8; ++i) if (lane + 32 * i < M) { sv[i] = expf(sv[i] - mx); sum += sv[i]; }
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) if (lane + 32 * i < M) { sv[i] = sigmoidf_(sv[i]); sum += sv[i]; }
      }
      sum = warp_sum(sum);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int m = lane + 32 * i;
        if (m < M) {
          float al = sv[i] / sum;
          if (hist_pre && blockIdx.y == 0) hist_pre[((size_t)b * npair + pr) * M + m] = al;
          if (mk8) al = (al / att_keep) * mv[i];
          a[m] = al;
          if (hist_t && blockIdx.y == 0) hist_t[((size_t)b * npair + pr) * M + m] = al;
        }
      }
      continue;
    }
    if (prob_fn == 0) {
      float mx = -INFINITY;
      for (int m = lane; m < M; m += 32) mx = fmaxf(mx, s[m]);
      mx = warp_max(mx);
      for (int m = lane; m < M; m += 32) {
        float e = expf(s[m] - mx);
        a[m] = e;
        sum += e;
      }
    } else {
      for (int m = lane; m < M; m += 32) {
        float e = sigmoidf_(s[m]);
        a[m] = e;
        sum += e;
      }
    }
    sum = warp_sum(sum);
    const float* mk = att_mask ? att_mask + ((size_t)b * npair + pr) * M : nullptr;
    for (int m = lane; m < M; m += 32) {
      float al = a[m] / sum;
      if (hist_pre && blockIdx.y == 0) hist_pre[((size_t)b * npair + pr) * M + m] = al;
      if (mk) al = (al / att_keep) * mk[m];
      a[m] = al;
      if (hist_t && blockIdx.y == 0) hist_t[((size_t)b * npair + pr) * M + m] = al;
    }
  }
  __syncthreads();
  const int cl = threadIdx.x & 127, sl = threadIdx.x >> 7;
  const int c = blockIdx.y * 128 + cl;
  const bool live = c < VAL;
  const int hd = live ? c / (VAL / H) : 0;
  const float* vb = values + (size_t)b * M * VAL + (live ? c : 0);
  const int per = (M + kCtxSlices - 1) / kCtxSlices;
  const int m0 = sl * per, m1 = min(M, m0 + per);
  for (int beam0 = 0; beam0 < k; beam0 += 4) {
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    const int nb = min(4, k - beam0);
    const float* a0 = sm_alpha + ((size_t)(beam0)*H + hd) * M;
    if (live) {
#pragma unroll 16
      for (int m = m0; m < m1; ++m) {
        float v = __ldg(vb + (size_t)m * VAL);
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (j < nb) acc[j] = fmaf(a0[(size_t)j * H * M + m], v, acc[j]);
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) sm_part[(sl * 4 + j) * 128 + cl] = acc[j];
    __syncthreads();
    if (sl == 0 && live) {
      for (int j = 0; j < nb; ++j) {
        float tot = sm_part[(0 * 4 + j) * 128 + cl];
#pragma unroll
        for (int q = 1; q < kCtxSlices; ++q) tot += sm_part[(q * 4 + j) * 128 + cl];
        ctx_out[(size_t)(b * k + beam0 + j) * ld_ctx + c] = tot;
      }
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------
// K10: TF r1.9 _beam_search_step, one CTA per image (body: search_steps.cuh).
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
beam_step_kernel(const float* __restrict__ logits, int ld, int k, int V, int eos, float lpw,
                 float* __restrict__ log_probs, uint8_t* __restrict__ finished, long long* __restrict__ lengths,
                 float* __restrict__ scores_out, int* __restrict__ word_out, int* __restrict__ parent_out,
                 int* __restrict__ tok_next, int* __restrict__ src_next, int* fin_count, int t, int n_rows) {
  if (step_stopped(fin_count, t, n_rows)) {
    // keep the stop condition visible to every later step
    if (blockIdx.x == 0 && threadIdx.x == 0) fin_count[t] = n_rows;
    return;
  }
  __shared__ BeamStepSmem S;
  __shared__ float s_stage[4096];   // k * V <= 4096 (radix / char vocabularies): logits staged once
  beam_step_block<false>(S, s_stage, 4096, threadIdx.x, blockIdx.x, logits, ld, k, V, eos, lpw, log_probs, finished, lengths,
                         scores_out, word_out, parent_out, tok_next, src_next, fin_count, t);
}

// K10 for small vocabularies at large batch: ONE WARP per image, four images per CTA, no block barriers (the 256-thread
// CTA of beam_step_kernel spends its 18 us in twelve barrier rounds over 774 candidates).  Per beam row the lane-strided
// max / sum(exp) / log are reduced with shuffles, every candidate's score is written to the warp's shared-memory slice once,
// and the k winners are drawn in k rounds of a warp arg-max with the same total order (score descending, flat index
// ascending).  Same per-candidate arithmetic as beam_step_block; only the order of the sum inside log-sum-exp differs.
constexpr int kBeamWarpImages = 4;
__global__ void __launch_bounds__(32 * kBeamWarpImages)
beam_step_warp_kernel(const BeamWarpArgs g, int B, int n_rows) {
  if (step_stopped(g.fin_count, g.t, n_rows)) {
    if (blockIdx.x == 0 && threadIdx.x == 0) g.fin_count[g.t] = n_rows;
    return;
  }
  extern __shared__ float s_sc[];                       // [kBeamWarpImages][k * V] candidate scores
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int b = blockIdx.x * kBeamWarpImages + warp;
  if (b >= B) return;
  beam_step_one_warp(g, b, s_sc + (size_t)warp * g.k * g.V, lane);
}

// Same step with one warp per BEAM ROW for the log-softmax part (k warps per image, kBeamRowImages images per CTA): the
// three serial row passes of the kernel above (max, sum exp, scores: ~2.5 k instructions per lane at V = 258) run side by
// side; the first warp of the image then draws the k winners exactly as above.  Per-candidate arithmetic and the order
// of every reduction are those of beam_step_warp_kernel: bit-identical outputs.
constexpr int kBeamRowImages = 2;
__global__ void __launch_bounds__(32 * 8 * kBeamRowImages)
beam_step_rows_kernel(const float* __restrict__ logits, int ld, int B, int k, int V, int eos, float lpw,
                      float* __restrict__ log_probs, uint8_t* __restrict__ finished, long long* __restrict__ lengths,
                      float* __restrict__ scores_out, int* __restrict__ word_out, int* __restrict__ parent_out,
                      int* __restrict__ tok_next, int* __restrict__ src_next, int* fin_count, int t, int n_rows) {
  if (step_stopped(fin_count, t, n_rows)) {
    if (blockIdx.x == 0 && threadIdx.x == 0) fin_count[t] = n_rows;
    return;
  }
  extern __shared__ float s_sc[];                       // [kBeamRowImages][k * V] candidate scores | [kBeamRowImages][k][2] max, lse
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int li = warp / k, j = warp - li * k;           // image within the CTA, beam row
  const int b = blockIdx.x * kBeamRowImages + li;
  const int ncand = k * V;
  float* sc = s_sc + (size_t)li * ncand;
  float* st = s_sc + (size_t)kBeamRowImages * ncand + (size_t)li * k * 2;
  const bool live = b < B;
  const float* base = logits + (size_t)(live ? b : 0) * k * ld;
  if (live) {
    const float cumj = log_probs[b * k + j];
    const bool finj = finished[b * k + j] != 0;
    const long long lenj = lengths[b * k + j];
    const float* row = base + (size_t)j * ld;
    float* srow = sc + j * V;
    float mx = -INFINITY;
    for (int i = lane; i < V; i += 32) {
      const float x = row[i];
      srow[i] = x;
      mx = fmaxf(mx, x);
    }
    mx = warp_max(mx);
    float sm = 0.f;
    for (int i = lane; i < V; i += 32) sm += expf(srow[i] - mx);
    sm = warp_sum(sm);
    const float lse = logf(sm);
    if (lane == 0) { st[j * 2] = mx; st[j * 2 + 1] = lse; }
    const float pen_live = (lpw == 0.0f) ? 1.0f : length_penalty_dev(lenj + (finj ? 0 : 1), lpw);
    const float pen_eos = (lpw == 0.0f) ? 1.0f : length_penalty_dev(lenj, lpw);
    for (int i = lane; i < V; i += 32) {
      float lp;
      if (finj) lp = (i == eos) ? 0.0f : -FLT_MAX;
      else lp = (srow[i] - mx) - lse;
      const float tot = cumj + lp;
      srow[i] = (lpw == 0.0f) ? tot : tot / ((i == eos) ? pen_eos : pen_live);
    }
  }
  __syncthreads();
  if (!live || j != 0) return;
  // lane j' < k keeps the state of beam row j'
  float cum = 0.f, mxr = 0.f, lser = 0.f;
  int fin = 0;
  long long len = 0;
  if (lane < k) {
    cum = log_probs[b * k + lane];
    fin = finished[b * k + lane];
    len = lengths[b * k + lane];
    mxr = st[lane * 2];
    lser = st[lane * 2 + 1];
  }
  float pv = INFINITY, myv = 0.f;
  int pi = -1, myi = 0x7fffffff;
  for (int sel = 0; sel < k; ++sel) {
    float bv = -INFINITY;
    int bi = 0x7fffffff;
    for (int idx = lane; idx < ncand; idx += 32) {
      const float s = sc[idx];
      const bool eligible = (s < pv) || (s == pv && idx > pi);
      if (eligible && better(s, idx, bv, bi)) { bv = s; bi = idx; }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (better(ov, oi, bv, bi)) { bv = ov; bi = oi; }
    }
    pv = bv; pi = bi;
    if (lane == sel) { myv = bv; myi = bi; }
  }
  int idx = myi;
  if (idx == 0x7fffffff) idx = 0;                      // only if every candidate is NaN
  const int par = (lane < k) ? idx / V : 0, w = idx - par * V;
  const float cum_p = __shfl_sync(0xffffffffu, cum, par), mx_p = __shfl_sync(0xffffffffu, mxr, par);
  const float lse_p = __shfl_sync(0xffffffffu, lser, par);
  const int fin_p = __shfl_sync(0xffffffffu, fin, par);
  const long long len_p = __shfl_sync(0xffffffffu, len, par);
  if (lane < k) {
    float lp;
    if (fin_p) lp = (w == eos) ? 0.0f : -FLT_MAX;
    else lp = (base[(size_t)par * ld + w] - mx_p) - lse_p;
    const bool nfin = fin_p || (w == eos);
    log_probs[b * k + lane] = cum_p + lp;
    finished[b * k + lane] = nfin ? 1 : 0;
    lengths[b * k + lane] = len_p + (fin_p ? 0 : 1);
    scores_out[b * k + lane] = myv;
    word_out[b * k + lane] = w;
    parent_out[b * k + lane] = par;
    if (tok_next) tok_next[b * k + lane] = w;
    if (src_next) src_next[b * k + lane] = b * k + par;
    if (fin_count && nfin) atomicAdd(&fin_count[t], 1);
  }
}

// Host-side choice between the two beam-step kernels.
static void launch_beam_step(const float* logits, int ld, int B, int k, int V, int eos, float lpw, float* log_probs,
                             uint8_t* finished, long long* lengths, float* scores_out, int* word_out, int* parent_out,
                             int* tok_next, int* src_next, int* fin_count, int t, int n_rows, cudaStream_t st) {
  if (k * V <= 1536 && k >= 2 && k <= 8 && B >= 2 * kBeamWarpImages) {
    const size_t smem = (size_t)kBeamRowImages * (k * V + 2 * k) * sizeof(float);
    beam_step_rows_kernel<<<(B + kBeamRowImages - 1) / kBeamRowImages, 32 * k * kBeamRowImages, smem, st>>>(
        logits, ld, B, k, V, eos, lpw, log_probs, finished, lengths, scores_out, word_out, parent_out, tok_next, src_next,
        fin_count, t, n_rows);
  } else if (k * V <= 1536 && k <= 32 && B >= 2 * kBeamWarpImages) {
    const size_t smem = (size_t)kBeamWarpImages * k * V * sizeof(float);
    BeamWarpArgs g{logits, ld, k, V, eos, lpw, log_probs, finished, lengths, scores_out, word_out, parent_out, tok_next, src_next,
                   fin_count, t};
    beam_step_warp_kernel<<<(B + kBeamWarpImages - 1) / kBeamWarpImages, 32 * kBeamWarpImages, smem, st>>>(g, B, n_rows);
  } else {
    beam_step_kernel<<<B, 256, 0, st>>>(logits, ld, k, V, eos, lpw, log_probs, finished, lengths, scores_out, word_out,
                                        parent_out, tok_next, src_next, fin_count, t, n_rows);
  }
}

// ---------------------------------------------------------------------------
// B2: GreedyEmbeddingHelper.sample + BasicDecoder bookkeeping, one CTA per row.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
greedy_step_kernel(const float* __restrict__ logits, int ld, int V, int eos, int* __restrict__ ids_t,
                   float* __restrict__ logits_t, int* __restrict__ tok_next, uint8_t* __restrict__ finished,
                   int* fin_count, int t, int n_rows) {
  if (step_stopped(fin_count, t, n_rows)) {
    if (blockIdx.x == 0 && threadIdx.x == 0) fin_count[t] = n_rows;
    return;
  }
  __shared__ GreedyStepSmem S;
  greedy_step_block<false>(S, threadIdx.x, blockIdx.x, logits, ld, V, eos, ids_t, logits_t, tok_next, finished,
                           fin_count, t);
}

// ---------------------------------------------------------------------------
// Loop end + finalisation.
// ---------------------------------------------------------------------------
// `abort` (persistent loop only): non-zero when the cooperative kernel gave up at a grid barrier -> T = -1.
__global__ void compute_T_kernel(const int* __restrict__ fin_count, int max_it, int n_rows, int* __restrict__ T_out,
                                 const unsigned* __restrict__ abort) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    if (abort && *abort) { *T_out = -1; return; }
    int T = max_it;
    for (int t = 0; t < max_it; ++t)
      if (fin_count[t] >= n_rows) { T = t + 1; break; }
    *T_out = T;
  }
}

// TF r1.9 beam_search_ops.gather_tree (CPU functor semantics), one thread per
// (batch, beam).  T_dev (optional) overrides max_time with the executed steps.
__global__ void gather_tree_kernel(const int* __restrict__ step_ids, const int* __restrict__ parent_ids,
                                   const int* __restrict__ max_seq_len, const long long* __restrict__ lengths64,
                                   int Tmax, const int* __restrict__ T_dev, int B, int k, int end_token,
                                   int* __restrict__ out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * k) return;
  int b = i / k, beam = i - b * k;
  int T = T_dev ? *T_dev : Tmax;
  for (int t = 0; t < Tmax; ++t) out[((size_t)t * B + b) * k + beam] = end_token;
  int msl;
  if (max_seq_len) msl = max_seq_len[b];
  else {
    long long mx = 0;
    for (int j = 0; j < k; ++j) mx = lengths64[b * k + j] > mx ? lengths64[b * k + j] : mx;
    msl = (int)mx;
  }
  int L = min(T, msl);
  if (L <= 0) return;
  out[((size_t)(L - 1) * B + b) * k + beam] = step_ids[((size_t)(L - 1) * B + b) * k + beam];
  int parent = parent_ids[((size_t)(L - 1) * B + b) * k + beam];
  for (int level = L - 2; level >= 0; --level) {
    if (parent < 0 || parent >= k) return;   // TF raises InvalidArgument; never happens for our parents
    out[((size_t)level * B + b) * k + beam] = step_ids[((size_t)level * B + b) * k + parent];
    parent = parent_ids[((size_t)level * B + b) * k + parent];
  }
  bool fin = false;
  for (int t = 0; t < L; ++t) {
    size_t o = ((size_t)t * B + b) * k + beam;
    if (fin) out[o] = end_token;
    else if (out[o] == end_token) fin = true;
  }
}

// TF r1.9 gather_tree_from_array restricted to the top beam: sorted0[t, b] =
// slot whose history row the reference gathers for (t, b, beam 0); -1 = the
// beam_width+1 sentinel (tf.gather_nd on GPU returns zeros there).
__global__ void sorted_top_beam_kernel(const int* __restrict__ parent_ids, const long long* __restrict__ lengths,
                                       int Tmax, const int* __restrict__ T_dev, int B, int k,
                                       int* __restrict__ sorted0) {
  int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const int T = *T_dev;
  const int sentinel = k + 1;
  long long mx = 0;
  for (int j = 0; j < k; ++j) mx = lengths[b * k + j] > mx ? lengths[b * k + j] : mx;
  int L = min(T, (int)mx);
  for (int t = 0; t < Tmax; ++t) sorted0[(size_t)t * B + b] = sentinel;
  auto masked = [&](int t, int j) -> int { return ((long long)t < lengths[b * k + j]) ? j : sentinel; };
  if (L > 0) {
    sorted0[(size_t)(L - 1) * B + b] = masked(L - 1, 0);
    int parent = parent_ids[((size_t)(L - 1) * B + b) * k + 0];
    for (int level = L - 2; level >= 0; --level) {
      if (parent < 0 || parent >= k) break;
      sorted0[(size_t)level * B + b] = masked(level, parent);
      parent = parent_ids[((size_t)level * B + b) * k + parent];
    }
    bool fin = false;
    for (int t = 0; t < L; ++t) {
      size_t o = (size_t)t * B + b;
      if (fin) sorted0[o] = sentinel;
      else if (sorted0[o] == sentinel) fin = true;
    }
  }
  // where(mask[t,b,0], sorted, beam_id 0)
  for (int t = 0; t < Tmax; ++t) {
    bool mk = (long long)t < lengths[b * k + 0];
    size_t o = (size_t)t * B + b;
    int s = mk ? sorted0[o] : 0;
    sorted0[o] = (s >= 0 && s < k) ? s : -1;
  }
}

// attn_out[b, h, t, m] = hist[t, b*k + sorted0[t,b], h*M + m]  (t < T), else 0.
// scale (optional, [T, B*k, H]): the streaming attention kernel leaves the history unnormalised and stores 1 / sum there.
__global__ void attn_top_gather_kernel(const float* __restrict__ hist, const float* __restrict__ scale,
                                       const int* __restrict__ sorted0, const int* __restrict__ T_dev, int Tmax, int B,
                                       int k, int HM, int M, float* __restrict__ out) {
  int t = blockIdx.x, b = blockIdx.y;
  int T = *T_dev;
  int s = sorted0 ? sorted0[(size_t)t * B + b] : 0;
  int H = HM / M;
  const size_t row = (size_t)t * B * k + (size_t)b * k + (s >= 0 ? s : 0);
  const float* src = (t < T && s >= 0) ? hist + row * HM : nullptr;
  const float* sc = (src && scale) ? scale + row * H : nullptr;
  for (int i = threadIdx.x; i < HM; i += blockDim.x) {
    int hh = i / M, m = i - hh * M;
    out[(((size_t)b * H + hh) * Tmax + t) * M + m] = src ? (sc ? src[i] * sc[hh] : src[i]) : 0.f;
  }
}

__global__ void fill_i32_kernel(int* p, int v, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}
__global__ void iota_div_kernel(int* p, int n, int div) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = i / div;
}
__global__ void beam_init_kernel(float* log_probs, uint8_t* finished, long long* lengths, int B, int k) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * k) return;
  int j = i % k;
  log_probs[i] = (j == 0) ? 0.0f : -INFINITY;
  finished[i] = (j == 0) ? 0 : 1;
  lengths[i] = 0;
}

// ---------------------------------------------------------------------------
// Bind-time packing: [W_o | pad | W_q] panel and its bias.
// ---------------------------------------------------------------------------
__global__ void pack_outq_kernel(const float* __restrict__ wo, const float* __restrict__ bo,
                                 const float* __restrict__ wq, float* __restrict__ outq,
                                 float* __restrict__ bias, int R, int V, int Vp) {
  int LQ = Vp + R;
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < (size_t)R * LQ) {
    int r = (int)(i / LQ), c = (int)(i % LQ);
    float v = 0.f;
    if (c < V) v = wo[(size_t)r * V + c];
    else if (c >= Vp) v = wq[(size_t)r * R + (c - Vp)];
    outq[i] = v;
  }
  if (i < (size_t)LQ) bias[i] = (i < (size_t)V) ? bo[i] : 0.f;
}

int decoder_configure() {
  COMIC_CHECK_CUDA(cudaFuncSetAttribute(attn_ctx_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
  return COMIC_OK;
}

// Tensor-path (3xTF32) panels of the decoder weights.
static int decoder_pack_tc(comic_handle_t h, Carver& cv, cudaStream_t st, bool dry) {
  int rc;
  const int XA = h->W + h->A;
  if (h->cell == COMIC_CELL_GRU) {
    if ((rc = pack_tc_weight(h, cv, h->pk.gru_gx, h->KX, 3 * h->R, 3 * h->R, 1, 1, h->pk.tc_gru_g, st, dry))) return rc;
    if ((rc = pack_tc_weight(h, cv, h->gru_cand_kernel + (size_t)XA * h->R, h->R, h->R, h->R, 1, 1, h->pk.tc_gru_c, st, dry)))
      return rc;
  } else {
    if ((rc = pack_tc_weight(h, cv, h->w.lstm_kernel, h->KX, 4 * h->R, 4 * h->R, 1, 1, h->pk.tc_lstm, st, dry))) return rc;
  }
  if ((rc = pack_tc_weight(h, cv, h->pk.outq, h->R, h->LQ, h->LQ, 1, 1, h->pk.tc_outq, st, dry))) return rc;
  if ((rc = pack_tc_weight(h, cv, h->w.memory_kernel, h->C, h->R, h->R, 1, 1, h->pk.tc_mem, st, dry))) return rc;
  if (h->cfg.fm_projection == 2)
    if ((rc = pack_tc_weight(h, cv, h->w.value_kernel, h->C, h->R, h->R, 1, 1, h->pk.tc_val, st, dry))) return rc;
  int ninit = (h->cfg.init_method == 1) ? h->R : XA;
  if ((rc = pack_tc_weight(h, cv, h->w.init_weight, h->E, ninit, ninit, 1, 1, h->pk.tc_init, st, dry))) return rc;
  return COMIC_OK;
}

int decoder_pack(comic_handle_t h, Carver& cv, cudaStream_t st, bool dry) {
  h->pk.outq = cv.take<float>((size_t)h->R * h->LQ);
  h->pk.outq_bias = cv.take<float>(h->LQ);
  if (h->cell == COMIC_CELL_GRU) h->pk.gru_gx = cv.take<float>((size_t)h->KX * 3 * h->R);
  if (dry) return decoder_pack_tc(h, cv, st, true);
  size_t n = (size_t)h->R * h->LQ;
  pack_outq_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(h->w.out_kernel, h->w.out_bias, h->w.query_kernel,
                                                               h->pk.outq, h->pk.outq_bias, h->R, h->V, h->Vp);
  COMIC_CHECK_CUDA(cudaGetLastError());
  if (h->cell == COMIC_CELL_GRU) {
    const size_t ng = (size_t)h->KX * 3 * h->R;
    pack_gru_gates_kernel<<<(unsigned)((ng + 255) / 256), 256, 0, st>>>(h->w.lstm_kernel, h->gru_cand_kernel, h->pk.gru_gx,
                                                                       h->KX, h->W + h->A, h->R);
    COMIC_CHECK_CUDA(cudaGetLastError());
  }
  return decoder_pack_tc(h, cv, st, false);
}

// ---------------------------------------------------------------------------
// Step driver shared by decode_step / greedy / beam.
// ---------------------------------------------------------------------------
static size_t step_smem_scores(int k, int R) { return (size_t)k * R * sizeof(float); }
static size_t step_smem_ctx(int k, int H, int M) {
  return ((((size_t)k * H * M + 3) & ~(size_t)3) + (size_t)kCtxSlices * 4 * 128) * sizeof(float);
}

template <int R, int H>
static cudaError_t launch_scores(comic_handle_t h, const StepIO& io, const StepBufs& sb, int B, int k,
                                 cudaStream_t st) {
  int M = h->M;
  // position slicing: fill the machine when there are few images
  int slices = (2 * h->num_sms) / B;
  if (slices < 1) slices = 1;
  if (slices > (M + 7) / 8) slices = (M + 7) / 8;
  int ppc = (M + slices - 1) / slices;
  ppc = (ppc + 7) / 8 * 8;
  slices = (M + ppc - 1) / ppc;
  dim3 grid(B, slices);
  size_t smem = step_smem_scores(k, R);
  if (h->cfg.alignment == 0)
    attn_scores_kernel<R, H, 0><<<grid, 256, smem, st>>>(io.keys, sb.lq, h->LQ, h->Vp, h->w.ln_gamma, h->w.ln_beta,
                                                       h->w.attention_v, h->w.temperature, sb.scores, k, M, ppc,
                                                       io.fin_count, io.t, io.n_rows);
  else
    attn_scores_kernel<R, H, 1><<<grid, 256, smem, st>>>(io.keys, sb.lq, h->LQ, h->Vp, h->w.ln_gamma, h->w.ln_beta,
                                                       h->w.attention_v, h->w.temperature, sb.scores, k, M, ppc,
                                                       io.fin_count, io.t, io.n_rows);
  return cudaGetLastError();
}

static int dispatch_scores(comic_handle_t h, const StepIO& io, const StepBufs& sb, int B, int k, cudaStream_t st) {
  cudaError_t e = cudaErrorInvalidValue;
  bool ok = true;
  Prof pf(h, T_SCORES, st, 0);
  if (h->R == 512) {
    switch (h->H) {
      case 1: e = launch_scores<512, 1>(h, io, sb, B, k, st); break;
      case 2: e = launch_scores<512, 2>(h, io, sb, B, k, st); break;
      case 4: e = launch_scores<512, 4>(h, io, sb, B, k, st); break;
      case 8: e = launch_scores<512, 8>(h, io, sb, B, k, st); break;
      case 16: e = launch_scores<512, 16>(h, io, sb, B, k, st); break;
      default: ok = false;
    }
  } else if (h->R == 256) {
    switch (h->H) {
      case 1: e = launch_scores<256, 1>(h, io, sb, B, k, st); break;
      case 4: e = launch_scores<256, 4>(h, io, sb, B, k, st); break;
      case 8: e = launch_scores<256, 8>(h, io, sb, B, k, st); break;
      default: ok = false;
    }
  } else if (h->R == 1024) {
    switch (h->H) {
      case 1: e = launch_scores<1024, 1>(h, io, sb, B, k, st); break;
      case 8: e = launch_scores<1024, 8>(h, io, sb, B, k, st); break;
      case 16: e = launch_scores<1024, 16>(h, io, sb, B, k, st); break;
      default: ok = false;
    }
  } else ok = false;
  COMIC_REQUIRE(ok, COMIC_E_UNSUPPORTED, "attention kernel not instantiated for rnn_size=%d heads=%d", h->R, h->H);
  h->launches++;
  COMIC_CHECK_CUDA(e);
  return COMIC_OK;
}

// Fused scores + softmax + context (attention.cuh), one CTA per image.
template <int R, int H, int MODE, bool FAST, int KB>
static cudaError_t launch_fused_kb(const AttnArgs& aa, int B, size_t smem, cudaStream_t st) {
  static PerDeviceOnce once;
  {
    cudaError_t e = once([&] { return cudaFuncSetAttribute(attn_fused_kernel<R, H, MODE, FAST, KB>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024); });
    if (e != cudaSuccess) return e;
  }
  attn_fused_kernel<R, H, MODE, FAST, KB><<<B, kAttnThreads, smem, st>>>(aa);
  return cudaGetLastError();
}

// KB = beams scored together per key row (register-resident ILP); k is covered by ceil(k / KB) chunks.
template <int R, int H, int MODE, bool FAST>
static cudaError_t launch_fused_one(const AttnArgs& aa, int B, size_t smem, cudaStream_t st) {
  const int k = aa.k;
  if (k == 1) return launch_fused_kb<R, H, MODE, FAST, 1>(aa, B, smem, st);
  if (k == 2 || k == 4) return launch_fused_kb<R, H, MODE, FAST, 2>(aa, B, smem, st);
  return launch_fused_kb<R, H, MODE, FAST, 3>(aa, B, smem, st);
}

template <int R, int H>
static cudaError_t launch_fused(comic_handle_t h, const AttnArgs& aa, int B, size_t smem, cudaStream_t st) {
  if (h->cfg.alignment != 0) return launch_fused_one<R, H, 1, false>(aa, B, smem, st);
  if (h->precision == 2) return launch_fused_one<R, H, 0, true>(aa, B, smem, st);
  return launch_fused_one<R, H, 0, false>(aa, B, smem, st);
}

// Returns 1 when the fused kernel was launched, 0 when the configuration is not covered
// (caller falls back to the sliced scores + context kernels), < 0 on error.
static int dispatch_fused(comic_handle_t h, const StepIO& io, const StepBufs& sb, int B, int k, float* ctx_dst,
                          int ld_ctx, cudaStream_t st) {
  if (io.no_fused) return 0;
  if (io.kstats != nullptr && io.att_mask == nullptr && io.alpha_pre == nullptr) {
    // streaming kernel (attention2.cuh); attn2_prepare has checked the configuration
    a2::Args aa{};
    aa.keys = io.keys; aa.kstats = io.kstats; aa.bound = io.abound; aa.lq = sb.lq; aa.ld_lq = h->LQ; aa.q_off = h->Vp;
    aa.gamma = h->w.ln_gamma; aa.beta = h->w.ln_beta; aa.vvec = h->w.attention_v; aa.temperature = h->w.temperature;
    aa.ctx_out = ctx_dst; aa.ld_ctx = ld_ctx; aa.hist_t = io.hist_t; aa.hist_scale = io.hist_scale; aa.B = B; aa.M = h->M;
    aa.fin_count = io.fin_count; aa.t = io.t; aa.n_rows = io.n_rows; aa.trace = nullptr;
    aa.scratch = io.a2_scratch; aa.counters = io.a2_counters;
    Prof pf(h, T_SCORES, st);
    COMIC_CHECK_CUDA(a2::launch(aa, k, h->num_sms, h->dev, st));
    return 1;
  }
  if (B < h->fused_min_images || h->VAL > 1024 || h->VAL % 4 != 0) return 0;
  size_t smem = attn_fused_smem(k, h->R, h->H, h->M, h->VAL);
  if (smem > 200 * 1024) return 0;
  AttnArgs aa{};
  aa.keys = io.keys; aa.values = io.values; aa.lq = sb.lq; aa.ld_lq = h->LQ; aa.q_off = h->Vp;
  aa.gamma = h->w.ln_gamma; aa.beta = h->w.ln_beta; aa.vvec = h->w.attention_v; aa.temperature = h->w.temperature;
  aa.ctx_out = ctx_dst; aa.ld_ctx = ld_ctx; aa.hist_t = io.hist_t; aa.hist_pre = io.alpha_pre; aa.att_mask = io.att_mask;
  aa.att_keep = io.att_keep; aa.k = k; aa.M = h->M; aa.VAL = h->VAL; aa.prob_fn = h->cfg.prob_fn;
  aa.fin_count = io.fin_count; aa.t = io.t; aa.n_rows = io.n_rows;
  cudaError_t e = cudaErrorInvalidValue;
  bool ok = true;
  Prof pf(h, T_SCORES, st);
  if (h->R == 512) {
    switch (h->H) {
      case 1: e = launch_fused<512, 1>(h, aa, B, smem, st); break;
      case 2: e = launch_fused<512, 2>(h, aa, B, smem, st); break;
      case 4: e = launch_fused<512, 4>(h, aa, B, smem, st); break;
      case 8: e = launch_fused<512, 8>(h, aa, B, smem, st); break;
      case 16: e = launch_fused<512, 16>(h, aa, B, smem, st); break;
      default: ok = false;
    }
  } else if (h->R == 256) {
    switch (h->H) {
      case 1: e = launch_fused<256, 1>(h, aa, B, smem, st); break;
      case 8: e = launch_fused<256, 8>(h, aa, B, smem, st); break;
      default: ok = false;
    }
  } else if (h->R == 1024) {
    switch (h->H) {
      case 1: e = launch_fused<1024, 1>(h, aa, B, smem, st); break;
      case 8: e = launch_fused<1024, 8>(h, aa, B, smem, st); break;
      default: ok = false;
    }
  } else ok = false;
  if (!ok) { h->launches--; return 0; }
  COMIC_CHECK_CUDA(e);
  return 1;
}

int attn2_prepare(comic_handle_t h, StepIO& io, const StepBufs& sb, int B, int k, bool masks, cudaStream_t st) {
  io.kstats = nullptr;
  io.abound = nullptr;
  io.a2_scratch = nullptr;
  io.a2_counters = nullptr;
  if (!h->attn2 || h->attn2_state < 0 || masks) return COMIC_OK;
  if (h->cfg.alignment != 0 || h->cfg.prob_fn != 0 || h->R != a2::kR || h->H != a2::kH || h->VAL != h->R ||
      io.values != io.keys || k < 1 || k > 3 || h->M % a2::kPos != 0 ||
      B < (h->fused_min_images == 48 ? h->attn2_min_images : h->fused_min_images) || !sb.kstats)
    return COMIC_OK;
  {
    Prof pf(h, T_MISC, st);
    COMIC_CHECK_CUDA(a2::launch_key_stats(io.keys, (long long)B * h->M, sb.kstats, h->w.attention_v, h->w.temperature,
                                          h->w.ln_gamma, h->w.ln_beta, sb.abound, st));
  }
  if (h->attn2_state == 0) {
    // once per weight binding: exp(score - bound) must not underflow to zero for a whole row, so the kernel is only
    // taken while 2 * bound stays well inside the fp32 exponent range (the one host synchronisation of this path)
    COMIC_REQUIRE(h->attn2_host != nullptr, COMIC_E_CUDA, "attn2: no pinned buffer");
    // the kernel writes entries 0..9 (8 head bounds, exponent shift, feasibility flag); the rest of the buffer is padding
    COMIC_CHECK_CUDA(cudaMemcpyAsync(h->attn2_host, sb.abound, 10 * sizeof(float), cudaMemcpyDeviceToHost, st));
    COMIC_CHECK_CUDA(cudaStreamSynchronize(st));
    bool ok = h->attn2_host[9] == 1.0f;                       // an exponent shift for the clamp-free reciprocal product exists
    for (int i = 0; i < a2::kH; ++i) ok = ok && (h->attn2_host[i] == h->attn2_host[i]) && h->attn2_host[i] <= 40.0f;
    h->attn2_state = ok ? 1 : -1;
    if (!ok) return COMIC_OK;
  }
  COMIC_CHECK_CUDA(cudaMemsetAsync(sb.a2_counters, 0, (size_t)B * sizeof(int), st));
  io.kstats = sb.kstats;
  io.abound = sb.abound;
  io.a2_scratch = sb.a2_scratch;
  io.a2_counters = sb.a2_counters;
  return COMIC_OK;
}

static int step_tail(comic_handle_t h, const StepIO& io, const StepBufs& sb, int B, int k, bool tma_lq, cudaStream_t st);

// The GRU cell of one step (see gru_gate_kernel): gate GEMM, gate kernel, candidate GEMM, update kernel.  The two GEMMs
// take the tensor / FFMA paths and split-K choices of the LSTM gate GEMM; their partials share StepBufs::gates.
static int run_gru_cell(comic_handle_t h, const StepIO& io, const StepBufs& sb, const APlain& a, int N, cudaStream_t st) {
  const int R = h->R, tot = N * R;
  const int* stop = io.fin_count ? io.fin_count + (io.t > 0 ? io.t - 1 : 0) : nullptr;
  const int stop_n = (io.fin_count && io.t > 0) ? io.n_rows : 0x7fffffff;
  const bool tc1 = use_tc_step(h, h->pk.tc_gru_g, N, 3 * R, h->KX, 1);
  GemmPlan p1 = plan_gemm(N, 3 * R, h->KX, h->num_sms, true);
  const int ks1 = tc1 ? tc_ksplit(h, N, 3 * R, h->KX, 1) : 1;
  const int nz1 = tc1 ? ks1 : gemm_num_partials(h->KX, p1);
  Epi e1{};
  e1.nroute = 1;
  e1.r[0] = Route{0, 3 * R, sb.gates, 3 * R, 0};
  e1.split_stride = (long long)N * 3 * R;
  e1.ksplit = ks1;
  e1.stop = stop;
  e1.stop_n = stop_n;
  {
    Prof pf(h, T_GATES, st);
    if (tc1) COMIC_CHECK_CUDA((tc::launch_gemm_tc<0>(a, h->pk.tc_gru_g, N, 3 * R, e1, h->num_sms, st)));
    else COMIC_CHECK_CUDA((launch_gemm<0, 4>(a, h->pk.gru_gx, 3 * R, N, 3 * R, h->KX, e1, p1, st)));
  }
  {
    Prof pf(h, T_LSTM, st);
    if (tc1)
      gru_gate_kernel<true><<<(tot + 255) / 256, 256, 0, st>>>(sb.gates, nz1, (size_t)N * 3 * R, h->w.lstm_bias, io.h_prev, io.src,
                                                              io.src_limit, N, R, sb.gru, io.fin_count, io.t, io.n_rows, io.gates_save);
    else
      gru_gate_kernel<false><<<(tot + 255) / 256, 256, 0, st>>>(sb.gates, nz1, (size_t)N * 3 * R, h->w.lstm_bias, io.h_prev, io.src,
                                                               io.src_limit, N, R, sb.gru, io.fin_count, io.t, io.n_rows, io.gates_save);
  }
  // candidate GEMM: (r*h) . candidate/kernel h-rows
  APlain ac{};
  ac.nseg = 1;
  ac.seg[0] = ASeg{sb.gru, nullptr, R, R, N};
  const float* kc_h = h->gru_cand_kernel + (size_t)(h->W + h->A) * R;
  const bool tc2 = use_tc_step(h, h->pk.tc_gru_c, N, R, R, 1);
  GemmPlan p2 = plan_gemm(N, R, R, h->num_sms, true);
  const int ks2 = tc2 ? tc_ksplit(h, N, R, R, 1) : 1;
  const int nz2 = tc2 ? ks2 : gemm_num_partials(R, p2);
  Epi e2{};
  e2.nroute = 1;
  e2.r[0] = Route{0, R, sb.gates, R, 0};
  e2.split_stride = (long long)N * R;
  e2.ksplit = ks2;
  e2.stop = stop;
  e2.stop_n = stop_n;
  {
    Prof pf(h, T_GATES, st);
    if (tc2) COMIC_CHECK_CUDA((tc::launch_gemm_tc<0>(ac, h->pk.tc_gru_c, N, R, e2, h->num_sms, st)));
    else COMIC_CHECK_CUDA((launch_gemm<0, 4>(ac, kc_h, R, N, R, R, e2, p2, st)));
  }
  {
    Prof pf(h, T_LSTM, st);
    if (tc1 || tc2)
      gru_update_kernel<true><<<(tot + 255) / 256, 256, 0, st>>>(sb.gates, nz2, (size_t)N * R, sb.gru, h->gru_cand_bias, io.h_prev,
                                                                io.src, io.src_limit, io.h_new, io.h_drop, io.out_mask, io.out_keep,
                                                                N, R, io.fin_count, io.t, io.n_rows, io.gates_save);
    else
      gru_update_kernel<false><<<(tot + 255) / 256, 256, 0, st>>>(sb.gates, nz2, (size_t)N * R, sb.gru, h->gru_cand_bias, io.h_prev,
                                                                 io.src, io.src_limit, io.h_new, io.h_drop, io.out_mask, io.out_keep,
                                                                 N, R, io.fin_count, io.t, io.n_rows, io.gates_save);
  }
  COMIC_CHECK_CUDA(cudaGetLastError());
  return COMIC_OK;
}

// One attention-wrapper step on N = B*k rows.
int run_step(comic_handle_t h, const StepIO& io, const StepBufs& sb, int B, int k, cudaStream_t st) {
  const int N = B * k, R = h->R, W = h->W, A = h->A;
  // --- gates = [emb(tok) ; ctx ; h] . K ---
  APlain a{};
  if (io.in_mask || io.force_dense) {
    // training path: x assembled densely so the input dropout mask can be applied (and x kept on the tape)
    assemble_x_kernel<<<N, 256, 0, st>>>(h->w.embedding_map, io.tok, h->V, h->cfg.embed_lookup, io.ctx_prev,
                                        sb.xdense, N, W, A);
    h->launches++;
    if (io.in_mask) {
      size_t nx = (size_t)N * (W + A);
      dropout_rows_kernel<<<(unsigned)((nx + 255) / 256), 256, 0, st>>>(sb.xdense, io.in_mask, io.in_keep, nx);
      h->launches++;
    }
    a.nseg = 2;
    a.seg[0] = ASeg{sb.xdense, nullptr, W + A, W + A, N};
    a.seg[1] = ASeg{io.h_prev, io.src, R, R, io.src_limit};
  } else {
    a.nseg = 3;
    a.seg[0] = ASeg{h->w.embedding_map, io.tok, W, W, h->V};
    a.seg[1] = ASeg{io.ctx_prev, io.src, A, A, io.src_limit};
    a.seg[2] = ASeg{io.h_prev, io.src, R, R, io.src_limit};
  }
  if (h->cell == COMIC_CELL_GRU) {
    const int rc = run_gru_cell(h, io, sb, a, N, st);
    if (rc) return rc;
    return step_tail(h, io, sb, B, k, false, st);
  }
  const bool tc1 = use_tc_step(h, h->pk.tc_lstm, N, 4 * R, h->KX, 1);
  GemmPlan p1 = plan_gemm(N, 4 * R, h->KX, h->num_sms, true);
  const int ks1 = tc1 ? tc_ksplit(h, N, 4 * R, h->KX, 1) : 1;
  int nz1 = tc1 ? ks1 : gemm_num_partials(h->KX, p1);
  Epi e1{};
  e1.nroute = 1;
  e1.r[0] = Route{0, 4 * R, sb.gates, 4 * R, 0};
  e1.split_stride = (long long)N * 4 * R;
  e1.ksplit = ks1;
  e1.stop = io.fin_count ? io.fin_count + (io.t > 0 ? io.t - 1 : 0) : nullptr;
  e1.stop_n = (io.fin_count && io.t > 0) ? io.n_rows : 0x7fffffff;
  // A operands as bf16 planes through TMA (inference decode on the tensor path: no dropout, no tape)
  const bool tma_ok = sb.tma_a && h->tma_a && h->precision >= 1 && !io.in_mask && !io.force_dense && !io.h_drop &&
                      !io.out_mask && !io.gates_save;
  const bool tma_gates = tma_ok && (h->tma_a & 2) && tc1 && ks1 == 1;
  // h' planes exist when the 4-units-per-thread LSTM kernel below runs
  const bool lstm4 = R % 4 == 0 && !io.h_drop && !io.out_mask && !io.gates_save && N >= 128 && (nz1 == 1 || (tc1 && h->precision >= 1));
  const bool tma_lq = tma_ok && (h->tma_a & 1) && lstm4 && R % 4 == 0 && N >= 128 &&
                      use_tc(h, h->pk.tc_outq, N);
  if (tma_gates) {
    Prof pf(h, T_GATES, st, 2);
    const int tot4 = N * (h->KX / 4);
    build_x_planes_kernel<<<(tot4 + 255) / 256, 256, 0, st>>>(h->w.embedding_map, io.tok, h->V, io.ctx_prev, io.h_prev, io.src,
                                                             io.src_limit, N, W, A, R, sb.xp_hi, sb.xp_lo, io.fin_count, io.t,
                                                             io.n_rows);
    COMIC_CHECK_CUDA((tc::launch_gemm_tc<4>(sb.xmaps, h->pk.tc_lstm, N, 4 * R, e1, h->num_sms, st)));
  } else {
    Prof pf(h, T_GATES, st);
    if (tc1) COMIC_CHECK_CUDA((tc::launch_gemm_tc<0>(a, h->pk.tc_lstm, N, 4 * R, e1, h->num_sms, st)));
    else COMIC_CHECK_CUDA((launch_gemm<0, 4>(a, h->w.lstm_kernel, 4 * R, N, 4 * R, h->KX, e1, p1, st)));
  }
  {
    Prof pf(h, T_LSTM, st);
    int tot = N * R;
    if (lstm4) {
      const int tot4 = N * (R / 4);
      if (h->precision >= 1 && nz1 > 1)
        lstm_pointwise4_kernel<true, true><<<(tot4 + 255) / 256, 256, 0, st>>>(
            sb.gates, h->w.lstm_bias, io.c_prev, io.src, io.src_limit, io.c_new, io.h_new, N, R, io.fin_count, io.t, io.n_rows,
            tma_lq ? sb.hp_hi : nullptr, tma_lq ? sb.hp_lo : nullptr, nz1, (size_t)N * 4 * R);
      else if (h->precision >= 1)
        lstm_pointwise4_kernel<true, false><<<(tot4 + 255) / 256, 256, 0, st>>>(
            sb.gates, h->w.lstm_bias, io.c_prev, io.src, io.src_limit, io.c_new, io.h_new, N, R, io.fin_count, io.t, io.n_rows,
            tma_lq ? sb.hp_hi : nullptr, tma_lq ? sb.hp_lo : nullptr, 1, (size_t)0);
      else
        lstm_pointwise4_kernel<false><<<(tot4 + 255) / 256, 256, 0, st>>>(sb.gates, h->w.lstm_bias, io.c_prev, io.src, io.src_limit,
                                                                         io.c_new, io.h_new, N, R, io.fin_count, io.t, io.n_rows);
    } else
    lstm_pointwise_kernel<<<(tot + 255) / 256, 256, 0, st>>>(sb.gates, nz1, (size_t)N * 4 * R, h->w.lstm_bias,
                                                          io.c_prev, io.src, io.src_limit, io.c_new, io.h_new,
                                                          io.h_drop, io.out_mask, io.out_keep, N, R, io.fin_count,
                                                          io.t, io.n_rows, io.gates_save);
  }
  return step_tail(h, io, sb, B, k, tma_lq, st);
}

// [logits | q] GEMM and attention of a step, after the cell has written h' (io.h_new / io.h_drop).
static int step_tail(comic_handle_t h, const StepIO& io, const StepBufs& sb, int B, int k, bool tma_lq, cudaStream_t st) {
  const int N = B * k, R = h->R, A = h->A;
  Epi e1{};   // stop condition of the step's launches
  e1.stop = io.fin_count ? io.fin_count + (io.t > 0 ? io.t - 1 : 0) : nullptr;
  e1.stop_n = (io.fin_count && io.t > 0) ? io.n_rows : 0x7fffffff;
  // --- [logits | q] = h_out . [W_o | W_q] + [b_o | 0] ---
  const float* hq = io.h_drop ? io.h_drop : io.h_new;
  APlain a2{};
  a2.nseg = 1;
  a2.seg[0] = ASeg{hq, nullptr, R, R, N};
  const bool tc2 = use_tc_step(h, h->pk.tc_outq, N, h->LQ, R, 2);
  GemmPlan p2 = plan_gemm(N, h->LQ, R, h->num_sms, true);
  const int ks2 = (tc2 && !tma_lq) ? tc_ksplit(h, N, h->LQ, R, 2) : 1;
  int nz2 = tc2 ? ks2 : gemm_num_partials(R, p2);
  Epi e2{};
  e2.nroute = 1;
  e2.stop = e1.stop;
  e2.stop_n = e1.stop_n;
  if (nz2 == 1) {
    e2.bias = h->pk.outq_bias;
    e2.r[0] = Route{0, h->LQ, sb.lq, h->LQ, 0};
    Prof pf(h, T_LQ, st);
    if (tc2 && tma_lq) COMIC_CHECK_CUDA((tc::launch_gemm_tc<4>(sb.hmaps, h->pk.tc_outq, N, h->LQ, e2, h->num_sms, st)));
    else if (tc2) COMIC_CHECK_CUDA((tc::launch_gemm_tc<0>(a2, h->pk.tc_outq, N, h->LQ, e2, h->num_sms, st)));
    else COMIC_CHECK_CUDA((launch_gemm<0, 4>(a2, h->pk.outq, h->LQ, N, h->LQ, R, e2, p2, st)));
  } else {
    e2.r[0] = Route{0, h->LQ, sb.lq_part, h->LQ, 0};
    e2.split_stride = (long long)N * h->LQ;
    e2.ksplit = tc2 ? ks2 : 0;
    Prof pf(h, T_LQ, st, 2);
    if (tc2) COMIC_CHECK_CUDA((tc::launch_gemm_tc<0>(a2, h->pk.tc_outq, N, h->LQ, e2, h->num_sms, st)));
    else COMIC_CHECK_CUDA((launch_gemm<0, 4>(a2, h->pk.outq, h->LQ, N, h->LQ, R, e2, p2, st)));
    size_t tot = (size_t)N * h->LQ;
    splitk_reduce_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(sb.lq_part, nz2, (size_t)N * h->LQ,
                                                                       h->pk.outq_bias, sb.lq, N, h->LQ,
                                                                       io.fin_count, io.t, io.n_rows);
  }
  // --- attention ---
  {
    int VAL = h->VAL;
    float* ctx_dst = h->cfg.context_layer ? sb.ctxraw : io.ctx_new;
    int ld_ctx = h->cfg.context_layer ? VAL : A;
    int rc = dispatch_fused(h, io, sb, B, k, ctx_dst, ld_ctx, st);
    if (rc < 0) return rc;
    if (rc == 0) {
      if ((rc = dispatch_scores(h, io, sb, B, k, st))) return rc;
      dim3 grid(B, (VAL + 127) / 128);
      size_t smem = step_smem_ctx(k, h->H, h->M);
      Prof pf(h, T_CTX, st);
      attn_ctx_kernel<<<grid, 128 * kCtxSlices, smem, st>>>(sb.scores, io.values, VAL, ctx_dst, ld_ctx, io.hist_t, io.att_mask,
                                              io.att_keep, k, h->H, h->M, h->cfg.prob_fn, io.fin_count, io.t,
                                              io.n_rows, io.alpha_pre);
    }
    COMIC_CHECK_CUDA(cudaGetLastError());
    if (h->cfg.context_layer) {
      APlain a3{};
      a3.nseg = 1;
      a3.seg[0] = ASeg{sb.ctxraw, nullptr, VAL, VAL, N};
      Epi e3{};
      e3.nroute = 1;
      e3.r[0] = Route{0, R, io.ctx_new, R, 0};
      e3.stop = e1.stop;
      e3.stop_n = e1.stop_n;
      GemmPlan p3 = plan_gemm(N, R, VAL, h->num_sms, false);
      Prof pf(h, T_CTX, st);
      COMIC_CHECK_CUDA((launch_gemm<0, 4>(a3, h->w.a_layer, R, N, R, VAL, e3, p3, st)));
    }
  }
  return COMIC_OK;
}

// GRU step from the zero state (first_input init, src/model_base.py:675-686): h0 = (1 - u0) * tanh(x0 . Kc_x + b_c), from the
// gate panel's x-rows; r * h is zero, so there is no candidate GEMM.  part: >= 16 * B * 3R floats of split-K partials,
// gru: [3][B][R]; tape (training) receives the rows [r0 | u0 | 0 | c0].
int gru_init_step(comic_handle_t h, const float* x0, int B, float* part, float* gru, float* h0, float* tape, cudaStream_t st) {
  const int R = h->R, XA = h->W + h->A;
  APlain a{};
  a.nseg = 1;
  a.seg[0] = ASeg{x0, nullptr, XA, XA, B};
  GemmPlan pg = plan_gemm(B, 3 * R, XA, h->num_sms, true);
  const int nz = gemm_num_partials(XA, pg);
  Epi eg{};
  eg.nroute = 1;
  eg.stop_n = 0x7fffffff;
  eg.r[0] = Route{0, 3 * R, part, 3 * R, 0};
  eg.split_stride = (long long)B * 3 * R;
  COMIC_CHECK_CUDA((launch_gemm<0, 4>(a, h->pk.gru_gx, 3 * R, B, 3 * R, XA, eg, pg, st)));
  const int tot = B * R;
  gru_gate_kernel<false><<<(tot + 255) / 256, 256, 0, st>>>(part, nz, (size_t)B * 3 * R, h->w.lstm_bias, nullptr, nullptr, 0, B, R,
                                                           gru, nullptr, 0, 0, tape);
  gru_update_kernel<false><<<(tot + 255) / 256, 256, 0, st>>>(nullptr, 0, 0, gru, h->gru_cand_bias, nullptr, nullptr, 0, h0, nullptr,
                                                             nullptr, 1.f, B, R, nullptr, 0, 0, tape);
  h->launches += 3;
  COMIC_CHECK_CUDA(cudaGetLastError());
  return COMIC_OK;
}

void carve_step(comic_handle_t h, Carver& cv, int N, StepBufs& sb, bool train_masks) {
  GemmPlan p1 = plan_gemm(N, 4 * h->R, h->KX, h->num_sms, true);
  int nz1 = gemm_num_partials(h->KX, p1);
  { const int ks = tc_ksplit_shape(h->num_sms, N, 4 * h->R, h->KX); if (nz1 < ks) nz1 = ks; }   // tensor-path split-K partials
  GemmPlan p2 = plan_gemm(N, h->LQ, h->R, h->num_sms, true);
  int nz2 = gemm_num_partials(h->R, p2);
  size_t ngates = (size_t)nz1 * N * 4 * h->R;
  if (h->cell == COMIC_CELL_GRU) {   // partials of the gate GEMM [N][3R] and, after the gate kernel, of the candidate GEMM [N][R]
    GemmPlan pg = plan_gemm(N, 3 * h->R, h->KX, h->num_sms, true), pc = plan_gemm(N, h->R, h->R, h->num_sms, true);
    const int nzg = std::max(gemm_num_partials(h->KX, pg), tc_ksplit_shape(h->num_sms, N, 3 * h->R, h->KX));
    const int nzc = std::max(gemm_num_partials(h->R, pc), tc_ksplit_shape(h->num_sms, N, h->R, h->R));
    ngates = std::max((size_t)nzg * N * 3 * h->R, (size_t)nzc * N * h->R);
  }
  sb.gates = cv.take<float>(ngates);
  sb.gru = (h->cell == COMIC_CELL_GRU) ? cv.take<float>((size_t)3 * N * h->R) : nullptr;
  { const int ks = tc_ksplit_shape(h->num_sms, N, h->LQ, h->R); if (nz2 < ks) nz2 = ks; }
  sb.lq_part = cv.take<float>(nz2 > 1 ? (size_t)nz2 * N * h->LQ : 1);
  sb.lq = cv.take<float>((size_t)N * h->LQ);
  sb.scores = cv.take<float>((size_t)N * h->H * h->M);
  sb.xdense = cv.take<float>(train_masks ? (size_t)N * (h->W + h->A) : 1);
  sb.ctxraw = cv.take<float>(h->cfg.context_layer ? (size_t)N * h->VAL : 1);
  const bool a2ok = h->cfg.alignment == 0 && h->cfg.prob_fn == 0 && h->R == a2::kR && h->H == a2::kH && h->VAL == h->R;
  sb.kstats = cv.take<float>(a2ok ? (size_t)N * h->M * 2 : 1);    // N >= number of images
  sb.abound = cv.take<float>(a2::kBoundFloats);
  sb.a2_scratch = cv.take<float>(a2ok ? a2::scratch_floats(h->num_sms) : 1);
  sb.a2_counters = cv.take<int>(a2ok ? (size_t)N : 1);
  // TMA-staged A planes (see StepBufs); the maps are encoded when the workspace is real
  const bool planes = h->tma_a && h->cell == COMIC_CELL_LSTM && !train_masks && N >= 128 && h->KX % 8 == 0 && h->R % 8 == 0 && h->W % 4 == 0 && h->A % 4 == 0;
  sb.xp_hi = cv.take<uint16_t>(planes ? (size_t)N * h->KX : 8);
  sb.xp_lo = cv.take<uint16_t>(planes ? (size_t)N * h->KX : 8);
  sb.hp_hi = cv.take<uint16_t>(planes ? (size_t)N * h->R : 8);
  sb.hp_lo = cv.take<uint16_t>(planes ? (size_t)N * h->R : 8);
  sb.tma_a = false;
  if (planes && cv.base != nullptr)
    sb.tma_a = tc::make_a_maps(sb.xmaps, sb.xp_hi, sb.xp_lo, N, h->KX) && tc::make_a_maps(sb.hmaps, sb.hp_hi, sb.hp_lo, N, h->R);
}

struct LoopBufs {
  StepBufs sb;
  float *c[2], *h[2], *ctx[2];
  float* hist;
  float* hist_scale;       // [T, N, H]: see attn_top_gather_kernel
  int *tok, *src, *src0;
  float* cum;
  uint8_t* fin;
  long long* len;
  int* fin_count;
  int *step_ids, *parents, *sorted0;
  float* scores_steps;
  unsigned* bar;
  long long* trace;
  float* part;
};

static void carve_loop(comic_handle_t h, Carver& cv, int B, int k, int T, bool want_hist, LoopBufs& lb) {
  int N = B * k;
  carve_step(h, cv, N, lb.sb, false);
  for (int i = 0; i < 2; ++i) {
    lb.c[i] = (h->cell == COMIC_CELL_GRU) ? nullptr : cv.take<float>((size_t)N * h->R);
    lb.h[i] = cv.take<float>((size_t)N * h->R);
    lb.ctx[i] = cv.take<float>((size_t)N * h->A);
  }
  lb.hist = cv.take<float>(want_hist ? (size_t)T * N * h->H * h->M : 1);
  lb.hist_scale = cv.take<float>(want_hist ? (size_t)T * N * h->H : 1);
  lb.tok = cv.take<int>(N);
  lb.src = cv.take<int>(N);
  lb.src0 = cv.take<int>(N);
  lb.cum = cv.take<float>(N);
  lb.fin = cv.take<uint8_t>(N);
  lb.len = cv.take<long long>(N);
  lb.fin_count = cv.take<int>(T + 1);
  lb.step_ids = cv.take<int>((size_t)T * N);
  lb.parents = cv.take<int>((size_t)T * N);
  lb.sorted0 = cv.take<int>((size_t)T * B);
  lb.scores_steps = cv.take<float>((size_t)T * N);
  lb.bar = cv.take<unsigned>(64);
  lb.trace = cv.take<long long>((size_t)T * 32 + 1);
  lb.part = cv.take<float>(N <= 32 ? (size_t)16 * N * 4 * h->R : 1);   // persistent loop only
}

int decoder_workspace_bytes(comic_handle_t h, int mode, int B, int k, int T, size_t* bytes) {
  Carver cv(nullptr);
  if (mode == 1) {
    LoopBufs lb;
    carve_loop(h, cv, B, 1, T, true, lb);
  } else if (mode == 2) {
    LoopBufs lb;
    carve_loop(h, cv, B, k, T, true, lb);
  } else if (mode == 3) {
    StepBufs sb;
    carve_step(h, cv, B * k, sb, true);
    cv.take<float>((size_t)B * k * h->R);
  } else if (mode == 4) {   // rnn_init
    cv.take<float>((size_t)B * (h->W + h->A));
    cv.take<float>((size_t)B * 4 * h->R * 16);
  } else {
    set_error("workspace_bytes: unknown mode %d", mode);
    return COMIC_E_BADARG;
  }
  *bytes = cv.off + 256;
  return COMIC_OK;
}

}  // namespace comic

using namespace comic;

// ===========================================================================
// C ABI
// ===========================================================================
extern "C" int comic_project_fm(comic_handle_t h, const float* fm, int B, float* keys_out, float* values_out,
                                void* stream) {
  COMIC_REQUIRE(h && h->bound, COMIC_E_BADARG, "project_fm: weights not bound");
  COMIC_REQUIRE(fm && keys_out && B > 0, COMIC_E_BADARG, "project_fm: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  int Mrows = B * h->M;
  APlain a{};
  a.nseg = 1;
  a.seg[0] = ASeg{fm, nullptr, h->C, h->C, Mrows};
  Epi e{};
  e.nroute = 1;
  e.r[0] = Route{0, h->R, keys_out, h->R, 0};
  e.stop_n = 0x7fffffff;
  GemmPlan p = plan_gemm(Mrows, h->R, h->C, h->num_sms, false);
  {
    Prof pf(h, T_PROJECT, st);
    if (use_tc(h, h->pk.tc_mem, Mrows)) COMIC_CHECK_CUDA((tc::launch_gemm_tc<0>(a, h->pk.tc_mem, Mrows, h->R, e, h->num_sms, st)));
    else COMIC_CHECK_CUDA((launch_gemm<0, 4>(a, h->w.memory_kernel, h->R, Mrows, h->R, h->C, e, p, st)));
  }
  if (h->cfg.fm_projection == 2) {
    COMIC_REQUIRE(values_out && h->w.value_kernel, COMIC_E_BADARG, "project_fm: independent projection needs values_out");
    e.r[0] = Route{0, h->R, values_out, h->R, 0};
    Prof pf(h, T_PROJECT, st);
    if (use_tc(h, h->pk.tc_val, Mrows)) COMIC_CHECK_CUDA((tc::launch_gemm_tc<0>(a, h->pk.tc_val, Mrows, h->R, e, h->num_sms, st)));
    else COMIC_CHECK_CUDA((launch_gemm<0, 4>(a, h->w.value_kernel, h->R, Mrows, h->R, h->C, e, p, st)));
  }
  return COMIC_OK;
}

extern "C" int comic_rnn_init(comic_handle_t h, const float* im_embed, int B, float* c0, float* h0,
                              const float* in_mask, float in_keep, void* ws, size_t ws_bytes, void* stream) {
  COMIC_REQUIRE(h && h->bound, COMIC_E_BADARG, "rnn_init: weights not bound");
  cudaStream_t st = (cudaStream_t)stream;
  const int R = h->R, XA = h->W + h->A;
  size_t need;
  decoder_workspace_bytes(h, 4, B, 1, 1, &need);
  COMIC_REQUIRE(ws_bytes >= need, COMIC_E_WORKSPACE, "rnn_init: workspace %zu < %zu", ws_bytes, need);
  Carver cv(ws);
  float* x0 = cv.take<float>((size_t)B * XA);
  float* gates = cv.take<float>((size_t)B * 4 * R * 16);
  APlain a{};
  a.nseg = 1;
  a.seg[0] = ASeg{im_embed, nullptr, h->E, h->E, B};
  Epi e{};
  e.nroute = 1;
  e.stop_n = 0x7fffffff;
  if (h->cfg.init_method == 1) {
    // project_hidden: h0 = im_embed . W, c0 = 0   (src/model_base.py:658-667)
    e.r[0] = Route{0, R, h0, R, 0};
    GemmPlan p = plan_gemm(B, R, h->E, h->num_sms, false);
    COMIC_CHECK_CUDA((launch_gemm<0, 4>(a, h->w.init_weight, R, B, R, h->E, e, p, st)));
    if (h->cell == COMIC_CELL_GRU) return COMIC_OK;   // state h only
    COMIC_CHECK_CUDA(cudaMemsetAsync(c0, 0, (size_t)B * R * sizeof(float), st));
    h->launches++;
    return COMIC_OK;
  }
  // first_input: x0 = im_embed . W_I ; one LSTM step from the zero state (:675-686)
  e.r[0] = Route{0, XA, x0, XA, 0};
  GemmPlan p = plan_gemm(B, XA, h->E, h->num_sms, false);
  COMIC_CHECK_CUDA((launch_gemm<0, 4>(a, h->w.init_weight, XA, B, XA, h->E, e, p, st)));
  h->launches++;
  if (in_mask) {
    size_t nx = (size_t)B * XA;
    dropout_rows_kernel<<<(unsigned)((nx + 255) / 256), 256, 0, st>>>(x0, in_mask, in_keep, nx);
    h->launches++;
  }
  APlain a2{};
  a2.nseg = 1;
  a2.seg[0] = ASeg{x0, nullptr, XA, XA, B};
  if (h->cell == COMIC_CELL_GRU) return gru_init_step(h, x0, B, gates, gates + (size_t)B * 3 * R * 16, h0, nullptr, st);
  GemmPlan p2 = plan_gemm(B, 4 * R, XA, h->num_sms, true);
  int nz = gemm_num_partials(XA, p2);
  Epi e2{};
  e2.nroute = 1;
  e2.stop_n = 0x7fffffff;
  e2.r[0] = Route{0, 4 * R, gates, 4 * R, 0};
  e2.split_stride = (long long)B * 4 * R;
  COMIC_CHECK_CUDA((launch_gemm<0, 4>(a2, h->w.lstm_kernel, 4 * R, B, 4 * R, XA, e2, p2, st)));
  int tot = B * R;
  lstm_pointwise_kernel<<<(tot + 255) / 256, 256, 0, st>>>(gates, nz, (size_t)B * 4 * R, h->w.lstm_bias, nullptr,
                                                        nullptr, 0, c0, h0, nullptr, nullptr, 1.f, B, R, nullptr, 0, 0, nullptr);
  h->launches += 2;
  COMIC_CHECK_CUDA(cudaGetLastError());
  return COMIC_OK;
}

extern "C" int comic_decode_step(comic_handle_t h, const float* keys, const float* values, int B, int k,
                                 const int32_t* tokens, const float* c_in, const float* h_in, const float* ctx_in,
                                 float* c_out, float* h_out, float* ctx_out, float* align_out, float* logits_out,
                                 const float* in_mask, const float* out_mask, const float* att_mask, float in_keep,
                                 float out_keep, float att_keep, void* ws, size_t ws_bytes, void* stream) {
  COMIC_REQUIRE(h && h->bound, COMIC_E_BADARG, "decode_step: weights not bound");
  COMIC_REQUIRE(keys && tokens && h_in && ctx_in && h_out && ctx_out && (h->cell == COMIC_CELL_GRU || (c_in && c_out)), COMIC_E_BADARG,
                "decode_step: null argument");
  COMIC_REQUIRE(B > 0 && k > 0 && k <= 16, COMIC_E_SHAPE, "decode_step: bad B=%d k=%d", B, k);
  cudaStream_t st = (cudaStream_t)stream;
  const int N = B * k;
  size_t need;
  decoder_workspace_bytes(h, 3, B, k, 1, &need);
  COMIC_REQUIRE(ws_bytes >= need, COMIC_E_WORKSPACE, "decode_step: workspace %zu < %zu", ws_bytes, need);
  Carver cv(ws);
  StepBufs sb;
  carve_step(h, cv, N, sb, true);
  float* hdrop = cv.take<float>((size_t)N * h->R);
  StepIO io{};
  io.keys = keys;
  io.values = (h->cfg.fm_projection == 1) ? keys : values;
  COMIC_REQUIRE(io.values, COMIC_E_BADARG, "decode_step: values required for this fm_projection");
  io.tok = tokens; io.src = nullptr; io.src_limit = N;
  io.c_prev = c_in; io.h_prev = h_in; io.ctx_prev = ctx_in;
  io.c_new = c_out; io.h_new = h_out; io.ctx_new = ctx_out;
  io.h_drop = out_mask ? hdrop : nullptr;
  io.hist_t = align_out;
  io.in_mask = in_mask; io.out_mask = out_mask; io.att_mask = att_mask;
  io.in_keep = in_keep; io.out_keep = out_keep; io.att_keep = att_keep;
  io.fin_count = nullptr; io.t = 0; io.n_rows = N;
  int rc = attn2_prepare(h, io, sb, B, k, in_mask || out_mask || att_mask, st);
  if (rc) return rc;
  rc = run_step(h, io, sb, B, k, st);
  if (rc) return rc;
  if (logits_out)
    COMIC_CHECK_CUDA(cudaMemcpy2DAsync(logits_out, (size_t)h->V * sizeof(float), sb.lq, (size_t)h->LQ * sizeof(float),
                                       (size_t)h->V * sizeof(float), N, cudaMemcpyDeviceToDevice, st));
  if (out_mask)   // the wrapper's cell_output is the dropped h; state h stays undropped
    (void)0;
  return COMIC_OK;
}

extern "C" int comic_decode_greedy(comic_handle_t h, const float* keys, const float* values, const float* c0,
                                   const float* h0, int B, int max_it, int32_t* ids_out, float* logits_out,
                                   float* attn_out, int32_t* T_out, void* ws, size_t ws_bytes, void* stream) {
  COMIC_REQUIRE(h && h->bound, COMIC_E_BADARG, "decode_greedy: weights not bound");
  COMIC_REQUIRE(keys && (c0 || h->cell == COMIC_CELL_GRU) && h0 && ids_out && T_out, COMIC_E_BADARG, "decode_greedy: null argument");
  COMIC_REQUIRE(B > 0 && max_it >= 0, COMIC_E_SHAPE, "decode_greedy: bad B=%d max_it=%d", B, max_it);
  cudaStream_t st = (cudaStream_t)stream;
  size_t need;
  decoder_workspace_bytes(h, 1, B, 1, max_it, &need);
  COMIC_REQUIRE(ws_bytes >= need, COMIC_E_WORKSPACE, "decode_greedy: workspace %zu < %zu", ws_bytes, need);
  const float* vals = (h->cfg.fm_projection == 1) ? keys : values;
  COMIC_REQUIRE(vals, COMIC_E_BADARG, "decode_greedy: values required for this fm_projection");
  Carver cv(ws);
  LoopBufs lb;
  carve_loop(h, cv, B, 1, max_it, true, lb);
  const int N = B;
  COMIC_CHECK_CUDA(cudaMemsetAsync(lb.fin_count, 0, (max_it + 1) * sizeof(int), st));
  COMIC_CHECK_CUDA(cudaMemsetAsync(lb.fin, 0, N, st));
  COMIC_CHECK_CUDA(cudaMemsetAsync(lb.ctx[0], 0, (size_t)N * h->A * sizeof(float), st));
  COMIC_CHECK_CUDA(cudaMemsetAsync(ids_out, 0, (size_t)max_it * N * sizeof(int), st));
  if (logits_out) COMIC_CHECK_CUDA(cudaMemsetAsync(logits_out, 0, (size_t)max_it * N * h->V * sizeof(float), st));
  fill_i32_kernel<<<(N + 255) / 256, 256, 0, st>>>(lb.tok, h->cfg.go_id, N);
  h->launches++;
  PersistCall pc{};
  pc.keys = keys; pc.values = vals; pc.c0 = c0; pc.h0 = h0;
  pc.B = B; pc.k = 1; pc.max_it = max_it; pc.greedy = 1; pc.lpw = 0.f;
  for (int i = 0; i < 2; ++i) { pc.c[i] = lb.c[i]; pc.h[i] = lb.h[i]; pc.ctx[i] = lb.ctx[i]; }
  pc.lq = lb.sb.lq; pc.scores = lb.sb.scores; pc.hist = attn_out ? lb.hist : nullptr;
  pc.tok = lb.tok; pc.src = lb.src; pc.cum = lb.cum; pc.fin = lb.fin; pc.len = lb.len; pc.fin_count = lb.fin_count;
  pc.step_ids = ids_out; pc.parents = nullptr; pc.sc = nullptr; pc.logits_out = logits_out; pc.bar = lb.bar; pc.trace = h->persist_trace ? lb.trace : nullptr; pc.part = lb.part;
  int persisted = (max_it > 0) ? decode_persistent(h, pc, st) : 0;
  if (persisted < 0) return persisted;
  StepIO io_a2{};
  io_a2.keys = keys; io_a2.values = vals;
  if (!persisted && max_it > 0) {
    int rc = attn2_prepare(h, io_a2, lb.sb, B, 1, false, st);
    if (rc) return rc;
  }
  for (int t = 0; t < max_it && !persisted; ++t) {
    int cur = t & 1;
    StepIO io{};
    io.keys = keys; io.values = vals;
    io.kstats = io_a2.kstats; io.abound = io_a2.abound; io.a2_scratch = io_a2.a2_scratch; io.a2_counters = io_a2.a2_counters;
    io.tok = lb.tok; io.src = nullptr; io.src_limit = N;
    io.c_prev = (t == 0) ? c0 : lb.c[cur];
    io.h_prev = (t == 0) ? h0 : lb.h[cur];
    io.ctx_prev = lb.ctx[cur];
    io.c_new = lb.c[cur ^ 1]; io.h_new = lb.h[cur ^ 1]; io.ctx_new = lb.ctx[cur ^ 1];
    io.hist_t = attn_out ? lb.hist + (size_t)t * N * h->H * h->M : nullptr;
    io.hist_scale = (attn_out && io.kstats) ? lb.hist_scale + (size_t)t * N * h->H : nullptr;
    io.in_keep = io.out_keep = io.att_keep = 1.f;
    io.fin_count = lb.fin_count; io.t = t; io.n_rows = N;
    int rc = run_step(h, io, lb.sb, B, 1, st);
    if (rc) return rc;
    greedy_step_kernel<<<N, 128, 0, st>>>(lb.sb.lq, h->LQ, h->V, h->cfg.eos_id, ids_out + (size_t)t * N,
                                         logits_out ? logits_out + (size_t)t * N * h->V : nullptr, lb.tok, lb.fin,
                                         lb.fin_count, t, N);
    h->launches++;
  }
  {
    Prof pf(h, T_FINAL, st);
    compute_T_kernel<<<1, 32, 0, st>>>(lb.fin_count, max_it, N, T_out, persisted ? lb.bar + 1 : nullptr);
    if (attn_out && max_it > 0) {
      dim3 g(max_it, B);
      attn_top_gather_kernel<<<g, 256, 0, st>>>(lb.hist, io_a2.kstats ? lb.hist_scale : nullptr, nullptr, T_out, max_it, B, 1,
                                               h->H * h->M, h->M, attn_out);
      h->launches++;
    }
  }
  COMIC_CHECK_CUDA(cudaGetLastError());
  return COMIC_OK;
}

extern "C" int comic_decode_beam(comic_handle_t h, const float* keys, const float* values, const float* c0,
                                 const float* h0, int B, int k, float lpw, int max_it, int32_t* pred_ids_out,
                                 int32_t* step_ids_out, int32_t* parent_ids_out, float* scores_out,
                                 int64_t* lengths_out, float* attn_top_out, int32_t* T_out, void* ws,
                                 size_t ws_bytes, void* stream) {
  COMIC_REQUIRE(h && h->bound, COMIC_E_BADARG, "decode_beam: weights not bound");
  COMIC_REQUIRE(keys && (c0 || h->cell == COMIC_CELL_GRU) && h0 && pred_ids_out && T_out, COMIC_E_BADARG, "decode_beam: null argument");
  COMIC_REQUIRE(B > 0 && k > 0 && k <= 16 && max_it >= 0, COMIC_E_SHAPE, "decode_beam: bad B=%d k=%d max_it=%d", B, k, max_it);
  COMIC_REQUIRE(k <= h->V, COMIC_E_SHAPE, "decode_beam: beam %d exceeds vocab %d", k, h->V);
  cudaStream_t st = (cudaStream_t)stream;
  size_t need;
  decoder_workspace_bytes(h, 2, B, k, max_it, &need);
  COMIC_REQUIRE(ws_bytes >= need, COMIC_E_WORKSPACE, "decode_beam: workspace %zu < %zu", ws_bytes, need);
  const float* vals = (h->cfg.fm_projection == 1) ? keys : values;
  COMIC_REQUIRE(vals, COMIC_E_BADARG, "decode_beam: values required for this fm_projection");
  Carver cv(ws);
  LoopBufs lb;
  carve_loop(h, cv, B, k, max_it, true, lb);
  const int N = B * k;
  int* step_ids = step_ids_out ? step_ids_out : lb.step_ids;
  int* parents = parent_ids_out ? parent_ids_out : lb.parents;
  float* sc = scores_out ? scores_out : lb.scores_steps;
  COMIC_CHECK_CUDA(cudaMemsetAsync(lb.fin_count, 0, (max_it + 1) * sizeof(int), st));
  COMIC_CHECK_CUDA(cudaMemsetAsync(lb.ctx[0], 0, (size_t)N * h->A * sizeof(float), st));
  COMIC_CHECK_CUDA(cudaMemsetAsync(step_ids, 0, (size_t)max_it * N * sizeof(int), st));
  COMIC_CHECK_CUDA(cudaMemsetAsync(parents, 0, (size_t)max_it * N * sizeof(int), st));
  COMIC_CHECK_CUDA(cudaMemsetAsync(sc, 0, (size_t)max_it * N * sizeof(float), st));
  fill_i32_kernel<<<(N + 255) / 256, 256, 0, st>>>(lb.tok, h->cfg.go_id, N);
  iota_div_kernel<<<(N + 255) / 256, 256, 0, st>>>(lb.src0, N, k);
  beam_init_kernel<<<(N + 255) / 256, 256, 0, st>>>(lb.cum, lb.fin, lb.len, B, k);
  h->launches += 3;
  PersistCall pc{};
  pc.keys = keys; pc.values = vals; pc.c0 = c0; pc.h0 = h0;
  pc.B = B; pc.k = k; pc.max_it = max_it; pc.greedy = 0; pc.lpw = lpw;
  for (int i = 0; i < 2; ++i) { pc.c[i] = lb.c[i]; pc.h[i] = lb.h[i]; pc.ctx[i] = lb.ctx[i]; }
  pc.lq = lb.sb.lq; pc.scores = lb.sb.scores; pc.hist = attn_top_out ? lb.hist : nullptr;
  pc.tok = lb.tok; pc.src = lb.src; pc.cum = lb.cum; pc.fin = lb.fin; pc.len = lb.len; pc.fin_count = lb.fin_count;
  pc.step_ids = step_ids; pc.parents = parents; pc.sc = sc; pc.logits_out = nullptr; pc.bar = lb.bar; pc.trace = h->persist_trace ? lb.trace : nullptr; pc.part = lb.part;
  int persisted = (max_it > 0) ? decode_persistent(h, pc, st) : 0;
  if (persisted < 0) return persisted;
  StepIO io_a2{};
  io_a2.keys = keys; io_a2.values = vals;
  if (!persisted && max_it > 0) {
    int rc = attn2_prepare(h, io_a2, lb.sb, B, k, false, st);
    if (rc) return rc;
  }
  for (int t = 0; t < max_it && !persisted; ++t) {
    int cur = t & 1;
    StepIO io{};
    io.keys = keys; io.values = vals;
    io.kstats = io_a2.kstats; io.abound = io_a2.abound; io.a2_scratch = io_a2.a2_scratch; io.a2_counters = io_a2.a2_counters;
    io.tok = lb.tok;
    if (t == 0) {
      io.src = lb.src0; io.src_limit = B;        // tile_batch: row n reads image n / k
      io.c_prev = c0; io.h_prev = h0;
      io.ctx_prev = lb.ctx[0];                   // zeros
    } else {
      io.src = lb.src; io.src_limit = N;
      io.c_prev = lb.c[cur]; io.h_prev = lb.h[cur]; io.ctx_prev = lb.ctx[cur];
    }
    io.c_new = lb.c[cur ^ 1]; io.h_new = lb.h[cur ^ 1]; io.ctx_new = lb.ctx[cur ^ 1];
    io.hist_t = attn_top_out ? lb.hist + (size_t)t * N * h->H * h->M : nullptr;
    io.hist_scale = (attn_top_out && io.kstats) ? lb.hist_scale + (size_t)t * N * h->H : nullptr;
    io.in_keep = io.out_keep = io.att_keep = 1.f;
    io.fin_count = lb.fin_count; io.t = t; io.n_rows = N;
    // (Tried: the beam-search step of an image inside the streaming attention kernel's finaliser warp -- it needs only the
    // logits -- to save the step's fifth launch.  The finaliser then prepares the next segment's queries late and the
    // attention launch grows by 29 us for the 15 us saved: profiles/r10a_bench512_fuse_beam=*.json.  Not kept.)
    int rc = run_step(h, io, lb.sb, B, k, st);
    if (rc) return rc;
    {
      Prof pf(h, T_BEAM, st);
      launch_beam_step(lb.sb.lq, h->LQ, B, k, h->V, h->cfg.eos_id, lpw, lb.cum, lb.fin, lb.len, sc + (size_t)t * N,
                       step_ids + (size_t)t * N, parents + (size_t)t * N, lb.tok, lb.src, lb.fin_count, t, N, st);
    }
  }
  Prof pf_final(h, T_FINAL, st, 2);
  compute_T_kernel<<<1, 32, 0, st>>>(lb.fin_count, max_it, N, T_out, persisted ? lb.bar + 1 : nullptr);
  gather_tree_kernel<<<(N + 127) / 128, 128, 0, st>>>(step_ids, parents, nullptr, lb.len, max_it, T_out, B, k,
                                                     h->cfg.eos_id, pred_ids_out);
  if (lengths_out)
    COMIC_CHECK_CUDA(cudaMemcpyAsync(lengths_out, lb.len, (size_t)N * sizeof(long long), cudaMemcpyDeviceToDevice, st));
  if (attn_top_out && max_it > 0) {
    sorted_top_beam_kernel<<<(B + 127) / 128, 128, 0, st>>>(parents, lb.len, max_it, T_out, B, k, lb.sorted0);
    dim3 g(max_it, B);
    attn_top_gather_kernel<<<g, 256, 0, st>>>(lb.hist, io_a2.kstats ? lb.hist_scale : nullptr, lb.sorted0, T_out, max_it, B, k,
                                             h->H * h->M, h->M, attn_top_out);
    h->launches += 2;
  }
  COMIC_CHECK_CUDA(cudaGetLastError());
  return COMIC_OK;
}

extern "C" int comic_beam_step(comic_handle_t h, const float* logits, int ld_logits, int B, int k, int V, int eos_id,
                               float lpw, float* log_probs, uint8_t* finished, int64_t* lengths, float* scores_out,
                               int32_t* word_out, int32_t* parent_out, void* stream) {
  COMIC_REQUIRE(h, COMIC_E_BADARG, "beam_step: null handle");
  COMIC_REQUIRE(logits && log_probs && finished && lengths && scores_out && word_out && parent_out, COMIC_E_BADARG,
                "beam_step: null argument");
  COMIC_REQUIRE(B > 0 && k > 0 && k <= 16 && V >= k && ld_logits >= V, COMIC_E_SHAPE, "beam_step: bad shape");
  launch_beam_step(logits, ld_logits, B, k, V, eos_id, lpw, log_probs, finished, (long long*)lengths, scores_out, word_out,
                   parent_out, nullptr, nullptr, nullptr, 0, B * k, (cudaStream_t)stream);
  h->launches++;
  COMIC_CHECK_CUDA(cudaGetLastError());
  return COMIC_OK;
}

extern "C" int comic_gather_tree(comic_handle_t h, const int32_t* step_ids, const int32_t* parent_ids,
                                 const int32_t* max_seq_len, int T, int B, int k, int end_token, int32_t* out,
                                 void* stream) {
  COMIC_REQUIRE(h && step_ids && parent_ids && max_seq_len && out, COMIC_E_BADARG, "gather_tree: null argument");
  if (T <= 0 || B <= 0 || k <= 0) return COMIC_OK;
  gather_tree_kernel<<<(B * k + 127) / 128, 128, 0, (cudaStream_t)stream>>>(step_ids, parent_ids, max_seq_len, nullptr,
                                                                            T, nullptr, B, k, end_token, out);
  h->launches++;
  COMIC_CHECK_CUDA(cudaGetLastError());
  return COMIC_OK;
}
