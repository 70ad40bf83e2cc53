// train.cu -- teacher-forced decoder forward + fused backward for the `decoder`
// and `scst` train modes, TF-form Adam and the L2 term, for sm_100a.
//
// Replaces the TF graph built by
//   rnn_decoder_training                  common/ops_rnn.py:183-243
//     (TrainingHelper + BasicDecoder + dynamic_decode(impute_finished=True))
//   ModelBase._train_caption_model        src/model_base.py:325-405
//     (sequence_loss XE / SCST weighting, attention-map loss, tf.gradients)
//   ModelBase._loss_regularisation        src/model_base.py:408-417
//   tf.train.AdamOptimizer                src/model_base.py:852-861 (epsilon-hat form)
// and the autodiff the reference gets from `slim.learning.create_train_op`.
//
// Forward: the inference step driver (decoder.cu run_step) with the dropout masks
// of DropoutWrapper / attention-map dropout, writing a tape (inputs, gate
// pre-activations, states, pre/post-dropout alignments).  Backward: one reverse
// sweep of small kernels (attention backward with LN-tanh recompute, LSTM
// pointwise backward) and two skinny GEMMs per step (dh = dlq.[W_o|W_q]^T,
// dxh = dgates.K^T); every weight gradient is ONE batched GEMM over all
// T*B rows after the sweep (dK = XH^T.dG, d[W_o|W_q] = Hout^T.dLQ,
// dW_k = F^T.dKeys, dW_I = E^T.dx0).  All reductions run in a fixed order:
// gradients are bit-reproducible run to run.
#include <math.h>

#include "comic_internal.cuh"

namespace comic {

__device__ __forceinline__ float sigm(float x) { return 1.0f / (1.0f + expf(-x)); }

__device__ __forceinline__ float wred_sum(float v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---------------------------------------------------------------------------
// Philox4x32-10 counter RNG -> 0/1 keep masks (tf.nn.dropout semantics: keep with
// probability `keep`; the scaling 1/keep is applied where the mask is consumed).
// ---------------------------------------------------------------------------
__device__ __forceinline__ void philox_round(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
  uint32_t hi0 = __umulhi(M0, c[0]), lo0 = M0 * c[0];
  uint32_t hi1 = __umulhi(M1, c[2]), lo1 = M1 * c[2];
  uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
  c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
}

__global__ void dropout_mask_kernel(float* __restrict__ out, size_t n, float keep, unsigned long long seed,
                                    unsigned long long stream_id) {
  size_t i4 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i4 * 4 >= n) return;
  uint32_t c[4] = {(uint32_t)i4, (uint32_t)(i4 >> 32), (uint32_t)stream_id, (uint32_t)(stream_id >> 32)};
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    philox_round(c, k0, k1);
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    size_t i = i4 * 4 + j;
    if (i < n) out[i] = ((c[j] >> 8) * (1.0f / 16777216.0f) < keep) ? 1.0f : 0.0f;
  }
}

// ---------------------------------------------------------------------------
// Generic helpers.
// ---------------------------------------------------------------------------
// dst[c, r] = src[r, c]   (src [rows, cols] row stride ld_src; dst row stride ld_dst)
__global__ void transpose_kernel(const float* __restrict__ src, int rows, int cols, int ld_src,
                                 float* __restrict__ dst, int ld_dst) {
  __shared__ float tile[32][33];
  int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    int r = r0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (r < rows && c < cols) ? src[(size_t)r * ld_src + c] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    int c = c0 + i, r = r0 + threadIdx.x;
    if (c < cols && r < rows) dst[(size_t)c * ld_dst + r] = tile[threadIdx.x][i];
  }
}

// out[c] (+)= sum_r src[r, c]; 32 columns x 8 row lanes per CTA (launch with 256 threads, grid = ceil(cols / 32)):
// each lane a strided partial, then a fixed-order sum of the 8 lanes (deterministic).  One thread walking all
// T*B rows of its column took 45 us per call (profiles/r02j).
__global__ void __launch_bounds__(256)
colsum_kernel(const float* __restrict__ src, int rows, int cols, int ld, float* __restrict__ out, int accumulate) {
  __shared__ float red[8][33];
  const int cl = threadIdx.x & 31, rl = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + cl;
  float s = 0.f;
  if (c < cols)
    for (int r = rl; r < rows; r += 8) s += src[(size_t)r * ld + c];
  red[rl][cl] = s;
  __syncthreads();
  if (rl == 0 && c < cols) {
    float t = red[0][cl];
#pragma unroll
    for (int j = 1; j < 8; ++j) t += red[j][cl];
    out[c] = accumulate ? out[c] + t : t;
  }
}

__global__ void copy2d_kernel(const float* __restrict__ src, int ld_src, float* __restrict__ dst, int ld_dst,
                              int rows, int cols) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)rows * cols) return;
  int r = (int)(i / cols), c = (int)(i % cols);
  dst[(size_t)r * ld_dst + c] = src[(size_t)r * ld_src + c];
}

// x = x / keep * mask
__global__ void mask_scale_kernel(float* __restrict__ x, const float* __restrict__ mask, float keep, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) x[i] = (x[i] / keep) * mask[i];
}

// BasicLSTMCell forward from the zero state (init step): gates = sum of split-K partials + bias.
__global__ void lstm_init_fwd_kernel(const float* __restrict__ gp, int nz, size_t zstride, const float* __restrict__ bias,
                                     float* __restrict__ gates_save, float* __restrict__ c_new, float* __restrict__ h_new,
                                     int B, int R) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * R) return;
  int n = i / R, j = i - n * R;
  float g[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    float s = 0.f;
    for (int z = 0; z < nz; ++z) s += gp[z * zstride + (size_t)n * 4 * R + q * R + j];
    g[q] = s + bias[q * R + j];
    gates_save[(size_t)n * 4 * R + q * R + j] = g[q];
  }
  float cn = sigm(g[0]) * tanhf(g[1]);
  c_new[i] = cn;
  h_new[i] = tanhf(cn) * sigm(g[3]);
}

// out[b, h, t, m] = hist[t, b, h*M + m]   (src/model_base.py:307-313)
__global__ void attn_maps_kernel(const float* __restrict__ hist, int T_run, int B, int H, int M, float* __restrict__ out) {
  int t = blockIdx.x, b = blockIdx.y;
  const float* src = hist + ((size_t)t * B + b) * H * M;
  for (int i = threadIdx.x; i < H * M; i += blockDim.x) {
    int hh = i / M, m = i - hh * M;
    out[(((size_t)b * H + hh) * T_run + t) * M + m] = src[i];
  }
}

__global__ void splitk_reduce2d_kernel(const float* __restrict__ part, int nz, size_t zstride, float* __restrict__ C,
                                       int ldc, int M, int N) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)M * N) return;
  int r = (int)(i / N), c = (int)(i % N);
  float s = 0.f;
  for (int z = 0; z < nz; ++z) s += part[z * zstride + i];
  C[(size_t)r * ldc + c] = s;
}

// TrainingHelper + impute_finished=True: rows with t >= len keep their previous state.
__global__ void impute_state_kernel(const int* __restrict__ lens, int t, int B, int R, int A,
                                    const float* __restrict__ c_old, const float* __restrict__ h_old,
                                    const float* __restrict__ ctx_old, float* __restrict__ c_new,
                                    float* __restrict__ h_new, float* __restrict__ ctx_new) {
  int b = blockIdx.x;
  if (t < lens[b]) return;
  for (int j = threadIdx.x; j < R; j += blockDim.x) {
    c_new[(size_t)b * R + j] = c_old[(size_t)b * R + j];
    h_new[(size_t)b * R + j] = h_old[(size_t)b * R + j];
  }
  for (int j = threadIdx.x; j < A; j += blockDim.x) ctx_new[(size_t)b * A + j] = ctx_old[(size_t)b * A + j];
}

// ---------------------------------------------------------------------------
// T3: sequence_loss.  One CTA per (t, b) row: log-softmax, xent * coef, and
// dlogits = coef * (softmax - onehot) written into dlq[t][b][0:V] (the query
// part of the row is filled by the attention backward).  coef[b, t] already
// holds weight / normaliser (XE) or reward/B * weight / row normaliser (SCST),
// src/model_base.py:337-347.  Also emits the imputed logits [B, T, V].
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
xent_kernel(const float* __restrict__ lq, int ld, int V, const int* __restrict__ targets_tm,
            const float* __restrict__ coef_tm, const int* __restrict__ lens, int B, int T_run, int T,
            float* __restrict__ dlq, float* __restrict__ row_loss, float* __restrict__ logits_out) {
  __shared__ float red[8];
  const int t = blockIdx.x / B, b = blockIdx.x - t * B;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float* row = lq + ((size_t)t * B + b) * ld;
  float* drow = dlq + ((size_t)t * B + b) * ld;
  const bool fin = t >= lens[b];           // imputed: the emitted logits are zeros
  const float cf = coef_tm[(size_t)t * B + b];
  const int tgt = targets_tm[(size_t)t * B + b];
  float mx = -INFINITY;
  for (int i = tid; i < V; i += 256) mx = fmaxf(mx, fin ? 0.f : row[i]);
#pragma unroll
  for (int o = 16; o; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if (lane == 0) red[warp] = mx;
  __syncthreads();
  mx = red[0];
#pragma unroll
  for (int w = 1; w < 8; ++w) mx = fmaxf(mx, red[w]);
  __syncthreads();
  float sm = 0.f;
  for (int i = tid; i < V; i += 256) sm += expf((fin ? 0.f : row[i]) - mx);
  sm = wred_sum(sm);
  if (lane == 0) red[warp] = sm;
  __syncthreads();
  float tot = 0.f;
#pragma unroll
  for (int w = 0; w < 8; ++w) tot += red[w];
  const float lse = logf(tot);
  for (int i = tid; i < V; i += 256) {
    float x = fin ? 0.f : row[i];
    float p = expf(x - mx) / tot;
    drow[i] = fin ? 0.f : cf * (p - (i == tgt ? 1.f : 0.f));
    if (logits_out) {
      // [B, T, V]; steps beyond T_run repeat the last executed step (ops_rnn.py:237-241)
      logits_out[((size_t)b * T + t) * V + i] = x;
      if (t == T_run - 1)
        for (int tt = T_run; tt < T; ++tt) logits_out[((size_t)b * T + tt) * V + i] = x;
    }
  }
  for (int i = V + tid; i < ld; i += 256) drow[i] = 0.f;     // pad + query columns (query filled later)
  if (tid == 0) {
    float x = fin ? 0.f : row[tgt];
    row_loss[(size_t)t * B + b] = cf * (-((x - mx) - lse));
  }
}

// ---------------------------------------------------------------------------
// Attention backward, part 1 (one CTA per image, k rows): from dctx and the map
// loss to dscore:  dalpha~ = V.dctx + dmap ; dalpha = dalpha~ * mask / keep ;
// ds = alpha (dalpha - <alpha, dalpha>)  (softmax), dT += -1/T sum ds log alpha.
// Also dvalues[b, m, c] += alpha~[h(c), m] dctx[c]   (tied: the keys' gradient).
// ---------------------------------------------------------------------------
// Part 1a, parallel over position slices (grid: image x slice): dalpha~[n, h, m] = sum_{c in h} dctx[c] V[m, c]
// into `dal_out` [N, H, M] and dV[b, m, c] += alpha~[h(c), m] dctx[c].  One CTA per image left 3/4 of the SMs idle
// at batch 32 (257 us per step = 47 % of the training step, profiles/r02c); every (image, position) is still
// owned by exactly one warp, so the accumulation into dV stays deterministic.
__global__ void __launch_bounds__(256)
attn_bwd_dalpha_kernel(const float* __restrict__ values, int VAL, const float* __restrict__ dctx, int ld_dctx,
                       const int* __restrict__ lens, int t, const float* __restrict__ a_post,
                       float* __restrict__ dvalues, float* __restrict__ dal_out, int k, int H, int M, int S) {
  const int b = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int dv = VAL / H;
  const int per = (M + S - 1) / S;
  const int m0 = blockIdx.y * per, m1 = min(M, m0 + per);
  for (int beam = 0; beam < k; ++beam) {
    const int n = b * k + beam;
    const bool fin = lens && t >= lens[n];
    const float* dc = dctx + (size_t)n * ld_dctx;
    const float* ap = a_post + (size_t)n * H * M;
    for (int m = m0 + warp; m < m1; m += 8) {
      const float* vr = values + ((size_t)b * M + m) * VAL;
      float* dvr = dvalues ? dvalues + ((size_t)b * M + m) * VAL : nullptr;
      for (int hh = 0; hh < H; ++hh) {
        float acc = 0.f;
        const float al = ap[(size_t)hh * M + m];
        for (int c = hh * dv + lane; c < (hh + 1) * dv; c += 32) {
          float g = fin ? 0.f : dc[c];
          acc = fmaf(g, vr[c], acc);
          if (dvr && !fin) dvr[c] += al * g;
        }
        acc = wred_sum(acc);
        if (lane == 0) dal_out[((size_t)n * H + hh) * M + m] = acc;
      }
    }
  }
}

// The same with lane-contiguous channels (VAL / 32 per lane, 128-bit accesses; needs head size % (VAL / 32) == 0): d ctx of
// the row is loaded once per beam instead of once per position and head, a position costs one round of independent loads
// (the scalar version's head loop was a chain of dependent L2 round trips: 36 us per launch at batch 32, long-scoreboard
// stall 17.9 per issued instruction, profiles/r12t_train_attn_summary.txt), and the per-head dot product is reduced over
// the 2..32 lanes of the head only.
template <int VAL>
__global__ void __launch_bounds__(256)
attn_bwd_dalpha_vec_kernel(const float* __restrict__ values, const float* __restrict__ dctx, int ld_dctx,
                           const int* __restrict__ lens, int t, const float* __restrict__ a_post,
                           float* __restrict__ dvalues, float* __restrict__ dal_out, int k, int H, int M, int S) {
  constexpr int CPL = VAL / 32;
  const int b = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int dv = VAL / H;
  const int c0 = lane * CPL;
  const int hh = c0 / dv;                       // this lane's head
  const int lph = dv / CPL;                     // lanes per head (a power of two)
  const int per = (M + S - 1) / S;
  const int m0 = blockIdx.y * per, m1 = min(M, m0 + per);
  for (int beam = 0; beam < k; ++beam) {
    const int n = b * k + beam;
    const bool fin = lens && t >= lens[n];
    float g[CPL];
#pragma unroll
    for (int c4 = 0; c4 < CPL / 4; ++c4) {
      const float4 v = fin ? make_float4(0.f, 0.f, 0.f, 0.f) : ldg4(dctx + (size_t)n * ld_dctx + c0 + c4 * 4);
      g[c4 * 4 + 0] = v.x; g[c4 * 4 + 1] = v.y; g[c4 * 4 + 2] = v.z; g[c4 * 4 + 3] = v.w;
    }
    const float* ap = a_post + ((size_t)n * H + hh) * M;
    for (int m = m0 + warp; m < m1; m += 8) {
      const float* vr = values + ((size_t)b * M + m) * VAL + c0;
      const float al = ap[m];
      float acc = 0.f;
      float4 vv[CPL / 4];
#pragma unroll
      for (int c4 = 0; c4 < CPL / 4; ++c4) vv[c4] = ldg4(vr + c4 * 4);
      if (dvalues != nullptr && !fin) {
        float* dvr = dvalues + ((size_t)b * M + m) * VAL + c0;
#pragma unroll
        for (int c4 = 0; c4 < CPL / 4; ++c4) {
          float4 d = *reinterpret_cast<const float4*>(dvr + c4 * 4);
          d.x = fmaf(al, g[c4 * 4 + 0], d.x); d.y = fmaf(al, g[c4 * 4 + 1], d.y);
          d.z = fmaf(al, g[c4 * 4 + 2], d.z); d.w = fmaf(al, g[c4 * 4 + 3], d.w);
          *reinterpret_cast<float4*>(dvr + c4 * 4) = d;
        }
      }
#pragma unroll
      for (int c4 = 0; c4 < CPL / 4; ++c4) {
        acc = fmaf(g[c4 * 4 + 0], vv[c4].x, acc); acc = fmaf(g[c4 * 4 + 1], vv[c4].y, acc);
        acc = fmaf(g[c4 * 4 + 2], vv[c4].z, acc); acc = fmaf(g[c4 * 4 + 3], vv[c4].w, acc);
      }
      for (int o = lph >> 1; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      if ((lane & (lph - 1)) == 0) dal_out[((size_t)n * H + hh) * M + m] = acc;
    }
  }
}

__global__ void __launch_bounds__(256)
attn_bwd_score_kernel(const float* __restrict__ values, int VAL, const float* __restrict__ dctx, int ld_dctx,
                      const int* __restrict__ lens, int t, const float* __restrict__ a_post,
                      const float* __restrict__ a_pre, const float* __restrict__ att_mask, float att_keep,
                      float map_coef, float* __restrict__ dvalues, float* __restrict__ ds_out,
                      float* __restrict__ dT_acc, float* __restrict__ map_rows, const float* __restrict__ temperature,
                      int k, int H, int M, const float* dal_in, const float* __restrict__ s_in) {
  extern __shared__ float sm[];            // dal [H][M]
  __shared__ float red[8];
  const int b = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int dv = VAL / H;
  for (int beam = 0; beam < k; ++beam) {
    const int n = b * k + beam;
    const bool fin = lens && t >= lens[n];   // imputed step: the cell's context output is discarded
    const float* dc = dctx + (size_t)n * ld_dctx;
    const float* ap = a_post + (size_t)n * H * M;
    // dalpha~[h, m] = sum_{c in h} dctx[c] V[m, c]; dV += alpha~ dctx  (or precomputed by attn_bwd_dalpha_kernel;
    // dal_in may alias ds_out: it is copied to shared memory before anything is written)
    if (dal_in) {
      for (int i = tid; i < H * M; i += 256) sm[i] = dal_in[(size_t)n * H * M + i];
    } else
    for (int m = warp; m < M; m += 8) {
      const float* vr = values + ((size_t)b * M + m) * VAL;
      float* dvr = dvalues ? dvalues + ((size_t)b * M + m) * VAL : nullptr;
      for (int hh = 0; hh < H; ++hh) {
        float acc = 0.f;
        const float al = ap[(size_t)hh * M + m];
        for (int c = hh * dv + lane; c < (hh + 1) * dv; c += 32) {
          float g = fin ? 0.f : dc[c];
          acc = fmaf(g, vr[c], acc);
          if (dvr && !fin) dvr[c] += al * g;
        }
        acc = wred_sum(acc);
        if (lane == 0) sm[hh * M + m] = acc;
      }
    }
    __syncthreads();
    // attention-map loss: d/dalpha~ of scale * mean((1 - sum_h alpha~)^2)   (model_base.py:356-365)
    float mrow = 0.f;
    for (int m = tid; m < M; m += 256) {
      float s = 0.f;
      for (int hh = 0; hh < H; ++hh) s += ap[(size_t)hh * M + m];
      float d = 1.0f - s;
      mrow += d * d;
      for (int hh = 0; hh < H; ++hh) sm[hh * M + m] += map_coef * d;
    }
    // deterministic block sum of mrow
    mrow = wred_sum(mrow);
    if (lane == 0) red[warp] = mrow;
    __syncthreads();
    if (tid == 0) {
      float s = 0.f;
      for (int w = 0; w < 8; ++w) s += red[w];
      map_rows[n] = s;
    }
    // softmax backward per head (warp per head)
    float dT_part = 0.f;
    for (int hh = warp; hh < H; hh += 8) {
      const float* al = a_pre + ((size_t)n * H + hh) * M;
      const float* mk = att_mask ? att_mask + ((size_t)n * H + hh) * M : nullptr;
      float dot = 0.f;
      for (int m = lane; m < M; m += 32) {
        float da = sm[hh * M + m];
        if (mk) da = (da / att_keep) * mk[m];
        sm[hh * M + m] = da;
        dot = fmaf(al[m], da, dot);
      }
      dot = wred_sum(dot);
      for (int m = lane; m < M; m += 32) {
        float a = al[m];
        float ds = a * (sm[hh * M + m] - dot);
        if (s_in) {
          // _signorm (src/model_base.py:599-603): alpha = g / sum g, g = sigmoid(s)  ->  ds = alpha (dalpha - <alpha, dalpha>) (1 - g)
          const float sv = s_in[((size_t)n * H + hh) * M + m];
          ds *= 1.0f - sigm(sv);
          dT_part += ds * sv;
        } else {
          dT_part += ds * logf(fmaxf(a, 1e-37f));       // = ds * s up to a per-row constant (sum ds = 0)
        }
        ds_out[((size_t)n * H + hh) * M + m] = ds;
      }
    }
    dT_part = wred_sum(dT_part);
    __syncthreads();
    if (lane == 0) red[warp] = dT_part;
    __syncthreads();
    if (tid == 0) {
      float s = 0.f;
      for (int w = 0; w < 8; ++w) s += red[w];
      if (temperature) dT_acc[n] += -s / temperature[0];   // MultiHeadDot has no temperature (common/ops_rnn.py:603-632)
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------
// Attention backward, part 2 (grid: image x position slice; 128 threads): LN-tanh
// recompute per (row, position) and the gradients of v, gamma, beta, the keys and
// the query.  Lane owns R/32 contiguous channels.  Per-(image, slice) partial sums
// of dv / dgamma / dbeta accumulate over time steps in `cpart` [B*S][3][R]
// (single owner -> deterministic); dq partials [S][N][R] are summed by
// sum_slices_kernel.
// ---------------------------------------------------------------------------
template <int R>
__global__ void __launch_bounds__(128)
attn_bwd_ln_kernel(const float* __restrict__ keys, const float* __restrict__ lq, int ld_lq, int q_off,
                   const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ vvec,
                   const float* __restrict__ temperature, const float* __restrict__ ds, float* __restrict__ dkeys,
                   float* __restrict__ dq_part, float* __restrict__ cpart, int k, int H, int M, int S, int N) {
  constexpr int CPL = R / 32;
  const int b = blockIdx.x, sl = blockIdx.y;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int c0 = lane * CPL;
  const int D = R / H;
  const int m_lo = (int)(((long long)M * sl) / S), m_hi = (int)(((long long)M * (sl + 1)) / S);
  const float invT = 1.0f / temperature[0];
  float gm[CPL], bt[CPL], vv[CPL];
  // 128-bit loads: as scalars these three rows were 3 * CPL requests of 32 sectors each per warp -- a per-CTA fixed cost
#pragma unroll
  for (int c4 = 0; c4 < CPL / 4; ++c4) {
    const float4 g4 = ldg4(gamma + c0 + c4 * 4), b4 = ldg4(beta + c0 + c4 * 4), v4 = ldg4(vvec + c0 + c4 * 4);
    gm[c4 * 4 + 0] = g4.x; gm[c4 * 4 + 1] = g4.y; gm[c4 * 4 + 2] = g4.z; gm[c4 * 4 + 3] = g4.w;
    bt[c4 * 4 + 0] = b4.x; bt[c4 * 4 + 1] = b4.y; bt[c4 * 4 + 2] = b4.z; bt[c4 * 4 + 3] = b4.w;
    vv[c4 * 4 + 0] = v4.x; vv[c4 * 4 + 1] = v4.y; vv[c4 * 4 + 2] = v4.z; vv[c4 * 4 + 3] = v4.w;
  }
  float dv_a[CPL], dg_a[CPL], db_a[CPL];
#pragma unroll
  for (int c = 0; c < CPL; ++c) { dv_a[c] = 0.f; dg_a[c] = 0.f; db_a[c] = 0.f; }
  __shared__ float red[4][R];
  // running sums of this (image, slice) over the time steps: fetched now, added to at the end (their three dependent
  // L2 round trips were part of every CTA's tail)
  float* cp = cpart + ((size_t)b * S + sl) * 3 * R;
  float cpv[3][R / 128];
#pragma unroll
  for (int which = 0; which < 3; ++which)
#pragma unroll
    for (int i = 0; i < R / 128; ++i) cpv[which][i] = cp[(size_t)which * R + threadIdx.x + 128 * i];
  for (int beam = 0; beam < k; ++beam) {
    const int n = b * k + beam;
    float q[CPL], dq_a[CPL];
    const float* qp = lq + (size_t)n * ld_lq + q_off + c0;
    if (((ld_lq | q_off) & 3) == 0) {
#pragma unroll
      for (int c4 = 0; c4 < CPL / 4; ++c4) {
        const float4 q4 = ldg4(qp + c4 * 4);
        q[c4 * 4 + 0] = q4.x; q[c4 * 4 + 1] = q4.y; q[c4 * 4 + 2] = q4.z; q[c4 * 4 + 3] = q4.w;
      }
    } else {
#pragma unroll
      for (int c = 0; c < CPL; ++c) q[c] = qp[c];
    }
#pragma unroll
    for (int c = 0; c < CPL; ++c) dq_a[c] = 0.f;
    const bool one_head = (D % CPL) == 0;          // a lane's CPL contiguous channels lie in one head
    for (int m = m_lo + warp; m < m_hi; m += 4) {
      const float* kr = keys + ((size_t)b * M + m) * R + c0;
      float* dkr = dkeys + ((size_t)b * M + m) * R + c0;
      float u[CPL];
      float s = 0.f;
      // the gradient row this position accumulates into is fetched WITH the key row: read at the end of the iteration
      // (where it is needed) its L2 round trip sat on the critical path of every position
      float4 dk[CPL / 4];
#pragma unroll
      for (int c4 = 0; c4 < CPL / 4; ++c4) dk[c4] = *reinterpret_cast<const float4*>(dkr + c4 * 4);
      // 128-bit accesses: a lane's slice is 4*CPL contiguous, 16-byte aligned bytes (scalar loads touched every
      // 32-byte sector of the row CPL times)
#pragma unroll
      for (int c4 = 0; c4 < CPL / 4; ++c4) {
        const float4 kv = ldg4(kr + c4 * 4);
        u[c4 * 4 + 0] = kv.x + q[c4 * 4 + 0]; u[c4 * 4 + 1] = kv.y + q[c4 * 4 + 1];
        u[c4 * 4 + 2] = kv.z + q[c4 * 4 + 2]; u[c4 * 4 + 3] = kv.w + q[c4 * 4 + 3];
      }
#pragma unroll
      for (int c = 0; c < CPL; ++c) s += u[c];
      const float mean = wred_sum(s) * (1.0f / R);
      float ss = 0.f;
#pragma unroll
      for (int c = 0; c < CPL; ++c) { u[c] -= mean; ss = fmaf(u[c], u[c], ss); }
      const float rstd = 1.0f / sqrtf(wred_sum(ss) * (1.0f / R) + 1e-12f);
      float du[CPL];
      float s1 = 0.f, s2 = 0.f;
      const float dz_lane = one_head ? ds[((size_t)n * H + c0 / D) * M + m] * invT : 0.f;
#pragma unroll
      for (int c = 0; c < CPL; ++c) {
        const float uh = u[c] * rstd;                      // normalised
        const float th = tanhf(fmaf(uh, gm[c], bt[c]));
        const float dz = one_head ? dz_lane : ds[((size_t)n * H + (c0 + c) / D) * M + m] * invT;
        dv_a[c] = fmaf(dz, th, dv_a[c]);
        const float dy = dz * vv[c] * (1.0f - th * th);
        dg_a[c] = fmaf(dy, uh, dg_a[c]);
        db_a[c] += dy;
        const float duh = dy * gm[c];
        du[c] = duh;
        u[c] = uh;
        s1 += duh;
        s2 = fmaf(duh, uh, s2);
      }
      s1 = wred_sum(s1) * (1.0f / R);
      s2 = wred_sum(s2) * (1.0f / R);
#pragma unroll
      for (int c4 = 0; c4 < CPL / 4; ++c4) {
        float4 acc = dk[c4];
        float g[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int c = c4 * 4 + j;
          g[j] = rstd * (du[c] - s1 - u[c] * s2);
          dq_a[c] += g[j];
        }
        acc.x += g[0]; acc.y += g[1]; acc.z += g[2]; acc.w += g[3];
        *reinterpret_cast<float4*>(dkr + c4 * 4) = acc;
      }
    }
    // dq partial of this (row, slice): fixed-order sum over the 4 warps
#pragma unroll
    for (int c = 0; c < CPL; ++c) red[warp][c0 + c] = dq_a[c];
    __syncthreads();
    for (int j = threadIdx.x; j < R; j += 128)
      dq_part[((size_t)sl * N + n) * R + j] = (red[0][j] + red[1][j]) + (red[2][j] + red[3][j]);
    __syncthreads();
  }
#pragma unroll
  for (int which = 0; which < 3; ++which) {
#pragma unroll
    for (int c = 0; c < CPL; ++c) red[warp][c0 + c] = which == 0 ? dv_a[c] : (which == 1 ? dg_a[c] : db_a[c]);
    __syncthreads();
#pragma unroll
    for (int i = 0; i < R / 128; ++i) {
      const int j = threadIdx.x + 128 * i;
      cp[(size_t)which * R + j] = cpv[which][i] + ((red[0][j] + red[1][j]) + (red[2][j] + red[3][j]));
    }
    __syncthreads();
  }
}

// MultiHeadDot backward (common/ops_rnn.py:603-632): s[n, h, m] = <k[b, m, h], q[n, h]> / sqrt(D).  Same grid, lane
// ownership and partial-sum layout as attn_bwd_ln_kernel (single owner per (image, position) -> deterministic).
template <int R>
__global__ void __launch_bounds__(128)
attn_bwd_dot_kernel(const float* __restrict__ keys, const float* __restrict__ lq, int ld_lq, int q_off,
                    const float* __restrict__ ds, float* __restrict__ dkeys, float* __restrict__ dq_part, int k, int H,
                    int M, int S, int N) {
  constexpr int CPL = R / 32;
  const int b = blockIdx.x, sl = blockIdx.y;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int c0 = lane * CPL;
  const int D = R / H;
  const int m_lo = (int)(((long long)M * sl) / S), m_hi = (int)(((long long)M * (sl + 1)) / S);
  const float inv = 1.0f / sqrtf((float)D);
  __shared__ float red[4][R];
  for (int beam = 0; beam < k; ++beam) {
    const int n = b * k + beam;
    float q[CPL], dq_a[CPL];
    const float* qp = lq + (size_t)n * ld_lq + q_off + c0;
#pragma unroll
    for (int c = 0; c < CPL; ++c) { q[c] = qp[c]; dq_a[c] = 0.f; }
    for (int m = m_lo + warp; m < m_hi; m += 4) {
      const float* kr = keys + ((size_t)b * M + m) * R + c0;
      float* dkr = dkeys + ((size_t)b * M + m) * R + c0;
#pragma unroll
      for (int c4 = 0; c4 < CPL / 4; ++c4) {
        const float4 kv = ldg4(kr + c4 * 4);
        float4 acc = *reinterpret_cast<const float4*>(dkr + c4 * 4);
        const float kk[4] = {kv.x, kv.y, kv.z, kv.w};
        float g[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int c = c4 * 4 + j;
          const float dz = ds[((size_t)n * H + (c0 + c) / D) * M + m] * inv;
          dq_a[c] = fmaf(dz, kk[j], dq_a[c]);
          g[j] = dz * q[c];
        }
        acc.x += g[0]; acc.y += g[1]; acc.z += g[2]; acc.w += g[3];
        *reinterpret_cast<float4*>(dkr + c4 * 4) = acc;
      }
    }
#pragma unroll
    for (int c = 0; c < CPL; ++c) red[warp][c0 + c] = dq_a[c];
    __syncthreads();
    for (int j = threadIdx.x; j < R; j += 128)
      dq_part[((size_t)sl * N + n) * R + j] = (red[0][j] + red[1][j]) + (red[2][j] + red[3][j]);
    __syncthreads();
  }
}

// dst[b, :] = (t >= lens[b]) ? 0 : src[b, :]   (imputed rows do not reach the context layer)
__global__ void mask_fin_copy_kernel(const float* __restrict__ src, const int* __restrict__ lens, int t,
                                     float* __restrict__ dst, int B, int A) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)B * A) return;
  const int b = (int)(i / A);
  dst[i] = (lens && t >= lens[b]) ? 0.f : src[i];
}

// dlq[n, q_off + j] = sum_s dq_part[s][n][j]
__global__ void sum_slices_kernel(const float* __restrict__ part, int S, int N, int R, float* __restrict__ dlq,
                                  int ld, int q_off) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N * R) return;
  int n = i / R, j = i - n * R;
  float s = 0.f;
  for (int sl = 0; sl < S; ++sl) s += part[((size_t)sl * N + n) * R + j];
  dlq[(size_t)n * ld + q_off + j] = s;
}

// ---------------------------------------------------------------------------
// LSTM pointwise backward (BasicLSTMCell, gate order i, j, f, o, forget_bias 1).
//   dh_cell = dHout * out_mask / keep + (fin ? 0 : gH);  dc_cell = (fin ? 0 : gC) + ...
//   writes dgates [B, 4R]; gC <- dc_prev(cell) + (fin ? gC : 0); gH_pass = fin ? gH : 0.
// ---------------------------------------------------------------------------
__global__ void lstm_bwd_kernel(const float* __restrict__ gates, const float* __restrict__ c_prev,
                                const float* __restrict__ dhout, const float* __restrict__ out_mask, float out_keep,
                                const int* __restrict__ lens, int t, float* __restrict__ gH, float* __restrict__ gC,
                                float* __restrict__ gH_pass, float* __restrict__ dgates, int B, int R, int nz = 1,
                                size_t zstride = 0) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * R) return;
  int b = i / R, j = i - b * R;
  const bool fin = lens && t >= lens[b];
  const float* g = gates + (size_t)b * 4 * R;
  const float gi = g[j], gj = g[R + j], gf = g[2 * R + j], go = g[3 * R + j];
  const float cp = c_prev ? c_prev[i] : 0.f;
  const float si = sigm(gi), tj = tanhf(gj), sf = sigm(gf + 1.0f), so = sigm(go);
  const float cn = cp * sf + si * tj;
  const float tc = tanhf(cn);
  float dh = dhout ? dhout[i] : 0.f;
  for (int z = 1; z < nz; ++z) dh += dhout[z * zstride + i];      // split-K partials of the producing GEMM, fixed order
  if (out_mask) dh = (dh / out_keep) * out_mask[i];
  const float gh = gH[i], gc = gC[i];
  if (!fin) dh += gh;
  float dc = (fin ? 0.f : gc) + dh * so * (1.0f - tc * tc);
  float* dg = dgates + (size_t)b * 4 * R;
  dg[j] = dc * tj * si * (1.0f - si);
  dg[R + j] = dc * si * (1.0f - tj * tj);
  dg[2 * R + j] = dc * cp * sf * (1.0f - sf);
  dg[3 * R + j] = dh * tc * so * (1.0f - so);
  gC[i] = dc * sf + (fin ? gc : 0.f);
  gH_pass[i] = fin ? gh : 0.f;
}

// GRU cell backward (TF r1.9 GRUCell; tape row [r | u | r*h | c], gradient row dG = [dR | dU | dC | dh'] of the r / u / candidate
// pre-activations, the last quarter a scratch copy of dh').
// Part a: dh' = dHout (split-K partials, output dropout) + (fin ? 0 : gH);  dC = dh' (1 - u)(1 - c^2).
__global__ void gru_bwd_a_kernel(const float* __restrict__ tape, const float* __restrict__ dhout, const float* __restrict__ out_mask,
                                 float out_keep, const int* __restrict__ lens, int t, const float* __restrict__ gH,
                                 float* __restrict__ dgates, int B, int R, int nz = 1, size_t zstride = 0) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * R) return;
  int b = i / R, j = i - b * R;
  const bool fin = lens && t >= lens[b];
  float dh = dhout ? dhout[i] : 0.f;
  for (int z = 1; z < nz; ++z) dh += dhout[z * zstride + i];      // split-K partials of the producing GEMM, fixed order
  if (out_mask) dh = (dh / out_keep) * out_mask[i];
  if (!fin) dh += gH[i];
  const float* tr = tape + (size_t)b * 4 * R;
  const float u = tr[R + j], c = tr[3 * R + j];
  float* dg = dgates + (size_t)b * 4 * R;
  dg[2 * R + j] = dh * (1.0f - u) * (1.0f - c * c);
  dg[3 * R + j] = dh;
}

// Part b, after d(r*h) = dC . candidate/kernel[h rows]^T (split-K partials drh; NULL = zero, the init step):
//   dR = d(rh) h r (1 - r),  dU = dh' (h - c) u (1 - u);
//   gH_pass = dh' u + d(rh) r + (fin ? gH : 0): what reaches h_prev outside the [x, h] . gates/kernel product (dx_split adds
//   that product's share).  h_prev: the state the step read (NULL = zero).
__global__ void gru_bwd_b_kernel(const float* __restrict__ tape, const float* __restrict__ h_prev, const float* __restrict__ drh, int nz,
                                 size_t zstride, const int* __restrict__ lens, int t, const float* __restrict__ gH,
                                 float* __restrict__ gH_pass, float* __restrict__ dgates, int B, int R) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * R) return;
  int b = i / R, j = i - b * R;
  const bool fin = lens && t >= lens[b];
  const float* tr = tape + (size_t)b * 4 * R;
  const float r = tr[j], u = tr[R + j], c = tr[3 * R + j];
  const float hp = h_prev ? h_prev[i] : 0.f;
  float d = 0.f;
  if (drh) {
    d = drh[i];
    for (int z = 1; z < nz; ++z) d += drh[z * zstride + i];
  }
  float* dg = dgates + (size_t)b * 4 * R;
  const float dh = dg[3 * R + j];
  dg[j] = d * hp * r * (1.0f - r);
  dg[R + j] = dh * (hp - c) * u * (1.0f - u);
  gH_pass[i] = dh * u + d * r + (fin ? gH[i] : 0.f);
}

// dxh [B, KX] -> demb [B, W], gCtx [B, A], gH [B, R] (input dropout backward + pass-through of finished rows)
__global__ void dx_split_kernel(const float* __restrict__ dxh, int KX, int W, int A, int R,
                                const float* __restrict__ in_mask, float in_keep, const int* __restrict__ lens, int t,
                                float* __restrict__ demb, float* __restrict__ gCtx, float* __restrict__ gH,
                                const float* __restrict__ gH_pass, int B, int nz = 1, size_t zstride = 0) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)B * KX) return;
  int b = (int)(i / KX), j = (int)(i % KX);
  float v = dxh[i];
  for (int z = 1; z < nz; ++z) v += dxh[z * zstride + i];         // split-K partials of the producing GEMM, fixed order
  const bool fin = lens && t >= lens[b];
  if (j < W + A) {
    if (in_mask) v = (v / in_keep) * in_mask[(size_t)b * (W + A) + j];
    if (j < W) {
      if (demb) demb[(size_t)b * W + j] = v;
    } else if (gCtx) {
      size_t o = (size_t)b * A + (j - W);
      gCtx[o] = v + (fin ? gCtx[o] : 0.f);
    }
  } else if (gH) {
    size_t o = (size_t)b * R + (j - W - A);
    gH[o] = v + gH_pass[o];
  }
}

// XH rows for the batched kernel gradient: block 0 = [x0 ; 0], block 1+t = [x_t ; h_{t-1}].
__global__ void build_xh_kernel(const float* __restrict__ xd, const float* __restrict__ hst, int XA, int R,
                                float* __restrict__ xh, size_t rows, int B) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int KX = XA + R;
  if (i >= rows * KX) return;
  size_t r = i / KX;
  int j = (int)(i % KX);
  float v;
  if (j < XA) v = xd[r * XA + j];
  else v = (r < (size_t)B) ? 0.f : hst[(r - B) * R + (j - XA)];   // state after step t-1 = h[t] slot (0 = init)
  xh[i] = v;
}

// GRU candidate-kernel rows: block 0 = [x0 ; 0], block 1+t = [x_t ; r_t * h_{t-1}] (r*h from the tape, zero at the init step).
__global__ void build_xrh_kernel(const float* __restrict__ xd, const float* __restrict__ tape, int XA, int R,
                                 float* __restrict__ xh, size_t rows) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int KX = XA + R;
  if (i >= rows * KX) return;
  size_t r = i / KX;
  int j = (int)(i % KX);
  xh[i] = (j < XA) ? xd[r * XA + j] : tape[r * 4 * R + 2 * R + (j - XA)];
}

// Deterministic embedding gradient: dE[id, :] = sum over rows with ids[row] == id.
__global__ void embed_grad_kernel(const int* __restrict__ ids, const float* __restrict__ demb, int rows, int W, int V,
                                  float* __restrict__ dE) {
  int id = blockIdx.x;
  for (int j = threadIdx.x; j < W; j += blockDim.x) {
    float s = 0.f;
    for (int r = 0; r < rows; ++r)
      if (ids[r] == id) s += demb[(size_t)r * W + j];
    dE[(size_t)id * W + j] = s;
  }
  (void)V;
}

__global__ void scalar_sum_kernel(const float* __restrict__ src, int n, float scale, float* __restrict__ out) {
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    float s = 0.f;
    for (int i = 0; i < n; ++i) s += src[i];
    *out = s * scale;
  }
}

// l2: grads += decay * theta ; reg = decay/2 * sum theta^2   (fixed-order two-level sum)
__global__ void l2_kernel(const float* __restrict__ theta, float* __restrict__ grads, size_t n, float decay,
                          float* __restrict__ partial) {
  __shared__ float red[8];
  size_t per = (n + gridDim.x - 1) / gridDim.x;
  size_t lo = (size_t)blockIdx.x * per, hi = lo + per < n ? lo + per : n;
  float s = 0.f;
  for (size_t i = lo + threadIdx.x; i < hi; i += blockDim.x) {
    float th = theta[i];
    s = fmaf(th, th, s);
    if (grads) grads[i] += decay * th;
  }
  s = wred_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tot = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += red[w];
    partial[blockIdx.x] = tot;
  }
}

// tf.train.AdamOptimizer dense update: lr_t = lr sqrt(1-b2^t)/(1-b1^t); theta -= lr_t m / (sqrt(v) + eps).
__global__ void adam_kernel(float* __restrict__ theta, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, size_t n, float lr_t, float beta1, float beta2, float eps,
                            float grad_scale) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float gi = g[i] * grad_scale;
  float mi = m[i] + (gi - m[i]) * (1.0f - beta1);
  float vi = v[i] + (gi * gi - v[i]) * (1.0f - beta2);
  m[i] = mi;
  v[i] = vi;
  theta[i] -= lr_t * mi / (sqrtf(vi) + eps);
}

// tf.train.MomentumOptimizer(use_nesterov=False) dense update (src/model_base.py:868-880): accum = momentum * accum + g;
// theta -= lr * accum.
__global__ void momentum_kernel(float* __restrict__ theta, const float* __restrict__ g, float* __restrict__ accum, size_t n,
                                float lr, float momentum, float grad_scale) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float a = momentum * accum[i] + g[i] * grad_scale;
  accum[i] = a;
  theta[i] -= lr * a;
}

// slim.learning.clip_gradient_norms (create_train_op(clip_gradient_norm=c), src/model_base.py:394-401): every variable's
// gradient is clipped by ITS OWN l2 norm, g <- g * c / max(|g|, c).  One CTA per variable, fixed-order block reduction.
__global__ void __launch_bounds__(1024)
clip_by_norm_kernel(float* __restrict__ grads, const long long* __restrict__ offsets, const long long* __restrict__ sizes,
                    float max_norm) {
  __shared__ float red[32];
  __shared__ float s_scale;
  float* g = grads + offsets[blockIdx.x];
  const long long n = sizes[blockIdx.x];
  float s = 0.f;
  for (long long i = threadIdx.x; i < n; i += blockDim.x) s = fmaf(g[i], g[i], s);
  s = wred_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tot = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += red[w];
    const float nrm = sqrtf(tot);
    s_scale = nrm > max_norm ? max_norm / nrm : 1.0f;
  }
  __syncthreads();
  const float sc = s_scale;
  if (sc != 1.0f)
    for (long long i = threadIdx.x; i < n; i += blockDim.x) g[i] *= sc;
}

// Legacy image-embedding head (src/model_base.py:80-91), recomputed for its backward: one CTA per image.
//   pool = mean over the 49 positions of Mixed_5c; xhat = (pool - mean) / sqrt(var + 1e-12); t1 = tanh(xhat * gamma + beta)
__global__ void __launch_bounds__(256)
legacy_head_recompute_kernel(const float* __restrict__ m5c, const float* __restrict__ gamma, const float* __restrict__ beta,
                             float* __restrict__ xhat, float* __restrict__ t1, int P, int C) {
  __shared__ float red[8];
  __shared__ float s_stat[2];
  const int b = blockIdx.x, tid = threadIdx.x;
  const float* src = m5c + (size_t)b * P * C;
  float pool[4] = {0.f, 0.f, 0.f, 0.f};                       // C = 1024 = 4 channels per thread
  for (int j = 0; j < 4; ++j) {
    const int c = tid + 256 * j;
    float s = 0.f;
    if (c < C)
      for (int p2 = 0; p2 < P; ++p2) s += src[(size_t)p2 * C + c];
    pool[j] = s * (1.0f / (float)P);
  }
  float s = (pool[0] + pool[1]) + (pool[2] + pool[3]);
  s = wred_sum(s);
  if ((tid & 31) == 0) red[tid >> 5] = s;
  __syncthreads();
  if (tid == 0) { float t = 0.f; for (int w = 0; w < 8; ++w) t += red[w]; s_stat[0] = t / (float)C; }
  __syncthreads();
  const float mean = s_stat[0];
  float v = 0.f;
  for (int j = 0; j < 4; ++j) { const float d = (tid + 256 * j < C) ? pool[j] - mean : 0.f; v = fmaf(d, d, v); }
  v = wred_sum(v);
  if ((tid & 31) == 0) red[tid >> 5] = v;
  __syncthreads();
  if (tid == 0) { float t = 0.f; for (int w = 0; w < 8; ++w) t += red[w]; s_stat[1] = 1.0f / sqrtf(t / (float)C + 1e-12f); }
  __syncthreads();
  const float rstd = s_stat[1];
  for (int j = 0; j < 4; ++j) {
    const int c = tid + 256 * j;
    if (c < C) {
      const float xh = (pool[j] - mean) * rstd;
      xhat[(size_t)b * C + c] = xh;
      t1[(size_t)b * C + c] = tanhf(fmaf(xh, gamma[c], beta[c]));
    }
  }
}

// d_ln = d_t1 * (1 - t1^2) (-> d beta rows) and gx = d_ln * xhat (-> d gamma rows), in place of d_t1 / xhat
__global__ void legacy_head_dln_kernel(float* __restrict__ d_t1, float* __restrict__ xhat, const float* __restrict__ t1, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float t = t1[i];
  const float d = d_t1[i] * (1.0f - t * t);
  d_t1[i] = d;
  xhat[i] = d * xhat[i];
}

// ---------------------------------------------------------------------------
// Host side.
// ---------------------------------------------------------------------------
// nz_out != nullptr: when the plan splits K, the partial sums stay in `part` ([nz][M][N]) for a consumer that adds them
// itself (in the same fixed order) and *nz_out = nz; otherwise *nz_out = 1 and C holds the product.
static int train_gemm(comic_handle_t h, const float* A, int lda, const float* Bm, int ldb, float* C, int ldc, int M,
                      int N, int K, float* part, size_t part_floats, cudaStream_t st, int* nz_out = nullptr) {
  APlain a{};
  a.nseg = 1;
  a.seg[0] = ASeg{A, nullptr, lda, K, M};
  GemmPlan p = plan_gemm(M, N, K, h->num_sms, true);
  int nz = gemm_num_partials(K, p);
  if (nz > 1 && (size_t)nz * M * N > part_floats) { p.splitk = 1; nz = 1; }
  Epi e{};
  e.nroute = 1;
  e.stop_n = 0x7fffffff;
  const bool vec = (K % 4 == 0) && (lda % 4 == 0);
  if (nz_out) *nz_out = 1;
  if (nz == 1) {
    e.r[0] = Route{0, N, C, ldc, 0};
    if (vec) COMIC_CHECK_CUDA((launch_gemm<0, 4>(a, Bm, ldb, M, N, K, e, p, st)));
    else COMIC_CHECK_CUDA((launch_gemm<0, 1>(a, Bm, ldb, M, N, K, e, p, st)));
    h->launches++;
    return COMIC_OK;
  }
  e.r[0] = Route{0, N, part, N, 0};
  e.split_stride = (long long)M * N;
  if (vec) COMIC_CHECK_CUDA((launch_gemm<0, 4>(a, Bm, ldb, M, N, K, e, p, st)));
  else COMIC_CHECK_CUDA((launch_gemm<0, 1>(a, Bm, ldb, M, N, K, e, p, st)));
  if (nz_out && ldc == N) {
    *nz_out = nz;
    h->launches++;
    COMIC_CHECK_CUDA(cudaGetLastError());
    return COMIC_OK;
  }
  // fixed-order reduction of the partials into C (ldc may differ from N)
  {
    size_t tot = (size_t)M * N;
    splitk_reduce2d_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(part, nz, (size_t)M * N, C, ldc, M, N);
  }
  h->launches += 2;
  COMIC_CHECK_CUDA(cudaGetLastError());
  return COMIC_OK;
}

static void transpose(const float* src, int rows, int cols, int ld_src, float* dst, int ld_dst, cudaStream_t st) {
  dim3 g((cols + 31) / 32, (rows + 31) / 32), blk(32, 8);
  transpose_kernel<<<g, blk, 0, st>>>(src, rows, cols, ld_src, dst, ld_dst);
}

struct TrainBufs {
  StepBufs sb;
  // tape
  float *xd, *gates, *c, *h, *ctx, *hdrop, *lq, *apre, *apost;
  // backward
  float *dlq, *dG, *demb, *gH, *gC, *gCtx, *gHp, *dHout, *dxh, *ds, *dqpart, *cpart, *dTacc, *maprows, *rowloss;
  float *dkeys, *dvals, *keys, *vals, *dx0;
  float *KT, *KcT, *outqT, *xh, *xhT, *hdT, *fmT, *embT, *dOutQ, *part, *scal;
  float *encT, *dfm_tmp;   // cnn_finetune: transposed W_k / W_v / W_I, second dfm term (independent)
  // variants: raw scores per step (signorm), context-layer input / masked output gradient per step, a_layer^T
  float *stape, *ctxraw, *gctx_tape, *dctxraw, *aT, *ctxrawT;
  size_t part_floats;
  int S, rows_pad;
};

static int attn_slices(int B, int num_sms) {
  // (image x position-slice) CTAs of the attention backward.  attn_bwd_ln_kernel<512> holds 212 registers x 128 threads:
  // two CTAs per SM, and its time is mostly a per-CTA fixed cost (28 slices: 3 waves = 64 us per launch against 51 us for
  // 10 slices, ncu launch lists profiles/r12t / r12u) -- so the grid is sized to ONE wave of 2 x SMs CTAs, rounded DOWN
  // (batch 32: 10 slices = 320 CTAs were 296 + a second wave of 24)
  int S = (2 * num_sms) / B;
  if (S < 1) S = 1;
  if (S > 28) S = 28;
  return S;
}

static void carve_train(comic_handle_t h, Carver& cv, int B, int T_run, TrainBufs& tb) {
  const int R = h->R, XA = h->W + h->A, A = h->A, LQ = h->LQ, HM = h->H * h->M, KX = h->KX;
  const size_t T1 = (size_t)T_run + 1;
  carve_step(h, cv, B, tb.sb, false);
  tb.xd = cv.take<float>(T1 * B * XA);
  tb.gates = cv.take<float>(T1 * B * 4 * R);
  tb.c = cv.take<float>(T1 * B * R);
  tb.h = cv.take<float>(T1 * B * R);
  tb.ctx = cv.take<float>(T1 * B * A);
  tb.hdrop = cv.take<float>((size_t)T_run * B * R + 4 * R);
  tb.lq = cv.take<float>((size_t)T_run * B * LQ);
  tb.apre = cv.take<float>((size_t)T_run * B * HM);
  tb.apost = cv.take<float>((size_t)T_run * B * HM);
  tb.rows_pad = (int)((T1 * B + 3) / 4 * 4);
  tb.dlq = cv.take<float>((size_t)tb.rows_pad * LQ);
  tb.dG = cv.take<float>((size_t)tb.rows_pad * 4 * R);
  tb.demb = cv.take<float>((size_t)T_run * B * h->W);
  tb.gH = cv.take<float>((size_t)B * R);
  tb.gC = cv.take<float>((size_t)B * R);
  tb.gCtx = cv.take<float>((size_t)B * A);
  tb.gHp = cv.take<float>((size_t)B * R);
  tb.dHout = cv.take<float>((size_t)B * R);
  tb.dxh = cv.take<float>((size_t)B * KX);
  tb.ds = cv.take<float>((size_t)B * HM);
  tb.S = attn_slices(B, h->num_sms);
  tb.dqpart = cv.take<float>((size_t)tb.S * B * R);
  tb.cpart = cv.take<float>((size_t)B * tb.S * 3 * R);
  tb.dTacc = cv.take<float>(B);
  tb.maprows = cv.take<float>((size_t)T_run * B);
  tb.rowloss = cv.take<float>((size_t)T_run * B);
  tb.dkeys = cv.take<float>((size_t)B * h->M * R);
  tb.dvals = cv.take<float>(h->cfg.fm_projection == 1 ? 1 : (size_t)B * h->M * h->VAL);
  tb.keys = cv.take<float>((size_t)B * h->M * R);
  tb.vals = cv.take<float>(h->cfg.fm_projection == 2 ? (size_t)B * h->M * R : 1);
  tb.dx0 = cv.take<float>((size_t)((B + 3) / 4 * 4) * XA);
  tb.KT = cv.take<float>((size_t)4 * R * KX);                 // GRU: [3R, KX] transpose of the gate panel
  tb.KcT = (h->cell == COMIC_CELL_GRU) ? cv.take<float>((size_t)R * R) : nullptr;
  tb.outqT = cv.take<float>((size_t)LQ * R);
  tb.xh = cv.take<float>((size_t)tb.rows_pad * KX);
  tb.xhT = cv.take<float>((size_t)KX * tb.rows_pad);
  tb.hdT = cv.take<float>((size_t)R * tb.rows_pad);
  int bm = (B * h->M + 3) / 4 * 4;
  tb.fmT = cv.take<float>((size_t)h->C * bm);
  tb.embT = cv.take<float>((size_t)h->E * ((B + 3) / 4 * 4));
  tb.dOutQ = cv.take<float>((size_t)R * LQ);
  tb.part_floats = (size_t)16 * B * (KX > 4 * R ? KX : 4 * R) + (size_t)4 * 1024 * 1024;
  tb.part = cv.take<float>(tb.part_floats);
  tb.scal = cv.take<float>(1024);
  {
    size_t a = (size_t)h->R * h->C, b = (size_t)(h->W + h->A) * h->E;
    tb.encT = cv.take<float>(a > b ? a : b);
    tb.dfm_tmp = cv.take<float>(h->cfg.fm_projection == 2 ? (size_t)B * h->M * h->C : 1);
  }
  tb.stape = cv.take<float>(h->cfg.prob_fn == 1 ? (size_t)T_run * B * HM : 1);
  const bool cl = h->cfg.context_layer != 0;
  tb.ctxraw = cv.take<float>(cl ? (size_t)T_run * B * h->VAL : 1);
  tb.gctx_tape = cv.take<float>(cl ? (size_t)tb.rows_pad * A : 1);
  tb.dctxraw = cv.take<float>(cl ? (size_t)B * h->VAL : 1);
  tb.aT = cv.take<float>(cl ? (size_t)A * h->VAL : 1);
  tb.ctxrawT = cv.take<float>(cl ? (size_t)h->VAL * tb.rows_pad : 1);
}

int train_workspace_bytes(comic_handle_t h, int B, int T_run, size_t* bytes) {
  Carver cv(nullptr);
  TrainBufs tb;
  carve_train(h, cv, B, T_run, tb);
  *bytes = cv.off + 256;
  return COMIC_OK;
}

}  // namespace comic

using namespace comic;

extern "C" int comic_train_workspace_bytes(comic_handle_t h, int B, int T_run, size_t* bytes) {
  COMIC_REQUIRE(h && bytes && B > 0 && T_run >= 0, COMIC_E_BADARG, "train_workspace_bytes: bad argument");
  h->sized = true;
  return train_workspace_bytes(h, B, T_run, bytes);
}

extern "C" int comic_dropout_masks(comic_handle_t h, float* out, size_t n, float keep, uint64_t seed, uint64_t stream_id,
                                   void* stream) {
  COMIC_REQUIRE(h && out, COMIC_E_BADARG, "dropout_masks: null argument");
  if (n == 0) return COMIC_OK;
  size_t n4 = (n + 3) / 4;
  dropout_mask_kernel<<<(unsigned)((n4 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(out, n, keep, seed, stream_id);
  h->launches++;
  COMIC_CHECK_CUDA(cudaGetLastError());
  return COMIC_OK;
}

extern "C" int comic_train_fwd_bwd(comic_handle_t h, const float* fm, const float* im_embed, int B,
                                   const int32_t* inputs_tm, const int32_t* targets_tm, const float* coef_tm,
                                   const int32_t* lens, int T, int T_run, const comic_train_masks_t* masks,
                                   float map_loss_scale, float* loss_out, float* logits_out, float* attn_out,
                                   const comic_decoder_grads_t* grads, void* ws, size_t ws_bytes, void* stream) {
  COMIC_REQUIRE(h && h->bound, COMIC_E_BADARG, "train_fwd_bwd: weights not bound");
  COMIC_REQUIRE(h->cell == COMIC_CELL_LSTM || !grads || (grads->cand_kernel && grads->cand_bias), COMIC_E_BADARG,
                "train_fwd_bwd: GRU cell needs the candidate/{kernel, bias} gradient buffers");
  COMIC_REQUIRE(fm && im_embed && inputs_tm && targets_tm && coef_tm && lens && loss_out, COMIC_E_BADARG,
                "train_fwd_bwd: null argument");   // grads == NULL: forward only (evaluation perplexity)
  COMIC_REQUIRE(B > 0 && T > 0 && T_run > 0 && T_run <= T, COMIC_E_SHAPE, "train_fwd_bwd: bad B=%d T=%d T_run=%d", B, T, T_run);
  COMIC_REQUIRE(!h->cfg.context_layer || (h->w.a_layer && (!grads || grads->a_layer)), COMIC_E_BADARG,
                "train_fwd_bwd: attn_context_layer needs a_layer/kernel and its gradient buffer");
  COMIC_REQUIRE(h->R == 512 || h->R == 256 || h->R == 1024, COMIC_E_UNSUPPORTED, "train_fwd_bwd: rnn_size %d", h->R);
  cudaStream_t st = (cudaStream_t)stream;
  size_t need;
  train_workspace_bytes(h, B, T_run, &need);
  COMIC_REQUIRE(ws && ws_bytes >= need, COMIC_E_WORKSPACE, "train_fwd_bwd: workspace %zu < %zu", ws_bytes, need);
  const int R = h->R, W = h->W, A = h->A, XA = W + A, LQ = h->LQ, KX = h->KX, V = h->V, HM = h->H * h->M;
  const int M = h->M, C = h->C, E = h->E, VAL = h->VAL;
  Carver cv(ws);
  TrainBufs tb;
  carve_train(h, cv, B, T_run, tb);
  const comic_train_masks_t mk = masks ? *masks : comic_train_masks_t{};
  const float in_keep = masks ? mk.in_keep : 1.f, out_keep = masks ? mk.out_keep : 1.f, att_keep = masks ? mk.att_keep : 1.f;
  const size_t T1 = (size_t)T_run + 1;
  const bool gru = h->cell == COMIC_CELL_GRU;   // tape row [r | u | r*h | c] in place of the LSTM's 4R gate pre-activations
  int rc;
  if (gru) COMIC_CHECK_CUDA(cudaMemsetAsync(tb.c, 0, T1 * B * R * sizeof(float), st));   // no c state: the imputation copies zeros

  // ---- keys / values: D0 (ops_rnn.py:441-477) ----
  float* keys_buf = tb.keys;
  float* vals_buf = (h->cfg.fm_projection == 2) ? tb.vals : nullptr;
  if ((rc = comic_project_fm(h, fm, B, keys_buf, vals_buf, stream))) return rc;
  const float* values = h->cfg.fm_projection == 1 ? keys_buf : (h->cfg.fm_projection == 2 ? vals_buf : fm);

  // ---- init state, tape slot 0 ----
  if (h->cfg.init_method == 1) {
    // project_hidden (model_base.py:658-667): h0 = im_embed . W, c0 = 0; there is no init LSTM step, so slot 0 of the
    // x / gate tapes stays zero (its rows then add nothing to the batched kernel gradient)
    APlain a{};
    a.nseg = 1;
    a.seg[0] = ASeg{im_embed, nullptr, E, E, B};
    Epi e{};
    e.nroute = 1;
    e.stop_n = 0x7fffffff;
    e.r[0] = Route{0, R, tb.h, R, 0};
    GemmPlan p = plan_gemm(B, R, E, h->num_sms, false);
    COMIC_CHECK_CUDA((launch_gemm<0, 4>(a, h->w.init_weight, R, B, R, E, e, p, st)));
    COMIC_CHECK_CUDA(cudaMemsetAsync(tb.c, 0, (size_t)B * R * sizeof(float), st));
    COMIC_CHECK_CUDA(cudaMemsetAsync(tb.xd, 0, (size_t)B * XA * sizeof(float), st));
    COMIC_CHECK_CUDA(cudaMemsetAsync(tb.gates, 0, (size_t)B * 4 * R * sizeof(float), st));
    COMIC_CHECK_CUDA(cudaMemsetAsync(tb.ctx, 0, (size_t)B * A * sizeof(float), st));
    h->launches += 1;
  } else {
    // first_input (model_base.py:675-686)
    APlain a{};
    a.nseg = 1;
    a.seg[0] = ASeg{im_embed, nullptr, E, E, B};
    Epi e{};
    e.nroute = 1;
    e.stop_n = 0x7fffffff;
    e.r[0] = Route{0, XA, tb.xd, XA, 0};
    GemmPlan p = plan_gemm(B, XA, E, h->num_sms, false);
    COMIC_CHECK_CUDA((launch_gemm<0, 4>(a, h->w.init_weight, XA, B, XA, E, e, p, st)));
    if (mk.init_in) {
      size_t nx = (size_t)B * XA;
      mask_scale_kernel<<<(unsigned)((nx + 255) / 256), 256, 0, st>>>(tb.xd, mk.init_in, in_keep, nx);
    }
    if (gru) {
      if ((rc = gru_init_step(h, tb.xd, B, tb.part, tb.sb.gru, tb.h, tb.gates, st))) return rc;
    } else {
      APlain a2{};
      a2.nseg = 1;
      a2.seg[0] = ASeg{tb.xd, nullptr, XA, XA, B};
      GemmPlan p2 = plan_gemm(B, 4 * R, XA, h->num_sms, true);
      int nz = gemm_num_partials(XA, p2);
      Epi e2{};
      e2.nroute = 1;
      e2.stop_n = 0x7fffffff;
      e2.r[0] = Route{0, 4 * R, tb.sb.gates, 4 * R, 0};
      e2.split_stride = (long long)B * 4 * R;
      COMIC_CHECK_CUDA((launch_gemm<0, 4>(a2, h->w.lstm_kernel, 4 * R, B, 4 * R, XA, e2, p2, st)));
      int tot = B * R;
      lstm_init_fwd_kernel<<<(tot + 255) / 256, 256, 0, st>>>(tb.sb.gates, nz, (size_t)B * 4 * R, h->w.lstm_bias, tb.gates,
                                                            tb.c, tb.h, B, R);
      h->launches += 2;
    }
    COMIC_CHECK_CUDA(cudaMemsetAsync(tb.ctx, 0, (size_t)B * A * sizeof(float), st));
    h->launches += 2;
  }

  // ---- forward over T_run steps ----
  for (int t = 0; t < T_run; ++t) {
    StepIO io{};
    io.keys = keys_buf; io.values = values;
    io.tok = inputs_tm + (size_t)t * B; io.src = nullptr; io.src_limit = B;
    io.c_prev = tb.c + (size_t)t * B * R; io.h_prev = tb.h + (size_t)t * B * R; io.ctx_prev = tb.ctx + (size_t)t * B * A;
    io.c_new = tb.c + (size_t)(t + 1) * B * R; io.h_new = tb.h + (size_t)(t + 1) * B * R;
    io.ctx_new = tb.ctx + (size_t)(t + 1) * B * A;
    io.h_drop = tb.hdrop + (size_t)t * B * R;
    io.hist_t = tb.apost + (size_t)t * B * HM;
    io.alpha_pre = tb.apre + (size_t)t * B * HM;
    io.gates_save = tb.gates + (size_t)(t + 1) * B * 4 * R;
    io.force_dense = 1;
    io.in_mask = mk.inp ? mk.inp + (size_t)t * B * XA : nullptr;
    io.out_mask = mk.out ? mk.out + (size_t)t * B * R : nullptr;
    io.att_mask = mk.att ? mk.att + (size_t)t * B * HM : nullptr;
    io.in_keep = in_keep; io.out_keep = out_keep; io.att_keep = att_keep;
    io.fin_count = nullptr; io.t = t; io.n_rows = B;
    StepBufs sb = tb.sb;
    sb.xdense = tb.xd + (size_t)(t + 1) * B * XA;
    sb.lq = tb.lq + (size_t)t * B * LQ;
    if (h->cfg.prob_fn == 1) {   // signorm: its backward needs the raw scores -> sliced kernels, scores kept per step
      io.no_fused = 1;
      sb.scores = tb.stape + (size_t)t * B * HM;
    }
    if (h->cfg.context_layer) sb.ctxraw = tb.ctxraw + (size_t)t * B * VAL;
    if ((rc = run_step(h, io, sb, B, 1, st))) return rc;
    impute_state_kernel<<<B, 128, 0, st>>>(lens, t, B, R, A, io.c_prev, io.h_prev, io.ctx_prev, io.c_new, io.h_new,
                                          io.ctx_new);
    h->launches++;
  }

  // ---- loss + dlogits ----
  COMIC_CHECK_CUDA(cudaMemsetAsync(tb.dlq, 0, (size_t)tb.rows_pad * LQ * sizeof(float), st));
  xent_kernel<<<T_run * B, 256, 0, st>>>(tb.lq, LQ, V, targets_tm, coef_tm, lens, B, T_run, T, tb.dlq, tb.rowloss,
                                        logits_out);
  h->launches++;
  if (grads == nullptr) {
    // forward only (train_fn._run_eval_loop, src/train_fn.py:320-338): cross-entropy, no gradient, no map loss
    const int rows_fwd = T_run * B;
    scalar_sum_kernel<<<1, 32, 0, st>>>(tb.rowloss, rows_fwd, 1.0f, loss_out + 1);
    h->launches++;
    if (attn_out) {
      dim3 g(T_run, B);
      attn_maps_kernel<<<g, 256, 0, st>>>(tb.apost, T_run, B, h->H, M, attn_out);
      h->launches++;
    }
    COMIC_CHECK_CUDA(cudaGetLastError());
    return COMIC_OK;
  }

  // ---- transposed weights for the per-step backward GEMMs ----
  if (gru) {
    transpose(h->pk.gru_gx, KX, 3 * R, 3 * R, tb.KT, KX, st);                           // [gates | cand x-rows ; 0]^T [3R, KX]
    transpose(h->gru_cand_kernel + (size_t)XA * R, R, R, R, tb.KcT, R, st);              // candidate h-rows^T
    h->launches++;
  } else {
    transpose(h->w.lstm_kernel, KX, 4 * R, 4 * R, tb.KT, KX, st);
  }
  transpose(h->pk.outq, R, LQ, LQ, tb.outqT, R, st);
  COMIC_CHECK_CUDA(cudaMemsetAsync(tb.gH, 0, (size_t)B * R * sizeof(float), st));
  COMIC_CHECK_CUDA(cudaMemsetAsync(tb.gC, 0, (size_t)B * R * sizeof(float), st));
  COMIC_CHECK_CUDA(cudaMemsetAsync(tb.gCtx, 0, (size_t)B * A * sizeof(float), st));
  COMIC_CHECK_CUDA(cudaMemsetAsync(tb.dkeys, 0, (size_t)B * M * R * sizeof(float), st));
  if (h->cfg.fm_projection != 1) COMIC_CHECK_CUDA(cudaMemsetAsync(tb.dvals, 0, (size_t)B * M * VAL * sizeof(float), st));
  COMIC_CHECK_CUDA(cudaMemsetAsync(tb.cpart, 0, (size_t)B * tb.S * 3 * R * sizeof(float), st));
  COMIC_CHECK_CUDA(cudaMemsetAsync(tb.dTacc, 0, (size_t)B * sizeof(float), st));
  COMIC_CHECK_CUDA(cudaMemsetAsync(tb.dG, 0, (size_t)tb.rows_pad * 4 * R * sizeof(float), st));
  h->launches += 2;
  const float map_coef = (map_loss_scale > 0.f) ? -2.0f * map_loss_scale / ((float)B * (float)T_run * (float)M) : 0.f;
  float* dvals_dst = h->cfg.fm_projection == 1 ? tb.dkeys : tb.dvals;
  const bool ctx_layer = h->cfg.context_layer != 0, dot = h->cfg.alignment == 1, signorm = h->cfg.prob_fn == 1;
  if (ctx_layer) {
    COMIC_CHECK_CUDA(cudaMemsetAsync(tb.gctx_tape, 0, (size_t)tb.rows_pad * A * sizeof(float), st));
    transpose(h->w.a_layer, VAL, A, A, tb.aT, VAL, st);       // [A, VAL]
    h->launches++;
  }

  // ---- reverse sweep ----
  for (int t = T_run - 1; t >= 0; --t) {
    float* dlq_t = tb.dlq + (size_t)t * B * LQ;
    const float* dctx = tb.gCtx;
    int ld_dctx = A;
    if (ctx_layer) {
      // attention = ctxraw . a_layer (common/ops_rnn.py:734-739): the live rows' gradient is kept for the batched
      // d a_layer = ctxraw^T . g and pulled back to the raw context
      float* g_t = tb.gctx_tape + (size_t)t * B * A;
      mask_fin_copy_kernel<<<(unsigned)(((size_t)B * A + 255) / 256), 256, 0, st>>>(tb.gCtx, lens, t, g_t, B, A);
      h->launches++;
      if ((rc = train_gemm(h, g_t, A, tb.aT, VAL, tb.dctxraw, VAL, B, VAL, A, tb.part, tb.part_floats, st))) return rc;
      dctx = tb.dctxraw;
      ld_dctx = VAL;
    }
    {
      dim3 g1(B, tb.S);
      const int dvh = VAL / h->H;
      const bool vec_ok = VAL % 128 == 0 && dvh % (VAL / 32) == 0 && ((dvh / (VAL / 32)) & ((dvh / (VAL / 32)) - 1)) == 0 &&
                          ld_dctx % 4 == 0;
      if (vec_ok && VAL == 512)
        attn_bwd_dalpha_vec_kernel<512><<<g1, 256, 0, st>>>(values, dctx, ld_dctx, lens, t, tb.apost + (size_t)t * B * HM,
                                                           dvals_dst, tb.ds, 1, h->H, M, tb.S);
      else if (vec_ok && VAL == 256)
        attn_bwd_dalpha_vec_kernel<256><<<g1, 256, 0, st>>>(values, dctx, ld_dctx, lens, t, tb.apost + (size_t)t * B * HM,
                                                           dvals_dst, tb.ds, 1, h->H, M, tb.S);
      else if (vec_ok && VAL == 1024)
        attn_bwd_dalpha_vec_kernel<1024><<<g1, 256, 0, st>>>(values, dctx, ld_dctx, lens, t, tb.apost + (size_t)t * B * HM,
                                                            dvals_dst, tb.ds, 1, h->H, M, tb.S);
      else
        attn_bwd_dalpha_kernel<<<g1, 256, 0, st>>>(values, VAL, dctx, ld_dctx, lens, t, tb.apost + (size_t)t * B * HM, dvals_dst,
                                                  tb.ds, 1, h->H, M, tb.S);
      h->launches++;
    }
    attn_bwd_score_kernel<<<B, 256, (size_t)HM * sizeof(float), st>>>(
        values, VAL, dctx, ld_dctx, lens, t, tb.apost + (size_t)t * B * HM, tb.apre + (size_t)t * B * HM,
        mk.att ? mk.att + (size_t)t * B * HM : nullptr, att_keep, map_coef, nullptr, tb.ds, tb.dTacc,
        tb.maprows + (size_t)t * B, dot ? nullptr : h->w.temperature, 1, h->H, M, tb.ds,
        signorm ? tb.stape + (size_t)t * B * HM : nullptr);
    dim3 g2(B, tb.S);
    const float* lq_t = tb.lq + (size_t)t * B * LQ;
    if (dot) {
      if (R == 512)
        attn_bwd_dot_kernel<512><<<g2, 128, 0, st>>>(keys_buf, lq_t, LQ, h->Vp, tb.ds, tb.dkeys, tb.dqpart, 1, h->H, M, tb.S, B);
      else if (R == 256)
        attn_bwd_dot_kernel<256><<<g2, 128, 0, st>>>(keys_buf, lq_t, LQ, h->Vp, tb.ds, tb.dkeys, tb.dqpart, 1, h->H, M, tb.S, B);
      else
        attn_bwd_dot_kernel<1024><<<g2, 128, 0, st>>>(keys_buf, lq_t, LQ, h->Vp, tb.ds, tb.dkeys, tb.dqpart, 1, h->H, M, tb.S, B);
    } else if (R == 512)
      attn_bwd_ln_kernel<512><<<g2, 128, 0, st>>>(keys_buf, lq_t, LQ, h->Vp, h->w.ln_gamma, h->w.ln_beta, h->w.attention_v,
                                                 h->w.temperature, tb.ds, tb.dkeys, tb.dqpart, tb.cpart, 1, h->H, M, tb.S, B);
    else if (R == 256)
      attn_bwd_ln_kernel<256><<<g2, 128, 0, st>>>(keys_buf, lq_t, LQ, h->Vp, h->w.ln_gamma, h->w.ln_beta, h->w.attention_v,
                                                 h->w.temperature, tb.ds, tb.dkeys, tb.dqpart, tb.cpart, 1, h->H, M, tb.S, B);
    else
      attn_bwd_ln_kernel<1024><<<g2, 128, 0, st>>>(keys_buf, lq_t, LQ, h->Vp, h->w.ln_gamma, h->w.ln_beta, h->w.attention_v,
                                                  h->w.temperature, tb.ds, tb.dkeys, tb.dqpart, tb.cpart, 1, h->H, M, tb.S, B);
    sum_slices_kernel<<<(B * R + 255) / 256, 256, 0, st>>>(tb.dqpart, tb.S, B, R, dlq_t, LQ, h->Vp);
    h->launches += 3;
    // the two skinny GEMMs of the step split K; their consumers add the partials themselves (no reduce launches)
    int nzh = 1, nzx = 1;
    if ((rc = train_gemm(h, dlq_t, LQ, tb.outqT, R, tb.dHout, R, B, R, LQ, tb.part, tb.part_floats, st, &nzh))) return rc;
    float* dG_t = tb.dG + (size_t)(t + 1) * B * 4 * R;
    const float* tape_t = tb.gates + (size_t)(t + 1) * B * 4 * R;
    if (gru) {
      gru_bwd_a_kernel<<<(B * R + 255) / 256, 256, 0, st>>>(tape_t, nzh > 1 ? tb.part : tb.dHout,
                                                           mk.out ? mk.out + (size_t)t * B * R : nullptr, out_keep, lens, t, tb.gH,
                                                           dG_t, B, R, nzh, (size_t)B * R);
      int nzr = 1;   // d(r*h) = dC . Kc_h^T
      if ((rc = train_gemm(h, dG_t + 2 * R, 4 * R, tb.KcT, R, tb.dHout, R, B, R, R, tb.part, tb.part_floats, st, &nzr))) return rc;
      gru_bwd_b_kernel<<<(B * R + 255) / 256, 256, 0, st>>>(tape_t, tb.h + (size_t)t * B * R, nzr > 1 ? tb.part : tb.dHout, nzr,
                                                           (size_t)B * R, lens, t, tb.gH, tb.gHp, dG_t, B, R);
      h->launches += 2;
      // d[x, h] = [dR | dU | dC] . [gates | cand x-rows ; 0]^T
      if ((rc = train_gemm(h, dG_t, 4 * R, tb.KT, KX, tb.dxh, KX, B, KX, 3 * R, tb.part, tb.part_floats, st, &nzx))) return rc;
    } else {
      lstm_bwd_kernel<<<(B * R + 255) / 256, 256, 0, st>>>(tape_t, tb.c + (size_t)t * B * R,
                                                          nzh > 1 ? tb.part : tb.dHout, mk.out ? mk.out + (size_t)t * B * R : nullptr,
                                                          out_keep, lens, t, tb.gH, tb.gC, tb.gHp, dG_t, B, R, nzh, (size_t)B * R);
      if ((rc = train_gemm(h, dG_t, 4 * R, tb.KT, KX, tb.dxh, KX, B, KX, 4 * R, tb.part, tb.part_floats, st, &nzx))) return rc;
    }
    dx_split_kernel<<<(unsigned)(((size_t)B * KX + 255) / 256), 256, 0, st>>>(
        nzx > 1 ? tb.part : tb.dxh, KX, W, A, R, mk.inp ? mk.inp + (size_t)t * B * XA : nullptr, in_keep, lens, t,
        tb.demb + (size_t)t * B * W, tb.gCtx, tb.gH, tb.gHp, B, nzx, (size_t)B * KX);
    h->launches += 2;
  }
  // ---- init step backward ----
  float* dx0 = tb.dx0;
  COMIC_CHECK_CUDA(cudaMemsetAsync(dx0, 0, (size_t)((B + 3) / 4 * 4) * XA * sizeof(float), st));
  const int NI = (h->cfg.init_method == 1) ? R : XA;     // columns of the init weight
  if (h->cfg.init_method == 1) {
    // project_hidden: h0 = im_embed . W  ->  dW = im_embed^T . dh0; dx0 [B, R] holds dh0 for comic_train_encoder_grads
    copy2d_kernel<<<(unsigned)(((size_t)B * R + 255) / 256), 256, 0, st>>>(tb.gH, R, dx0, R, B, R);
    h->launches += 1;
  } else {
    if (gru) {
      gru_bwd_a_kernel<<<(B * R + 255) / 256, 256, 0, st>>>(tb.gates, nullptr, nullptr, 1.f, nullptr, 0, tb.gH, tb.dG, B, R);
      gru_bwd_b_kernel<<<(B * R + 255) / 256, 256, 0, st>>>(tb.gates, nullptr, nullptr, 0, 0, nullptr, 0, tb.gH, tb.gHp, tb.dG, B, R);
      h->launches++;
      if ((rc = train_gemm(h, tb.dG, 4 * R, tb.KT, KX, tb.dxh, KX, B, KX, 3 * R, tb.part, tb.part_floats, st))) return rc;
    } else {
      lstm_bwd_kernel<<<(B * R + 255) / 256, 256, 0, st>>>(tb.gates, nullptr, nullptr, nullptr, 1.f, nullptr, 0, tb.gH, tb.gC,
                                                          tb.gHp, tb.dG, B, R);
      if ((rc = train_gemm(h, tb.dG, 4 * R, tb.KT, KX, tb.dxh, KX, B, KX, 4 * R, tb.part, tb.part_floats, st))) return rc;
    }
    // dx0 = dxh[:, :XA] * init mask / keep
    copy2d_kernel<<<(unsigned)(((size_t)B * XA + 255) / 256), 256, 0, st>>>(tb.dxh, KX, dx0, XA, B, XA);
    if (mk.init_in) {
      size_t nx = (size_t)B * XA;
      mask_scale_kernel<<<(unsigned)((nx + 255) / 256), 256, 0, st>>>(dx0, mk.init_in, in_keep, nx);
    }
    h->launches += 3;
  }
  // dW_I [E, NI] = im_embed^T [E, B] . dx0 [B, NI]
  {
    int Bp = (B + 3) / 4 * 4;
    COMIC_CHECK_CUDA(cudaMemsetAsync(tb.embT, 0, (size_t)E * Bp * sizeof(float), st));
    transpose(im_embed, B, E, E, tb.embT, Bp, st);
    if ((rc = train_gemm(h, tb.embT, Bp, dx0, NI, grads->init_weight, NI, E, NI, Bp, tb.part, tb.part_floats, st))) return rc;
  }

  // ---- batched weight gradients ----
  const int rows = (int)(T1 * B), rows_pad = tb.rows_pad, rows_t = T_run * B;
  // dK = XH^T . dG ; db = colsum(dG)
  COMIC_CHECK_CUDA(cudaMemsetAsync(tb.xhT, 0, (size_t)KX * rows_pad * sizeof(float), st));
  {
    size_t n = (size_t)rows * KX;
    build_xh_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(tb.xd, tb.h, XA, R, tb.xh, rows, B);
  }
  transpose(tb.xh, rows, KX, KX, tb.xhT, rows_pad, st);
  if (gru) {
    // d gates/kernel = [x, h_prev]^T . [dR | dU];  d candidate/kernel = [x, r*h]^T . dC  (one GEMM each over all rows)
    if ((rc = train_gemm(h, tb.xhT, rows_pad, tb.dG, 4 * R, grads->lstm_kernel, 2 * R, KX, 2 * R, rows_pad, tb.part,
                         tb.part_floats, st))) return rc;
    colsum_kernel<<<(2 * R + 31) / 32, 256, 0, st>>>(tb.dG, rows, 2 * R, 4 * R, grads->lstm_bias, 0);
    size_t n = (size_t)rows * KX;
    build_xrh_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(tb.xd, tb.gates, XA, R, tb.xh, rows);
    transpose(tb.xh, rows, KX, KX, tb.xhT, rows_pad, st);
    if ((rc = train_gemm(h, tb.xhT, rows_pad, tb.dG + 2 * R, 4 * R, grads->cand_kernel, R, KX, R, rows_pad, tb.part,
                         tb.part_floats, st))) return rc;
    colsum_kernel<<<(R + 31) / 32, 256, 0, st>>>(tb.dG + 2 * R, rows, R, 4 * R, grads->cand_bias, 0);
    h->launches += 3;
  } else {
    if ((rc = train_gemm(h, tb.xhT, rows_pad, tb.dG, 4 * R, grads->lstm_kernel, 4 * R, KX, 4 * R, rows_pad, tb.part,
                         tb.part_floats, st))) return rc;
    colsum_kernel<<<(4 * R + 31) / 32, 256, 0, st>>>(tb.dG, rows, 4 * R, 4 * R, grads->lstm_bias, 0);
  }
  // d[W_o | W_q] = Hout^T . dLQ
  COMIC_CHECK_CUDA(cudaMemsetAsync(tb.hdT, 0, (size_t)R * rows_pad * sizeof(float), st));
  transpose(tb.hdrop, rows_t, R, R, tb.hdT, rows_pad, st);
  if ((rc = train_gemm(h, tb.hdT, rows_pad, tb.dlq, LQ, tb.dOutQ, LQ, R, LQ, rows_pad, tb.part, tb.part_floats, st))) return rc;
  copy2d_kernel<<<(unsigned)(((size_t)R * V + 255) / 256), 256, 0, st>>>(tb.dOutQ, LQ, grads->out_kernel, V, R, V);
  copy2d_kernel<<<(unsigned)(((size_t)R * R + 255) / 256), 256, 0, st>>>(tb.dOutQ + h->Vp, LQ, grads->query_kernel, R, R, R);
  colsum_kernel<<<(V + 31) / 32, 256, 0, st>>>(tb.dlq, rows_t, V, LQ, grads->out_bias, 0);
  // embedding
  embed_grad_kernel<<<V, 256, 0, st>>>(inputs_tm, tb.demb, rows_t, W, V, grads->embedding_map);
  // attention constants: column sums of the per-(image, slice) partials
  colsum_kernel<<<(R + 31) / 32, 256, 0, st>>>(tb.cpart, B * tb.S, R, 3 * R, grads->attention_v, 0);
  colsum_kernel<<<(R + 31) / 32, 256, 0, st>>>(tb.cpart + R, B * tb.S, R, 3 * R, grads->ln_gamma, 0);
  colsum_kernel<<<(R + 31) / 32, 256, 0, st>>>(tb.cpart + 2 * R, B * tb.S, R, 3 * R, grads->ln_beta, 0);
  scalar_sum_kernel<<<1, 32, 0, st>>>(tb.dTacc, B, 1.0f, grads->temperature);
  h->launches += 11;
  if (ctx_layer) {
    // d a_layer [VAL, A] = ctxraw^T [VAL, T*B] . g [T*B, A]   (rows of finished steps are zero in g)
    COMIC_CHECK_CUDA(cudaMemsetAsync(tb.ctxrawT, 0, (size_t)VAL * rows_pad * sizeof(float), st));
    transpose(tb.ctxraw, rows_t, VAL, VAL, tb.ctxrawT, rows_pad, st);
    if ((rc = train_gemm(h, tb.ctxrawT, rows_pad, tb.gctx_tape, A, grads->a_layer, A, VAL, A, rows_pad, tb.part,
                         tb.part_floats, st))) return rc;
    h->launches++;
  }
  // dW_k = F^T . dKeys  (tied: dKeys also holds the value-path gradient)
  {
    int bm = B * M, bmp = (bm + 3) / 4 * 4;
    COMIC_CHECK_CUDA(cudaMemsetAsync(tb.fmT, 0, (size_t)C * bmp * sizeof(float), st));
    transpose(fm, bm, C, C, tb.fmT, bmp, st);
    const int Kd = bm;                  // B * 196 is always a multiple of 4
    if ((rc = train_gemm(h, tb.fmT, bmp, tb.dkeys, R, grads->memory_kernel, R, C, R, Kd, tb.part, tb.part_floats, st))) return rc;
    if (h->cfg.fm_projection == 2 && grads->value_kernel)
      if ((rc = train_gemm(h, tb.fmT, bmp, tb.dvals, R, grads->value_kernel, R, C, R, Kd, tb.part, tb.part_floats, st))) return rc;
    h->launches++;
  }
  // ---- losses: [total (without reg), xe, map, 0] ----
  scalar_sum_kernel<<<1, 32, 0, st>>>(tb.rowloss, rows_t, 1.0f, loss_out + 1);
  scalar_sum_kernel<<<1, 32, 0, st>>>(tb.maprows, rows_t,
                                     map_loss_scale > 0.f ? map_loss_scale / ((float)B * (float)T_run * (float)M) : 0.f,
                                     loss_out + 2);
  h->launches += 2;
  // attention maps [B, H, T_run, M] (post-dropout history, model_base.py:307-313)
  if (attn_out) {
    dim3 g(T_run, B);
    attn_maps_kernel<<<g, 256, 0, st>>>(tb.apost, T_run, B, h->H, M, attn_out);
    h->launches++;
  }
  COMIC_CHECK_CUDA(cudaGetLastError());
  return COMIC_OK;
}

__global__ void add_inplace_kernel(float* __restrict__ dst, const float* __restrict__ src, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] += src[i];
}

extern "C" int comic_train_encoder_grads(comic_handle_t h, int B, int T_run, float* dfm_out, float* dim_embed_out,
                                         void* ws, size_t ws_bytes, void* stream) {
  COMIC_REQUIRE(h && h->bound && dfm_out && dim_embed_out && ws, COMIC_E_BADARG, "train_encoder_grads: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  size_t need;
  train_workspace_bytes(h, B, T_run, &need);
  COMIC_REQUIRE(ws_bytes >= need, COMIC_E_WORKSPACE, "train_encoder_grads: workspace %zu < %zu", ws_bytes, need);
  Carver cv(ws);
  TrainBufs tb;
  carve_train(h, cv, B, T_run, tb);
  const int R = h->R, C = h->C, E = h->E, XA = h->W + h->A, M = h->M;
  const int bm = B * M;
  int rc;
  // dfm = dkeys . W_k^T  (tied: dkeys already carries the value-path gradient)
  transpose(h->w.memory_kernel, C, R, R, tb.encT, C, st);
  if ((rc = train_gemm(h, tb.dkeys, R, tb.encT, C, dfm_out, C, bm, C, R, tb.part, tb.part_floats, st))) return rc;
  size_t n = (size_t)bm * C;
  if (h->cfg.fm_projection == 2) {
    transpose(h->w.value_kernel, C, R, R, tb.encT, C, st);
    if ((rc = train_gemm(h, tb.dvals, R, tb.encT, C, tb.dfm_tmp, C, bm, C, R, tb.part, tb.part_floats, st))) return rc;
    add_inplace_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(dfm_out, tb.dfm_tmp, n);
    h->launches += 2;
  } else if (h->cfg.fm_projection == 0) {
    add_inplace_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(dfm_out, tb.dvals, n);   // values = fm itself
    h->launches++;
  }
  // dim_embed = dx0 . W_I^T   (project_hidden: dx0 holds dh0 [B, R] and W_I is [E, R])
  const int NI = (h->cfg.init_method == 1) ? R : XA;
  transpose(h->w.init_weight, E, NI, NI, tb.encT, E, st);
  if ((rc = train_gemm(h, tb.dx0, NI, tb.encT, E, dim_embed_out, E, B, E, NI, tb.part, tb.part_floats, st))) return rc;
  h->launches += 2;
  COMIC_CHECK_CUDA(cudaGetLastError());
  return COMIC_OK;
}

// floats of workspace comic_legacy_head_bwd needs for B images
static size_t legacy_head_ws_floats(int B) {
  const size_t Bp = (size_t)(B + 3) / 4 * 4, C = 1024;
  return 5 * Bp * C + C * C + C * Bp + (size_t)4 * 1024 * 1024 + 64;
}

extern "C" int comic_legacy_head_bwd_bytes(comic_handle_t h, int B, size_t* bytes) {
  COMIC_REQUIRE(h && bytes && B > 0, COMIC_E_BADARG, "legacy_head_bwd_bytes: bad argument");
  *bytes = legacy_head_ws_floats(B) * sizeof(float);
  return COMIC_OK;
}

extern "C" int comic_legacy_head_bwd(comic_handle_t h, const float* mixed5c, int B, const float* d_im_embed, float* d_gamma,
                                     float* d_beta, float* d_weight, void* ws, size_t ws_bytes, void* stream) {
  COMIC_REQUIRE(h && h->bound && mixed5c && d_im_embed && d_gamma && d_beta && d_weight && ws && B > 0, COMIC_E_BADARG,
                "legacy_head_bwd: bad argument");
  COMIC_REQUIRE(h->cfg.legacy && h->w.enc_ln_gamma && h->w.enc_ln_beta && h->w.enc_embed_weight, COMIC_E_BADARG,
                "legacy_head_bwd: the model has no legacy head");
  COMIC_REQUIRE(ws_bytes >= legacy_head_ws_floats(B) * sizeof(float), COMIC_E_WORKSPACE, "legacy_head_bwd: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  const int C = 1024, Bp = (B + 3) / 4 * 4;
  Carver cv(ws);
  float* xhat = cv.take<float>((size_t)Bp * C);
  float* t1 = cv.take<float>((size_t)Bp * C);
  float* d_t1 = cv.take<float>((size_t)Bp * C);
  float* d_im_p = cv.take<float>((size_t)Bp * C);
  float* t1T = cv.take<float>((size_t)C * Bp);
  float* WT = cv.take<float>((size_t)C * C);
  const size_t part_floats = (size_t)4 * 1024 * 1024;
  float* part = cv.take<float>(part_floats);
  int rc;
  legacy_head_recompute_kernel<<<B, 256, 0, st>>>(mixed5c, h->w.enc_ln_gamma, h->w.enc_ln_beta, xhat, t1, 49, C);
  // d t1 = d im_embed . W^T
  transpose(h->w.enc_embed_weight, C, C, C, WT, C, st);
  if ((rc = train_gemm(h, d_im_embed, C, WT, C, d_t1, C, B, C, C, part, part_floats, st))) return rc;
  // d W [C, C] = t1^T [C, B] . d im_embed [B, C]   (rows padded to a multiple of 4 with zeros)
  COMIC_CHECK_CUDA(cudaMemsetAsync(t1T, 0, (size_t)C * Bp * sizeof(float), st));
  COMIC_CHECK_CUDA(cudaMemsetAsync(d_im_p, 0, (size_t)Bp * C * sizeof(float), st));
  transpose(t1, B, C, C, t1T, Bp, st);
  COMIC_CHECK_CUDA(cudaMemcpyAsync(d_im_p, d_im_embed, (size_t)B * C * sizeof(float), cudaMemcpyDeviceToDevice, st));
  if ((rc = train_gemm(h, t1T, Bp, d_im_p, C, d_weight, C, C, C, Bp, part, part_floats, st))) return rc;
  // through tanh and the layer norm's affine part: d beta = sum_b d_ln, d gamma = sum_b d_ln * xhat
  {
    const size_t n = (size_t)B * C;
    legacy_head_dln_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_t1, xhat, t1, n);
  }
  colsum_kernel<<<(C + 31) / 32, 256, 0, st>>>(d_t1, B, C, C, d_beta, 0);
  colsum_kernel<<<(C + 31) / 32, 256, 0, st>>>(xhat, B, C, C, d_gamma, 0);
  h->launches += 7;
  COMIC_CHECK_CUDA(cudaGetLastError());
  return COMIC_OK;
}

extern "C" int comic_l2_regularise(comic_handle_t h, const float* params, float* grads, size_t n, float decay,
                                   float* reg_out, void* ws, size_t ws_bytes, void* stream) {
  COMIC_REQUIRE(h && params && reg_out && ws && ws_bytes >= 1024 * sizeof(float), COMIC_E_BADARG, "l2_regularise: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  float* partial = static_cast<float*>(ws);
  int blocks = 512;
  l2_kernel<<<blocks, 256, 0, st>>>(params, grads, n, decay, partial);
  scalar_sum_kernel<<<1, 32, 0, st>>>(partial, blocks, 0.5f * decay, reg_out);
  h->launches += 2;
  COMIC_CHECK_CUDA(cudaGetLastError());
  return COMIC_OK;
}

extern "C" int comic_adam_step(comic_handle_t h, float* params, const float* grads, float* m, float* v, size_t n,
                               float lr, float beta1, float beta2, float eps, int step, float grad_scale, void* stream) {
  COMIC_REQUIRE(h && params && grads && m && v && step >= 1, COMIC_E_BADARG, "adam_step: bad argument");
  double lr_t = (double)lr * sqrt(1.0 - pow((double)beta2, step)) / (1.0 - pow((double)beta1, step));
  adam_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(params, grads, m, v, n, (float)lr_t, beta1,
                                                                            beta2, eps, grad_scale);
  h->launches++;
  h->attn2_state = 0;   // attention_v / temperature may have moved: re-check the score bound (decoder.cu attn2_prepare)
  COMIC_CHECK_CUDA(cudaGetLastError());
  return COMIC_OK;
}

extern "C" int comic_momentum_step(comic_handle_t h, float* params, const float* grads, float* accum, size_t n, float lr,
                                   float momentum, float grad_scale, void* stream) {
  COMIC_REQUIRE(h && params && grads && accum, COMIC_E_BADARG, "momentum_step: bad argument");
  momentum_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(params, grads, accum, n, lr, momentum,
                                                                                grad_scale);
  h->launches++;
  h->attn2_state = 0;
  COMIC_CHECK_CUDA(cudaGetLastError());
  return COMIC_OK;
}

extern "C" int comic_clip_by_norm(comic_handle_t h, float* grads, const int64_t* offsets, const int64_t* sizes, int nvars,
                                  float max_norm, void* stream) {
  COMIC_REQUIRE(h && grads && offsets && sizes && nvars > 0 && max_norm > 0.f, COMIC_E_BADARG, "clip_by_norm: bad argument");
  clip_by_norm_kernel<<<nvars, 1024, 0, (cudaStream_t)stream>>>(grads, reinterpret_cast<const long long*>(offsets),
                                                               reinterpret_cast<const long long*>(sizes), max_norm);
  h->launches++;
  COMIC_CHECK_CUDA(cudaGetLastError());
  return COMIC_OK;
}

// Re-derive the decoder's engine-layout copies of the weights (packed [W_o|W_q] panel, tensor-path
// bf16 panels) after the optimiser changed the variables in place.  `packed` is the buffer given
// to comic_bind_weights (the decoder packs sit at its start, so their addresses do not move).
extern "C" int comic_refresh_packed(comic_handle_t h, void* packed, size_t packed_bytes, void* stream) {
  COMIC_REQUIRE(h && h->bound && packed, COMIC_E_BADARG, "refresh_packed: not bound");
  (void)packed_bytes;
  h->attn2_state = 0;
  Carver cv(packed);
  return decoder_pack(h, cv, (cudaStream_t)stream, false);
}
