// gemm_f32.cuh -- fp32 FFMA GEMM / implicit-GEMM convolution for sm_100a.
//
// C[M,N] = A[M,K] . B[K,N] with fp32 operands and fp32 accumulation, i.e. the
// exact-parity ("f32") arithmetic of the reference graph (all reference math is
// fp32, SURVEY.md §8).  Two A-operand providers:
//   APlain : up to 3 concatenated column segments, each with an optional row
//            indirection -> [emb(tok) ; ctx[src] ; h[src]] is read in place, the
//            beam-search state gather (TF _beam_search_step) is never materialised.
//   AConv  : NHWC implicit GEMM with TF `SAME` asymmetric zero padding
//            (im2col done by the loader; weights HWIO = row-major [K,N]).
// Epilogue: optional per-column scale/shift (folded inference BN), ReLU, and a
// column-range routing table so that one GEMM over the concatenated 1x1
// branch weights of an inception block stores each branch where it belongs
// (concat output at a channel offset / temporaries).  Split-K (gridDim.z)
// writes deterministic partials that the consumer reduces in a fixed order.
//
// 256 threads, BMxBNxBK tiles, TMxTN register tiles, register-prefetch double
// buffering through shared memory, 128-bit loads/stores.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace comic {

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-DEVICE attribute of a kernel: a process that drives several
// GPUs (one Engine per device) has to set it once on each.  One flag set per launch-site template instantiation.
struct PerDeviceOnce {
  bool done[64] = {};
  template <typename F>
  cudaError_t operator()(F&& configure) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= 64) return configure();
    if (done[dev]) return cudaSuccess;
    e = configure();
    if (e == cudaSuccess) done[dev] = true;
    return e;
  }
};


struct ASeg {
  const float* ptr;
  const int* idx;   // row indirection (nullptr = identity); value < 0 or >= idx_limit -> zero row
  int ld;
  int ncols;
  int idx_limit;    // exclusive upper bound for idx values (rows available in ptr)
};

struct APlain {
  ASeg seg[3];
  int nseg;
};

struct AConv {
  const float* x;   // [B, H, W, ldx] NHWC, channels [0, Cin)
  int H, W, Cin, ldx;
  int KH, KW, stride, pad_t, pad_l, Ho, Wo;
};

struct Route {
  int n0, n1;   // column range [n0, n1)
  float* dst;
  int ld;
  int coff;
};

struct Epi {
  const float* bias;   // per-column add (after scale), nullable
  const float* scale;  // per-column multiply, nullable
  int relu;
  int nroute;
  Route r[3];
  long long split_stride;  // elements between split-K partials of route 0
  int ksplit;              // tensor path (gemm_tc.cuh, AMODE 0, single-CTA kernel): K blocks cut into this many ranges, partial
                           // z of tile (m, n) goes to route dst + z * split_stride (0 / 1 = off); no bias / scale then
  const int* stop;         // optional device flag: skip the launch when *stop >= stop_n
  int stop_n;              // (decode loops: every beam finished in the previous step)
};

// sigmoid / tanh of the big-batch decode path (engine precision >= 1): ex2.approx + rcp, relative error ~1e-6 against
// expf / tanhf -- the same budget as the bf16x3 GEMM feeding them.  FAST = false: libm.
template <bool FAST>
__device__ __forceinline__ float sig_(float x) {
  if (FAST) return __frcp_rn(1.0f + __expf(-x));
  return 1.0f / (1.0f + expf(-x));
}
template <bool FAST>
__device__ __forceinline__ float tanh_(float x) {
  if (FAST) {
    const float e = __expf(-2.0f * fabsf(x));           // in (0, 1]: no overflow
    return copysignf((1.0f - e) * __frcp_rn(1.0f + e), x);
  }
  return tanhf(x);
}

// Stem conv over the space-to-depth image (bf16 planes [nimg,112,112,16]) with the im2col tile built from a
// shared-memory halo patch instead of 16 L2 reads per input element (tensor path, gemm_tc.cuh AMODE 3).
struct AHalo {
  const uint16_t* hi;
  const uint16_t* lo;
  int nimg;
};

template <int AMODE> struct AParam;
template <> struct AParam<0> { typedef APlain type; };
template <> struct AParam<1> { typedef AConv type; };
template <> struct AParam<3> { typedef AHalo type; };
// AMODE 4 (tensor path only): the A operand exists as bf16 (hi, lo) planes [rows, K] in global memory and is staged by
// TMA like the weights -- no loader warps, no per-CTA gather / split (decoder GEMMs: gemm_tc.cuh, decoder.cu)
struct ATma {
  CUtensorMap hi, lo;
};
template <> struct AParam<4> { typedef ATma type; };

__device__ __forceinline__ float4 ldg4(const float* p) {
  return __ldg(reinterpret_cast<const float4*>(p));
}

// Row context of one A-tile slot owned by a thread.
template <int AMODE> struct RowCtx;
template <> struct RowCtx<0> {
  const float* base[3];
  bool valid;
};
template <> struct RowCtx<1> {
  const float* base;  // image base
  int hi0, wi0;
  bool valid;
};

template <int AMODE>
__device__ __forceinline__ void make_row(const typename AParam<AMODE>::type& a, int m, int M,
                                         RowCtx<AMODE>& rc);

template <>
__device__ __forceinline__ void make_row<0>(const APlain& a, int m, int M, RowCtx<0>& rc) {
  rc.valid = m < M;
#pragma unroll
  for (int s = 0; s < 3; ++s) {
    rc.base[s] = nullptr;
    if (s < a.nseg && rc.valid) {
      int r = m;
      if (a.seg[s].idx) r = a.seg[s].idx[m];
      if (r >= 0 && r < a.seg[s].idx_limit) rc.base[s] = a.seg[s].ptr + (size_t)r * a.seg[s].ld;
    }
  }
}

template <>
__device__ __forceinline__ void make_row<1>(const AConv& a, int m, int M, RowCtx<1>& rc) {
  rc.valid = m < M;
  int hw = a.Ho * a.Wo;
  int b = rc.valid ? m / hw : 0;
  int rem = rc.valid ? m - b * hw : 0;
  int ho = rem / a.Wo;
  int wo = rem - ho * a.Wo;
  rc.hi0 = ho * a.stride - a.pad_t;
  rc.wi0 = wo * a.stride - a.pad_l;
  rc.base = a.x + (size_t)b * a.H * a.W * a.ldx;
}

// Load 4 consecutive K elements [kk, kk+4) of one row.
template <int AMODE, int VEC>
__device__ __forceinline__ float4 load_a4(const typename AParam<AMODE>::type& a,
                                          const RowCtx<AMODE>& rc, int kk, int K);

template <>
__device__ __forceinline__ float4 load_a4<0, 4>(const APlain& a, const RowCtx<0>& rc, int kk, int K) {
  float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
  if (!rc.valid || kk >= K) return z;
  int k0 = kk;
#pragma unroll
  for (int s = 0; s < 3; ++s) {
    if (s < a.nseg) {
      if (k0 < a.seg[s].ncols) {
        return rc.base[s] ? ldg4(rc.base[s] + k0) : z;
      }
      k0 -= a.seg[s].ncols;
    }
  }
  return z;
}

template <>
__device__ __forceinline__ float4 load_a4<0, 1>(const APlain& a, const RowCtx<0>& rc, int kk, int K) {
  float v[4] = {0.f, 0.f, 0.f, 0.f};
  if (rc.valid) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int k0 = kk + j;
      if (k0 < K) {
#pragma unroll
        for (int s = 0; s < 3; ++s) {
          if (s < a.nseg) {
            if (k0 >= 0 && k0 < a.seg[s].ncols) {
              if (rc.base[s]) v[j] = __ldg(rc.base[s] + k0);
              k0 = -1;
            } else if (k0 >= 0) {
              k0 -= a.seg[s].ncols;
            }
          }
        }
      }
    }
  }
  return make_float4(v[0], v[1], v[2], v[3]);
}

template <>
__device__ __forceinline__ float4 load_a4<1, 4>(const AConv& a, const RowCtx<1>& rc, int kk, int K) {
  float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
  if (!rc.valid || kk >= K) return z;
  int tap = kk / a.Cin;
  int ci = kk - tap * a.Cin;
  int kh = tap / a.KW;
  int kw = tap - kh * a.KW;
  int hi = rc.hi0 + kh, wi = rc.wi0 + kw;
  if (hi < 0 || hi >= a.H || wi < 0 || wi >= a.W) return z;
  return ldg4(rc.base + ((size_t)hi * a.W + wi) * a.ldx + ci);
}

template <>
__device__ __forceinline__ float4 load_a4<1, 1>(const AConv& a, const RowCtx<1>& rc, int kk, int K) {
  float v[4] = {0.f, 0.f, 0.f, 0.f};
  if (rc.valid) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int k0 = kk + j;
      if (k0 < K) {
        int tap = k0 / a.Cin;
        int ci = k0 - tap * a.Cin;
        int kh = tap / a.KW;
        int kw = tap - kh * a.KW;
        int hi = rc.hi0 + kh, wi = rc.wi0 + kw;
        if (hi >= 0 && hi < a.H && wi >= 0 && wi < a.W)
          v[j] = __ldg(rc.base + ((size_t)hi * a.W + wi) * a.ldx + ci);
      }
    }
  }
  return make_float4(v[0], v[1], v[2], v[3]);
}

template <int BM, int BN, int BK, int TM, int TN, int AMODE, int VEC>
__global__ void __launch_bounds__(256, 2)
gemm_f32_kernel(typename AParam<AMODE>::type a, const float* __restrict__ Bm, int ldb, int M, int N,
                int K, int k_per_split, Epi epi) {
  static_assert((BM / TM) * (BN / TN) == 256, "thread tiling must cover the CTA tile");
  constexpr int LA = BM * BK / 1024;  // float4 slots per thread for A
  constexpr int LB = BK * BN / 1024;
  static_assert(LA >= 1 && LB >= 1, "tile too small");
  constexpr int PAD = 4;
  __shared__ __align__(16) float As[2][BK][BM + PAD];
  __shared__ __align__(16) float Bs[2][BK][BN];

  if (epi.stop != nullptr && *epi.stop >= epi.stop_n) return;
  const int tid = threadIdx.x;
  const int m0 = blockIdx.y * BM;
  const int n0 = blockIdx.x * BN;
  const int kbeg = blockIdx.z * k_per_split;
  const int kend = min(K, kbeg + k_per_split);

  RowCtx<AMODE> rc[LA];
  int a_row[LA], a_kq[LA];
#pragma unroll
  for (int i = 0; i < LA; ++i) {
    int s = tid + 256 * i;
    a_row[i] = s / (BK / 4);
    a_kq[i] = s % (BK / 4);
    make_row<AMODE>(a, m0 + a_row[i], M, rc[i]);
  }
  int b_k[LB], b_n[LB];
#pragma unroll
  for (int i = 0; i < LB; ++i) {
    int s = tid + 256 * i;
    b_k[i] = s / (BN / 4);
    b_n[i] = (s % (BN / 4)) * 4;
  }

  float4 ra[LA], rb[LB];
  auto gload = [&](int kt) {
#pragma unroll
    for (int i = 0; i < LA; ++i) {
      int kk = kt + a_kq[i] * 4;
      // VEC == 4 requires K % 4 == 0 and 4-aligned segments (checked by the dispatcher).
      ra[i] = (kk < kend) ? load_a4<AMODE, VEC>(a, rc[i], kk, kend) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int i = 0; i < LB; ++i) {
      int kk = kt + b_k[i];
      int n = n0 + b_n[i];
      rb[i] = (kk < kend && n < N) ? ldg4(Bm + (size_t)kk * ldb + n) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  auto sstore = [&](int buf) {
#pragma unroll
    for (int i = 0; i < LA; ++i) {
      As[buf][a_kq[i] * 4 + 0][a_row[i]] = ra[i].x;
      As[buf][a_kq[i] * 4 + 1][a_row[i]] = ra[i].y;
      As[buf][a_kq[i] * 4 + 2][a_row[i]] = ra[i].z;
      As[buf][a_kq[i] * 4 + 3][a_row[i]] = ra[i].w;
    }
#pragma unroll
    for (int i = 0; i < LB; ++i) {
      *reinterpret_cast<float4*>(&Bs[buf][b_k[i]][b_n[i]]) = rb[i];
    }
  };

  const int tx = tid % (BN / TN);
  const int ty = tid / (BN / TN);
  // Row / column ownership: 4-wide groups, second group offset by half a tile
  // (conflict-free 128-bit shared loads).
  int rowoff[TM], coloff[TN];
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    if (TM == 8) rowoff[i] = (i < 4) ? ty * 4 + i : BM / 2 + ty * 4 + (i - 4);
    else rowoff[i] = ty * TM + i;
  }
#pragma unroll
  for (int j = 0; j < TN; ++j) {
    if (TN == 8) coloff[j] = (j < 4) ? tx * 4 + j : BN / 2 + tx * 4 + (j - 4);
    else coloff[j] = tx * TN + j;
  }

  float acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

  int buf = 0;
  if (kbeg < kend) {
    gload(kbeg);
    sstore(0);
  }
  __syncthreads();
  for (int kt = kbeg; kt < kend; kt += BK) {
    const bool more = kt + BK < kend;
    if (more) gload(kt + BK);
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      float av[TM], bv[TN];
      if (TM == 8) {
        float4 t0 = *reinterpret_cast<const float4*>(&As[buf][kk][ty * 4]);
        float4 t1 = *reinterpret_cast<const float4*>(&As[buf][kk][BM / 2 + ty * 4]);
        av[0] = t0.x; av[1] = t0.y; av[2] = t0.z; av[3] = t0.w;
        av[4] = t1.x; av[5] = t1.y; av[6] = t1.z; av[7] = t1.w;
      } else if (TM == 4) {
        float4 t0 = *reinterpret_cast<const float4*>(&As[buf][kk][ty * 4]);
        av[0] = t0.x; av[1] = t0.y; av[2] = t0.z; av[3] = t0.w;
      } else {
#pragma unroll
        for (int i = 0; i < TM; ++i) av[i] = As[buf][kk][ty * TM + i];
      }
      if (TN == 8) {
        float4 t0 = *reinterpret_cast<const float4*>(&Bs[buf][kk][tx * 4]);
        float4 t1 = *reinterpret_cast<const float4*>(&Bs[buf][kk][BN / 2 + tx * 4]);
        bv[0] = t0.x; bv[1] = t0.y; bv[2] = t0.z; bv[3] = t0.w;
        bv[4] = t1.x; bv[5] = t1.y; bv[6] = t1.z; bv[7] = t1.w;
      } else {
        float4 t0 = *reinterpret_cast<const float4*>(&Bs[buf][kk][tx * 4]);
        bv[0] = t0.x; bv[1] = t0.y; bv[2] = t0.z; bv[3] = t0.w;
      }
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    if (more) sstore(buf ^ 1);
    __syncthreads();
    buf ^= 1;
  }

  // Epilogue: 4 consecutive columns at a time.
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    int m = m0 + rowoff[i];
    if (m >= M) continue;
#pragma unroll
    for (int jg = 0; jg < TN / 4; ++jg) {
      int n = n0 + coloff[jg * 4];
      if (n >= N) continue;
      float4 v = make_float4(acc[i][jg * 4 + 0], acc[i][jg * 4 + 1], acc[i][jg * 4 + 2],
                             acc[i][jg * 4 + 3]);
      if (epi.scale) {
        float4 s = ldg4(epi.scale + n);
        v.x *= s.x; v.y *= s.y; v.z *= s.z; v.w *= s.w;
      }
      if (epi.bias) {
        float4 s = ldg4(epi.bias + n);
        v.x += s.x; v.y += s.y; v.z += s.z; v.w += s.w;
      }
      if (epi.relu) {
        v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f);
      }
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        if (r < epi.nroute && n >= epi.r[r].n0 && n < epi.r[r].n1) {
          float* dst = epi.r[r].dst + (size_t)blockIdx.z * epi.split_stride + (size_t)m * epi.r[r].ld +
                       epi.r[r].coff + (n - epi.r[r].n0);
          *reinterpret_cast<float4*>(dst) = v;
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------
// Host-side dispatch.
// ---------------------------------------------------------------------------
struct GemmPlan {
  int cfg;     // 0: 128x128x16 (8x8), 1: 64x64x16 (4x4), 2: 32x64x32 (2x4)
  int splitk;  // >= 1
};

inline GemmPlan plan_gemm(int M, int N, int K, int num_sms, bool allow_split) {
  GemmPlan p;
  auto tiles = [&](int bm, int bn) { return ((M + bm - 1) / bm) * ((N + bn - 1) / bn); };
  if (M <= 32) p.cfg = 2;
  else if (M <= 64 || tiles(128, 128) < num_sms) p.cfg = 1;
  else p.cfg = 0;
  p.splitk = 1;
  if (allow_split) {
    int t = p.cfg == 0 ? tiles(128, 128) : (p.cfg == 1 ? tiles(64, 64) : tiles(32, 64));
    int bk = p.cfg == 2 ? 32 : 16;
    int maxsplit = K / (bk * 4);   // at least 4 K-tiles per split
    if (maxsplit < 1) maxsplit = 1;
    // small-M launches are K-loop latency chains (load -> barrier -> FMA per K tile, ~35 % issue activity at 8 warps per SM):
    // two CTAs per SM overlap them, so the split may fill up to 2.5 waves of one CTA per SM (was 1.5)
    const int fill = (p.cfg == 2) ? 2 * num_sms + num_sms / 2 : num_sms + num_sms / 2;
    while (t * p.splitk * 2 <= fill && p.splitk * 2 <= maxsplit && p.splitk < 16) p.splitk *= 2;
  }
  return p;
}

template <int AMODE, int VEC>
inline cudaError_t launch_gemm(const typename AParam<AMODE>::type& a, const float* Bm, int ldb, int M,
                               int N, int K, const Epi& epi, GemmPlan p, cudaStream_t st) {
  if (M <= 0 || N <= 0) return cudaSuccess;
  int bk = p.cfg == 2 ? 32 : 16;
  int kps = K;
  if (p.splitk > 1) {
    kps = (K + p.splitk - 1) / p.splitk;
    kps = ((kps + bk - 1) / bk) * bk;
  }
  int nz = (K + kps - 1) / kps;
  if (nz < 1) nz = 1;
  if (p.cfg == 0) {
    dim3 g((N + 127) / 128, (M + 127) / 128, nz);
    gemm_f32_kernel<128, 128, 16, 8, 8, AMODE, VEC><<<g, 256, 0, st>>>(a, Bm, ldb, M, N, K, kps, epi);
  } else if (p.cfg == 1) {
    dim3 g((N + 63) / 64, (M + 63) / 64, nz);
    gemm_f32_kernel<64, 64, 16, 4, 4, AMODE, VEC><<<g, 256, 0, st>>>(a, Bm, ldb, M, N, K, kps, epi);
  } else {
    dim3 g((N + 63) / 64, (M + 31) / 32, nz);
    gemm_f32_kernel<32, 64, 32, 2, 4, AMODE, VEC><<<g, 256, 0, st>>>(a, Bm, ldb, M, N, K, kps, epi);
  }
  return cudaGetLastError();
}

// Number of split-K partials launch_gemm will produce for (K, plan).
inline int gemm_num_partials(int K, GemmPlan p) {
  if (p.splitk <= 1) return 1;
  int bk = p.cfg == 2 ? 32 : 16;
  int kps = (K + p.splitk - 1) / p.splitk;
  kps = ((kps + bk - 1) / bk) * bk;
  return (K + kps - 1) / kps;
}

}  // namespace comic
