// encoder_train.cu -- InceptionV1 forward-with-tape and backward for train_mode=cnn_finetune.
//
// The reference fine-tunes the CNN by letting TF autodiff run through the slim graph of
// common/nets/inception_v1.py:29-266 with `is_training=False` (src/model_base.py:71-77): batch
// norm keeps using its MOVING statistics, so the trainable CNN variables are the 57 conv kernels
// and the 57 BN betas (src/train.py:241-250 clears freeze_scopes; src/model_base.py:367-401).
// With y = relu(s * conv(x, W) + beta - mean * s), s = rsqrt(var + 1e-3):
//     dz    = dy * [y > 0] * s          (gradient at the conv output)
//     dbeta = sum_rows dy * [y > 0]
//     dW    = im2col(x)^T . dz           (wgrad: reduction over all B*Ho*Wo output pixels)
//     dx    = conv(dz, flip(W)^T)        (dgrad: every conv that needs it has stride 1, odd k)
// Max-pool backward sends dy to the first maximum of each window in row-major scan order (the
// rule of TF's MaxPoolGrad and of torch's max_pool2d backward); it is written as a gather so the
// overlapping 3x3 windows need no atomics and the result is bit-reproducible.
//
// Kernels: wgrad_kernel (FFMA, 64x64 output tile, split over the pixel dimension with a
// fixed-order partial reduction), relu_bn_bwd_kernel (+ per-chunk beta partials), the dgrad runs
// on the forward's implicit-GEMM kernels over a flipped/transposed weight panel (FFMA, or the
// tcgen05 bf16x3 kernel when precision >= 1), maxpool_bwd_kernel, avgpool_bwd_kernel.
#include "comic_internal.cuh"

namespace comic {

static const int kBlkS[kNumBlocks] = {28, 28, 14, 14, 14, 14, 14, 7, 7};

struct EncTape {
  float *c1, *p1, *c2b, *c2c, *p2, *p3, *p4;
  float *y[kNumBlocks], *t1[kNumBlocks], *t2[kNumBlocks], *p[kNumBlocks];
};

static inline int blk_cout(const BlockDesc& b) { return b.b0 + b.b1b + b.b2b + b.b3; }

static void carve_tape(Carver& cv, int B, EncTape& tp) {
  const BlockDesc* blk = block_table();
  tp.c1 = cv.take<float>((size_t)B * 112 * 112 * 64);
  tp.p1 = cv.take<float>((size_t)B * 56 * 56 * 64);
  tp.c2b = cv.take<float>((size_t)B * 56 * 56 * 64);
  tp.c2c = cv.take<float>((size_t)B * 56 * 56 * 192);
  tp.p2 = cv.take<float>((size_t)B * 28 * 28 * 192);
  tp.p3 = cv.take<float>((size_t)B * 14 * 14 * 480);
  tp.p4 = cv.take<float>((size_t)B * 7 * 7 * 832);
  for (int i = 0; i < kNumBlocks; ++i) {
    size_t M = (size_t)B * kBlkS[i] * kBlkS[i];
    tp.y[i] = cv.take<float>(M * blk_cout(blk[i]));
    tp.t1[i] = cv.take<float>(M * blk[i].b1a);
    tp.t2[i] = cv.take<float>(M * blk[i].b2a);
    tp.p[i] = cv.take<float>(M * blk[i].cin);
  }
}

static const float* blk_input(const EncTape& tp, int i) {
  if (i == 0) return tp.p2;
  if (i == 2) return tp.p3;
  if (i == 7) return tp.p4;
  return tp.y[i - 1];
}

// The tape tensor that is attention end point `tap` (COMIC_FM_*).
static const float* fm_tap_tensor(const EncTape& tp, int tap) {
  if (tap == COMIC_FM_MAXPOOL_4A_3X3) return tp.p3;
  if (tap == COMIC_FM_MAXPOOL_5A_2X2) return tp.p4;
  return tp.y[fm_tap_block(tap)];
}

// ---------------------------------------------------------------------------
// Backward kernels.
// ---------------------------------------------------------------------------

// dz[m, c] = dy[m, c] * [y[m, c] > 0] * scale[c]; bpart[chunk, c] = sum over the chunk's rows of
// dy * [y > 0].  Block = 64 columns x 4 row lanes; grid = (row chunks, column groups of 64).
__global__ void __launch_bounds__(256)
relu_bn_bwd_kernel(const float* __restrict__ dy, int ld_dy, int coff_dy, const float* __restrict__ y, int ld_y,
                   int coff_y, const float* __restrict__ scale, float* __restrict__ dz, int ld_dz, int coff_dz,
                   int M, int n, int rows_per_chunk, float* __restrict__ bpart) {
  __shared__ float red[4][64];
  const int cl = threadIdx.x & 63, rl = threadIdx.x >> 6;
  const int c = blockIdx.y * 64 + cl;
  const int r0 = blockIdx.x * rows_per_chunk;
  const int r1 = min(M, r0 + rows_per_chunk);
  float acc = 0.f;
  if (c < n) {
    const float s = scale[c];
    for (int r = r0 + rl; r < r1; r += 4) {
      float g = dy[(size_t)r * ld_dy + coff_dy + c];
      float v = y[(size_t)r * ld_y + coff_y + c];
      g = v > 0.f ? g : 0.f;
      acc += g;
      dz[(size_t)r * ld_dz + coff_dz + c] = g * s;
    }
  }
  red[rl][cl] = acc;
  __syncthreads();
  if (rl == 0 && c < n) bpart[(size_t)blockIdx.x * n + c] = (red[0][cl] + red[1][cl]) + (red[2][cl] + red[3][cl]);
}

// out[c] = sum_chunks part[chunk, c]: 32 columns x 8 chunk lanes per CTA (coalesced 128-byte rows), each lane a
// strided partial sum, then a fixed-order sum of the 8 lanes -> deterministic, ~chunks/8 dependent loads per thread
// instead of `chunks` (592 sequential loads per column took 31 us x 57 launches, profiles/r02f).
__global__ void __launch_bounds__(256)
chunk_sum_kernel(const float* __restrict__ part, int chunks, int n, float* __restrict__ out) {
  __shared__ float red[8][33];
  const int cl = threadIdx.x & 31, rl = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + cl;
  float s = 0.f;
  if (c < n)
    for (int i = rl; i < chunks; i += 8) s += part[(size_t)i * n + c];
  red[rl][cl] = s;
  __syncthreads();
  if (rl == 0 && c < n) {
    float t = red[0][cl];
#pragma unroll
    for (int j = 1; j < 8; ++j) t += red[j][cl];
    out[c] = t;
  }
}

// W [k, k, ci, co] (HWIO) -> Wf [k, k, co, ci] with both spatial axes reversed: the dgrad of a
// stride-1 SAME conv with odd k is the SAME conv of dz with Wf.
__global__ void flip_transpose_kernel(const float* __restrict__ W, float* __restrict__ Wf, int k, int ci, int co) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  int tot = k * k * ci * co;
  if (i >= tot) return;
  int c_i = i % ci;
  int r = i / ci;
  int c_o = r % co;
  int tap = r / co;
  int kh = tap / k, kw = tap % k;
  Wf[i] = W[(((size_t)(k - 1 - kh) * k + (k - 1 - kw)) * ci + c_i) * co + c_o];
}

// dst[r, c] = src[r, coff + c] for c < cols (un-concatenate the grouped 1x1 panel gradient)
__global__ void take_cols_kernel(const float* __restrict__ src, int rows, int ld, int coff, int cols,
                                 float* __restrict__ dst) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < rows * cols) {
    int r = i / cols, c = i - r * cols;
    dst[i] = src[(size_t)r * ld + coff + c];
  }
}

// dW partials: part[z][k, n] = sum_{m in split z} im2col(x)[m, k] * dz[m, n].
// 64 (k) x 64 (n) tile per CTA, 4x4 per thread, 16 pixels per smem stage, register prefetch.
template <int VEC>
__global__ void __launch_bounds__(256, 2)
wgrad_kernel(AConv a, const float* __restrict__ dz, int ld_dz, int M, int N, int K, int m_per_split,
             float* __restrict__ part) {
  constexpr int BMK = 16;
  __shared__ __align__(16) float As[2][BMK][64];
  __shared__ __align__(16) float Bs[2][BMK][64];
  const int tid = threadIdx.x;
  const int n0 = blockIdx.x * 64, k0 = blockIdx.y * 64;
  const int mbeg = blockIdx.z * m_per_split;
  const int mend = min(M, mbeg + m_per_split);
  const int mm = tid >> 4, q = tid & 15;
  const int tx = q, ty = mm;   // output: k rows ty*4.., n cols tx*4..
  float4 ra, rb;
  auto gload = [&](int m0) {
    const int m = m0 + mm;
    RowCtx<1> rc;
    make_row<1>(a, m, mend, rc);
    ra = load_a4<1, VEC>(a, rc, k0 + q * 4, K);
    const int n = n0 + q * 4;
    rb = (m < mend && n < N) ? ldg4(dz + (size_t)m * ld_dz + n) : make_float4(0.f, 0.f, 0.f, 0.f);
  };
  auto sstore = [&](int buf) {
    *reinterpret_cast<float4*>(&As[buf][mm][q * 4]) = ra;
    *reinterpret_cast<float4*>(&Bs[buf][mm][q * 4]) = rb;
  };
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  int buf = 0;
  if (mbeg < mend) {
    gload(mbeg);
    sstore(0);
  }
  __syncthreads();
  for (int m0 = mbeg; m0 < mend; m0 += BMK) {
    const bool more = m0 + BMK < mend;
    if (more) gload(m0 + BMK);
#pragma unroll
    for (int r = 0; r < BMK; ++r) {
      const float4 av = *reinterpret_cast<const float4*>(&As[buf][r][ty * 4]);
      const float4 bv = *reinterpret_cast<const float4*>(&Bs[buf][r][tx * 4]);
      const float a4[4] = {av.x, av.y, av.z, av.w};
      const float b4[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a4[i], b4[j], acc[i][j]);
    }
    if (more) sstore(buf ^ 1);
    __syncthreads();
    buf ^= 1;
  }
  float* dst = part + (size_t)blockIdx.z * K * N;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int k = k0 + ty * 4 + i;
    const int n = n0 + tx * 4;
    if (k < K && n < N)
      *reinterpret_cast<float4*>(dst + (size_t)k * N + n) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
  }
}

// Same contraction with a 128 (k) x 64 (n) output tile, 8 x 4 per thread: 3 shared-memory vector loads per 32 FMAs
// instead of 2 per 16 (the 64 x 64 kernel is shared-memory-load bound: 21 TFLOP/s on Conv2d_2c, profiles/r02f).
template <int VEC>
__global__ void __launch_bounds__(256, 2)
wgrad128_kernel(AConv a, const float* __restrict__ dz, int ld_dz, int M, int N, int K, int m_per_split,
                float* __restrict__ part) {
  constexpr int BMK = 16;
  __shared__ __align__(16) float As[2][BMK][128];
  __shared__ __align__(16) float Bs[2][BMK][64];
  const int tid = threadIdx.x;
  const int n0 = blockIdx.x * 64, k0 = blockIdx.y * 128;
  const int mbeg = blockIdx.z * m_per_split;
  const int mend = min(M, mbeg + m_per_split);
  const int mm = tid >> 4, q = tid & 15;          // loads: row mm of the stage; A k-quads q and q + 16, B n-quad q
  const int tx = tid & 15, ty = tid >> 4;         // outputs: k rows ty*4.. and 64 + ty*4.., n cols tx*4..
  float4 ra0, ra1, rb;
  auto gload = [&](int m0) {
    const int m = m0 + mm;
    RowCtx<1> rc;
    make_row<1>(a, m, mend, rc);
    ra0 = load_a4<1, VEC>(a, rc, k0 + q * 4, K);
    ra1 = load_a4<1, VEC>(a, rc, k0 + 64 + q * 4, K);
    const int n = n0 + q * 4;
    rb = (m < mend && n < N) ? ldg4(dz + (size_t)m * ld_dz + n) : make_float4(0.f, 0.f, 0.f, 0.f);
  };
  auto sstore = [&](int buf) {
    *reinterpret_cast<float4*>(&As[buf][mm][q * 4]) = ra0;
    *reinterpret_cast<float4*>(&As[buf][mm][64 + q * 4]) = ra1;
    *reinterpret_cast<float4*>(&Bs[buf][mm][q * 4]) = rb;
  };
  float acc[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  int buf = 0;
  if (mbeg < mend) {
    gload(mbeg);
    sstore(0);
  }
  __syncthreads();
  for (int m0 = mbeg; m0 < mend; m0 += BMK) {
    const bool more = m0 + BMK < mend;
    if (more) gload(m0 + BMK);
#pragma unroll
    for (int r = 0; r < BMK; ++r) {
      const float4 a0 = *reinterpret_cast<const float4*>(&As[buf][r][ty * 4]);
      const float4 a1 = *reinterpret_cast<const float4*>(&As[buf][r][64 + ty * 4]);
      const float4 bv = *reinterpret_cast<const float4*>(&Bs[buf][r][tx * 4]);
      const float a8[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float b4[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a8[i], b4[j], acc[i][j]);
    }
    if (more) sstore(buf ^ 1);
    __syncthreads();
    buf ^= 1;
  }
  float* dst = part + (size_t)blockIdx.z * K * N;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int k = k0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
    const int n = n0 + tx * 4;
    if (k < K && n < N)
      *reinterpret_cast<float4*>(dst + (size_t)k * N + n) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
  }
}

__global__ void wgrad_reduce_kernel(const float* __restrict__ part, int nz, size_t zstride, float* __restrict__ out,
                                    size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float s = 0.f;
  for (int z = 0; z < nz; ++z) s += part[z * zstride + i];
  out[i] = s;
}

// dx[b,h,w,c] = (add ? add[b,h,w,c] : 0) (+ add2[b,h,w,c]) + sum over the pooling windows that contain (h,w) of
// dy[window] * [x[b,h,w,c] is the FIRST maximum of that window in row-major scan order].
template <int K>
__global__ void __launch_bounds__(256)
maxpool_bwd_kernel(const float* __restrict__ x, const float* __restrict__ dy, const float* add,
                   float* dx, unsigned total, int H, int W, int C4, int stride, int pad_t,
                   int pad_l, int Ho, int Wo, const float* __restrict__ add2) {
  unsigned i = blockIdx.x * 256u + threadIdx.x;
  if (i >= total) return;
  unsigned c4 = i % (unsigned)C4, p = i / (unsigned)C4;
  int w = (int)(p % (unsigned)W);
  unsigned qq = p / (unsigned)W;
  int hh = (int)(qq % (unsigned)H);
  unsigned b = qq / (unsigned)H;
  const float4* xb = reinterpret_cast<const float4*>(x) + (size_t)b * H * W * C4 + c4;
  const float4* dyb = reinterpret_cast<const float4*>(dy) + (size_t)b * Ho * Wo * C4 + c4;
  const float4 xs = __ldg(xb + ((size_t)hh * W + w) * C4);
  float4 g = add ? reinterpret_cast<const float4*>(add)[i] : make_float4(0.f, 0.f, 0.f, 0.f);
  if (add2) {
    const float4 a2 = __ldg(reinterpret_cast<const float4*>(add2) + i);
    g.x += a2.x; g.y += a2.y; g.z += a2.z; g.w += a2.w;
  }
  // windows ho with ho*stride - pad_t <= hh <= ho*stride - pad_t + K - 1
  int ho_lo = hh + pad_t - (K - 1);
  ho_lo = ho_lo <= 0 ? 0 : (ho_lo + stride - 1) / stride;
  int ho_hi = (hh + pad_t) / stride;
  if (ho_hi > Ho - 1) ho_hi = Ho - 1;
  int wo_lo = w + pad_l - (K - 1);
  wo_lo = wo_lo <= 0 ? 0 : (wo_lo + stride - 1) / stride;
  int wo_hi = (w + pad_l) / stride;
  if (wo_hi > Wo - 1) wo_hi = Wo - 1;
  for (int ho = ho_lo; ho <= ho_hi; ++ho) {
    for (int wo = wo_lo; wo <= wo_hi; ++wo) {
      const int h0 = ho * stride - pad_t, w0 = wo * stride - pad_l;
      const int self = (hh - h0) * K + (w - w0);
      bool a0 = true, a1 = true, a2 = true, a3 = true;
#pragma unroll
      for (int dh = 0; dh < K; ++dh) {
#pragma unroll
        for (int dw = 0; dw < K; ++dw) {
          const int hi = h0 + dh, wi = w0 + dw;
          const int pos = dh * K + dw;
          if (pos == self || hi < 0 || hi >= H || wi < 0 || wi >= W) continue;
          const float4 v = __ldg(xb + ((size_t)hi * W + wi) * C4);
          if (pos < self) {
            a0 = a0 && (v.x < xs.x); a1 = a1 && (v.y < xs.y); a2 = a2 && (v.z < xs.z); a3 = a3 && (v.w < xs.w);
          } else {
            a0 = a0 && (v.x <= xs.x); a1 = a1 && (v.y <= xs.y); a2 = a2 && (v.z <= xs.z); a3 = a3 && (v.w <= xs.w);
          }
        }
      }
      const float4 d = __ldg(dyb + ((size_t)ho * Wo + wo) * C4);
      if (a0) g.x += d.x;
      if (a1) g.y += d.y;
      if (a2) g.z += d.z;
      if (a3) g.w += d.w;
    }
  }
  reinterpret_cast<float4*>(dx)[i] = g;
}

// 7x7 VALID average pool backward: dx[b, p, c] = dy[b, c] / HW (+ add[b, p, c]: the attention feature map's gradient when
// Mixed_5c is the end point)
__global__ void avgpool_bwd_kernel(const float* __restrict__ dy, float* __restrict__ dx, int B, int HW, int C,
                                   const float* __restrict__ add) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)B * HW * C) return;
  int c = (int)(i % C);
  int b = (int)(i / ((size_t)HW * C));
  float v = dy[(size_t)b * C + c] / (float)HW;
  if (add) v += add[i];
  dx[i] = v;
}

// ---------------------------------------------------------------------------
// Backward plan.
// ---------------------------------------------------------------------------
constexpr int kBetaChunks = 592;   // 4 x 148 row chunks
constexpr size_t kWPartFloats = (size_t)16 * 1024 * 1024;

struct BwdBufs {
  float *ga, *gb, *dz, *dzg, *dt1, *dt2, *dp, *wflip, *dwg, *wpart, *bpart;
  void* tcws;
  size_t tcws_bytes;
};

static void carve_bwd(Carver& cv, int B, BwdBufs& bb) {
  bb.ga = cv.take<float>((size_t)B * 112 * 112 * 64);
  bb.gb = cv.take<float>((size_t)B * 112 * 112 * 64);
  bb.dz = cv.take<float>((size_t)B * 112 * 112 * 64);
  bb.dzg = cv.take<float>((size_t)B * 28 * 28 * 288);
  bb.dt1 = cv.take<float>((size_t)B * 28 * 28 * 128);
  bb.dt2 = cv.take<float>((size_t)B * 28 * 28 * 32);
  bb.dp = cv.take<float>((size_t)B * 28 * 28 * 256);
  bb.wflip = cv.take<float>((size_t)3 * 3 * 192 * 384 + 1024);
  bb.dwg = cv.take<float>((size_t)832 * 640);
  bb.wpart = cv.take<float>(kWPartFloats);
  bb.bpart = cv.take<float>((size_t)kBetaChunks * 1024);
  // scratch for the tensor-path dgrad weight pack: hi + lo bf16 panels of the largest flipped weight
  bb.tcws_bytes = 2 * (size_t)round_up(832, 16) * round_up(3 * 3 * 384, tc::BK) * sizeof(uint16_t) + 4096;
  bb.tcws = cv.take<char>(bb.tcws_bytes);
}

static int relu_bn_bwd(comic_handle_t h, const float* dy, int ld_dy, int coff_dy, const float* y, int ld_y, int coff_y,
                       int ci, float* dz, int ld_dz, int coff_dz, int M, float* dbeta, BwdBufs& bb, cudaStream_t st) {
  const int n = conv_table()[ci].c_out;
  int chunks = M < kBetaChunks * 8 ? (M + 7) / 8 : kBetaChunks;
  int rpc = (M + chunks - 1) / chunks;
  chunks = (M + rpc - 1) / rpc;
  dim3 g(chunks, (n + 63) / 64);
  relu_bn_bwd_kernel<<<g, 256, 0, st>>>(dy, ld_dy, coff_dy, y, ld_y, coff_y, h->pk.bn_scale[ci], dz, ld_dz, coff_dz, M, n,
                                       rpc, bb.bpart);
  chunk_sum_kernel<<<(n + 31) / 32, 256, 0, st>>>(bb.bpart, chunks, n, dbeta);
  h->launches += 2;
  COMIC_CHECK_CUDA(cudaGetLastError());
  return COMIC_OK;
}

// dW[K, N] = im2col(x)^T . dz  (x: [B,H,W,ldx] NHWC with cin channels; conv k / stride)
static int wgrad(comic_handle_t h, const float* x, int B, int H, int W, int ldx, int cin, int k, int stride,
                 const float* dz, int ld_dz, int N, float* dW, BwdBufs& bb, cudaStream_t st) {
  AConv a;
  a.x = x; a.H = H; a.W = W; a.Cin = cin; a.ldx = ldx; a.KH = k; a.KW = k; a.stride = stride;
  same_pads(H, k, stride, &a.Ho, &a.pad_t);
  same_pads(W, k, stride, &a.Wo, &a.pad_l);
  const int M = B * a.Ho * a.Wo, K = k * k * cin;
  const bool big = K >= 256;                       // 128-row tiles (<= 20 % padding from K = 256 on)
  const int kt = big ? 128 : 64;
  const int tiles = ((K + kt - 1) / kt) * ((N + 63) / 64);
  int nz = (4 * h->num_sms + tiles - 1) / tiles;
  int cap = (int)(kWPartFloats / ((size_t)K * N));
  if (nz > cap) nz = cap;
  if (nz > M / 64) nz = M / 64;
  if (nz < 1) nz = 1;
  int mps = (M + nz - 1) / nz;
  mps = (mps + 15) / 16 * 16;
  nz = (M + mps - 1) / mps;
  dim3 g((N + 63) / 64, (K + kt - 1) / kt, nz);
  float* dst = nz == 1 ? dW : bb.wpart;
  const bool vec = cin % 4 == 0 && ldx % 4 == 0;
  if (big) {
    if (vec) wgrad128_kernel<4><<<g, 256, 0, st>>>(a, dz, ld_dz, M, N, K, mps, dst);
    else wgrad128_kernel<1><<<g, 256, 0, st>>>(a, dz, ld_dz, M, N, K, mps, dst);
  } else {
    if (vec) wgrad_kernel<4><<<g, 256, 0, st>>>(a, dz, ld_dz, M, N, K, mps, dst);
    else wgrad_kernel<1><<<g, 256, 0, st>>>(a, dz, ld_dz, M, N, K, mps, dst);
  }
  h->launches++;
  if (nz > 1) {
    size_t n = (size_t)K * N;
    wgrad_reduce_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(bb.wpart, nz, n, dW, n);
    h->launches++;
  }
  COMIC_CHECK_CUDA(cudaGetLastError());
  return COMIC_OK;
}

// dx[M, N] (row stride ld_dst) = SAME stride-1 conv of dz [B,S,S,cz] with the panel Wp [k*k*cz, N].
static int dgrad_conv(comic_handle_t h, const float* dz, int B, int S, int cz, int k, const float* Wp, int N, float* dst,
                      int ld_dst, BwdBufs& bb, cudaStream_t st) {
  AConv a;
  a.x = dz; a.H = S; a.W = S; a.Cin = cz; a.ldx = cz; a.KH = k; a.KW = k; a.stride = 1;
  same_pads(S, k, 1, &a.Ho, &a.pad_t);
  same_pads(S, k, 1, &a.Wo, &a.pad_l);
  const int M = B * S * S, K = k * k * cz;
  Epi e{};
  e.nroute = 1;
  e.r[0] = Route{0, N, dst, ld_dst, 0};
  e.stop_n = 0x7fffffff;
  cudaError_t err;
  if (h->precision >= 1 && M >= 128) {
    Carver cv(bb.tcws);
    tc::TcWeight tw;
    int rc = pack_tc_weight(h, cv, Wp, K, N, N, cz, cz, tw, st, false);
    if (rc) return rc;
    err = tc::launch_gemm_tc<1>(a, tw, M, N, e, h->num_sms, st);
    h->launches += 2;
  } else {
    GemmPlan p = plan_gemm(M, N, K, h->num_sms, false);
    err = launch_gemm<1, 4>(a, Wp, N, M, N, K, e, p, st);
    h->launches++;
  }
  COMIC_CHECK_CUDA(err);
  return COMIC_OK;
}

static void flip_transpose(comic_handle_t h, const float* W, float* Wf, int k, int ci, int co, cudaStream_t st) {
  int tot = k * k * ci * co;
  flip_transpose_kernel<<<(tot + 255) / 256, 256, 0, st>>>(W, Wf, k, ci, co);
  h->launches++;
}

static int maxpool_bwd(comic_handle_t h, const float* x, const float* dy, const float* add, float* dx, int B, int H,
                       int W, int C, int k, int s, cudaStream_t st, const float* add2 = nullptr) {
  int Ho, Wo, pt, pl;
  same_pads(H, k, s, &Ho, &pt);
  same_pads(W, k, s, &Wo, &pl);
  size_t total = (size_t)B * H * W * (C / 4);
  COMIC_REQUIRE(total < 0xffffffffull && C % 4 == 0 && (k == 2 || k == 3), COMIC_E_UNSUPPORTED,
                "maxpool_bwd: unsupported shape (total %zu, C %d, k %d)", total, C, k);
  unsigned grid = (unsigned)((total + 255) / 256);
  if (k == 3)
    maxpool_bwd_kernel<3><<<grid, 256, 0, st>>>(x, dy, add, dx, (unsigned)total, H, W, C / 4, s, pt, pl, Ho, Wo, add2);
  else maxpool_bwd_kernel<2><<<grid, 256, 0, st>>>(x, dy, add, dx, (unsigned)total, H, W, C / 4, s, pt, pl, Ho, Wo, add2);
  h->launches++;
  COMIC_CHECK_CUDA(cudaGetLastError());
  return COMIC_OK;
}

// One inception block backward.  dy [M, cout] -> dx [M, cin] (+ dx_add [M, cin] when the block input is also the
// attention feature map); weight / beta gradients into g.
static int block_bwd(comic_handle_t h, int bi, const EncTape& tp, const float* dy, float* dx, int B,
                     const comic_cnn_grads_t* g, BwdBufs& bb, cudaStream_t st, const float* dx_add = nullptr) {
  const BlockDesc& bd = block_table()[bi];
  const comic_conv_desc_t* cd = conv_table();
  const int S = kBlkS[bi], M = B * S * S, cout = blk_cout(bd), cin = bd.cin;
  const int ng = bd.b0 + bd.b1a + bd.b2a;
  const float* x = blk_input(tp, bi);
  const float* y = tp.y[bi];
  const int off1 = bd.b0, off2 = bd.b0 + bd.b1b, off3 = bd.b0 + bd.b1b + bd.b2b;
  int rc;
  // Branch_3: maxpool 3x3/1 -> 1x1 conv (conv[5])
  {
    const int ci = bd.conv[5];
    if ((rc = relu_bn_bwd(h, dy, cout, off3, y, cout, off3, ci, bb.dz, bd.b3, 0, M, g->bn_beta[ci], bb, st))) return rc;
    if ((rc = wgrad(h, tp.p[bi], B, S, S, cin, cin, 1, 1, bb.dz, bd.b3, bd.b3, g->conv_w[ci], bb, st))) return rc;
    flip_transpose(h, h->w.conv_w[ci], bb.wflip, 1, cin, bd.b3, st);
    if ((rc = dgrad_conv(h, bb.dz, B, S, bd.b3, 1, bb.wflip, cin, bb.dp, cin, bb, st))) return rc;
  }
  // Branch_2: 1x1 (conv[3]) -> 3x3 (conv[4])
  {
    const int ci = bd.conv[4];
    if ((rc = relu_bn_bwd(h, dy, cout, off2, y, cout, off2, ci, bb.dz, bd.b2b, 0, M, g->bn_beta[ci], bb, st))) return rc;
    if ((rc = wgrad(h, tp.t2[bi], B, S, S, bd.b2a, bd.b2a, cd[ci].k, 1, bb.dz, bd.b2b, bd.b2b, g->conv_w[ci], bb, st)))
      return rc;
    flip_transpose(h, h->w.conv_w[ci], bb.wflip, cd[ci].k, bd.b2a, bd.b2b, st);
    if ((rc = dgrad_conv(h, bb.dz, B, S, bd.b2b, cd[ci].k, bb.wflip, bd.b2a, bb.dt2, bd.b2a, bb, st))) return rc;
  }
  // Branch_1: 1x1 (conv[1]) -> 3x3 (conv[2])
  {
    const int ci = bd.conv[2];
    if ((rc = relu_bn_bwd(h, dy, cout, off1, y, cout, off1, ci, bb.dz, bd.b1b, 0, M, g->bn_beta[ci], bb, st))) return rc;
    if ((rc = wgrad(h, tp.t1[bi], B, S, S, bd.b1a, bd.b1a, cd[ci].k, 1, bb.dz, bd.b1b, bd.b1b, g->conv_w[ci], bb, st)))
      return rc;
    flip_transpose(h, h->w.conv_w[ci], bb.wflip, cd[ci].k, bd.b1a, bd.b1b, st);
    if ((rc = dgrad_conv(h, bb.dz, B, S, bd.b1b, cd[ci].k, bb.wflip, bd.b1a, bb.dt1, bd.b1a, bb, st))) return rc;
  }
  // grouped 1x1: [Branch_0 | Branch_1/0a | Branch_2/0a] read the block input
  {
    const int c0 = bd.conv[0], c1 = bd.conv[1], c3 = bd.conv[3];
    if ((rc = relu_bn_bwd(h, dy, cout, 0, y, cout, 0, c0, bb.dzg, ng, 0, M, g->bn_beta[c0], bb, st))) return rc;
    if ((rc = relu_bn_bwd(h, bb.dt1, bd.b1a, 0, tp.t1[bi], bd.b1a, 0, c1, bb.dzg, ng, bd.b0, M, g->bn_beta[c1], bb, st)))
      return rc;
    if ((rc = relu_bn_bwd(h, bb.dt2, bd.b2a, 0, tp.t2[bi], bd.b2a, 0, c3, bb.dzg, ng, bd.b0 + bd.b1a, M, g->bn_beta[c3],
                          bb, st)))
      return rc;
    if ((rc = wgrad(h, x, B, S, S, cin, cin, 1, 1, bb.dzg, ng, ng, bb.dwg, bb, st))) return rc;
    const int srcs[3] = {c0, c1, c3};
    int coff = 0;
    for (int j = 0; j < 3; ++j) {
      const int n = cd[srcs[j]].c_out;
      take_cols_kernel<<<(cin * n + 255) / 256, 256, 0, st>>>(bb.dwg, cin, ng, coff, n, g->conv_w[srcs[j]]);
      coff += n;
    }
    h->launches += 3;
    if (dx) {
      // dx = dzg . Wg^T, then += dx_add and the maxpool backward of Branch_3's input gradient
      flip_transpose(h, h->pk.grp_w[bi], bb.wflip, 1, cin, ng, st);
      if ((rc = dgrad_conv(h, bb.dzg, B, S, ng, 1, bb.wflip, cin, dx, cin, bb, st))) return rc;
      if ((rc = maxpool_bwd(h, x, bb.dp, dx, dx, B, S, S, cin, 3, 1, st, dx_add))) return rc;
    }
  }
  COMIC_CHECK_CUDA(cudaGetLastError());
  return COMIC_OK;
}

}  // namespace comic

using namespace comic;

extern "C" int comic_encode_train_bytes(comic_handle_t h, int B, size_t* tape_bytes, size_t* ws_bytes) {
  COMIC_REQUIRE(h && tape_bytes && ws_bytes && B > 0, COMIC_E_BADARG, "encode_train_bytes: bad argument");
  {
    Carver cv(nullptr);
    EncTape tp;
    carve_tape(cv, B, tp);
    *tape_bytes = cv.off + 256;
  }
  {
    Carver cv(nullptr);
    BwdBufs bb;
    carve_bwd(cv, B, bb);
    size_t fwd = (size_t)B * 224 * 224 * 4 * sizeof(float) + 1024;   // NHWC4 image for the tensor-path stem conv
    *ws_bytes = (cv.off > fwd ? cv.off : fwd) + 256;
  }
  return COMIC_OK;
}

extern "C" int comic_encode_train_fwd(comic_handle_t h, const float* images, int B, float* fm_out, float* im_embed_out,
                                      void* tape, size_t tape_bytes, void* ws, size_t ws_bytes, void* stream) {
  COMIC_REQUIRE(h && images && fm_out && im_embed_out && tape && ws && B > 0, COMIC_E_BADARG, "encode_train_fwd: bad argument");
  COMIC_REQUIRE(h->cnn_bound, COMIC_E_BADARG, "encode_train_fwd: CNN weights not bound");
  COMIC_REQUIRE(!h->cfg.legacy, COMIC_E_UNSUPPORTED, "encode_train_fwd: the legacy head is not built for cnn_finetune");
  COMIC_REQUIRE(fm_tap_matches(h), COMIC_E_UNSUPPORTED,
                "encode_train_fwd: feature map [%d, %d] is not end point %d's (comic_set_fm_endpoint)", h->M, h->C, h->fm_tap);
  size_t tb, wb;
  comic_encode_train_bytes(h, B, &tb, &wb);
  COMIC_REQUIRE(tape_bytes >= tb && ws_bytes >= wb, COMIC_E_WORKSPACE, "encode_train_fwd: tape %zu < %zu or workspace %zu < %zu",
                tape_bytes, tb, ws_bytes, wb);
  cudaStream_t st = (cudaStream_t)stream;
  Carver cv(tape);
  EncTape tp;
  carve_tape(cv, B, tp);
  int rc;
  // stem (inception_v1.py:70-93)
  if (use_tc(h, h->pk.tc_conv[0], B * 112 * 112)) {
    float* img4 = static_cast<float*>(ws);
    run_pad_c3_c4(h, images, img4, (size_t)B * 224 * 224, st);
    if ((rc = run_conv(h, img4, B, 224, 224, 4, 0, tp.c1, 64, 0, nullptr, nullptr, st))) return rc;
  } else {
    if ((rc = run_conv(h, images, B, 224, 224, 3, 0, tp.c1, 64, 0, nullptr, nullptr, st))) return rc;
  }
  if ((rc = run_maxpool(h, tp.c1, tp.p1, B, 112, 112, 64, 3, 2, nullptr, nullptr, st))) return rc;
  if ((rc = run_conv(h, tp.p1, B, 56, 56, 64, 1, tp.c2b, 64, 0, nullptr, nullptr, st))) return rc;
  if ((rc = run_conv(h, tp.c2b, B, 56, 56, 64, 2, tp.c2c, 192, 0, nullptr, nullptr, st))) return rc;
  if ((rc = run_maxpool(h, tp.c2c, tp.p2, B, 56, 56, 192, 3, 2, nullptr, nullptr, st))) return rc;
  for (int i = 0; i < kNumBlocks; ++i) {
    EncBufs eb{};
    eb.t1 = tp.t1[i]; eb.t2 = tp.t2[i]; eb.p = tp.p[i];
    if ((rc = run_block(h, i, blk_input(tp, i), tp.y[i], B, kBlkS[i], eb, st))) return rc;
    if (i == 1 && (rc = run_maxpool(h, tp.y[1], tp.p3, B, 28, 28, 480, 3, 2, nullptr, nullptr, st))) return rc;
    if (i == 6 && (rc = run_maxpool(h, tp.y[6], tp.p4, B, 14, 14, 832, 2, 2, nullptr, nullptr, st))) return rc;
  }
  COMIC_CHECK_CUDA(cudaMemcpyAsync(fm_out, fm_tap_tensor(tp, h->fm_tap), (size_t)B * h->M * h->C * sizeof(float),
                                   cudaMemcpyDeviceToDevice, st));
  run_avgpool_global(h, tp.y[8], im_embed_out, B, 49, 1024, st);
  COMIC_CHECK_CUDA(cudaGetLastError());
  return COMIC_OK;
}

extern "C" int comic_encode_bwd(comic_handle_t h, const float* images, int B, const float* dfm, const float* dim_embed,
                                const void* tape, size_t tape_bytes, const comic_cnn_grads_t* grads, void* ws,
                                size_t ws_bytes, void* stream) {
  COMIC_REQUIRE(h && images && dfm && dim_embed && tape && grads && ws && B > 0, COMIC_E_BADARG, "encode_bwd: bad argument");
  COMIC_REQUIRE(h->cnn_bound, COMIC_E_BADARG, "encode_bwd: CNN weights not bound");
  COMIC_REQUIRE(fm_tap_matches(h), COMIC_E_UNSUPPORTED,
                "encode_bwd: feature map [%d, %d] is not end point %d's (comic_set_fm_endpoint)", h->M, h->C, h->fm_tap);
  for (int i = 0; i < COMIC_NUM_CONVS; ++i)
    COMIC_REQUIRE(grads->conv_w[i] && grads->bn_beta[i], COMIC_E_BADARG, "encode_bwd: missing gradient buffer %d", i);
  size_t tb, wb;
  comic_encode_train_bytes(h, B, &tb, &wb);
  COMIC_REQUIRE(tape_bytes >= tb && ws_bytes >= wb, COMIC_E_WORKSPACE, "encode_bwd: tape %zu < %zu or workspace %zu < %zu",
                tape_bytes, tb, ws_bytes, wb);
  cudaStream_t st = (cudaStream_t)stream;
  EncTape tp;
  {
    Carver cv(const_cast<void*>(tape));
    carve_tape(cv, B, tp);
  }
  BwdBufs bb;
  {
    Carver cv(ws);
    carve_bwd(cv, B, bb);
  }
  const comic_conv_desc_t* cd = conv_table();
  int rc;
  float *ga = bb.ga, *gb = bb.gb;
  // The end point feeds the next layer AND the attention: dfm is an addend of the kernel that finishes the gradient at
  // the end point (the average pool's backward at Mixed_5c, the 2x2 pool's at Mixed_4f, otherwise the last kernel of the
  // backward of the block the end point feeds).
  const int tap = h->fm_tap;
  auto at = [&](int t) { return t == tap ? dfm : nullptr; };
  // head: im_embed = mean over the 7x7 positions of Mixed_5c (inception_v1.py:326)
  {
    size_t n = (size_t)B * 49 * 1024;
    avgpool_bwd_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(dim_embed, ga, B, 49, 1024, at(COMIC_FM_MIXED_5C));
    h->launches++;
  }
  if ((rc = block_bwd(h, 8, tp, ga, gb, B, grads, bb, st, at(COMIC_FM_MIXED_5B)))) return rc;        // d(Mixed_5b out) in gb
  if ((rc = block_bwd(h, 7, tp, gb, ga, B, grads, bb, st, at(COMIC_FM_MAXPOOL_5A_2X2)))) return rc;  // d(pool4) in ga
  if ((rc = maxpool_bwd(h, tp.y[6], ga, at(COMIC_FM_MIXED_4F), gb, B, 14, 14, 832, 2, 2, st))) return rc;
  if ((rc = block_bwd(h, 6, tp, gb, ga, B, grads, bb, st, at(COMIC_FM_MIXED_4E)))) return rc;
  if ((rc = block_bwd(h, 5, tp, ga, gb, B, grads, bb, st, at(COMIC_FM_MIXED_4D)))) return rc;
  if ((rc = block_bwd(h, 4, tp, gb, ga, B, grads, bb, st, at(COMIC_FM_MIXED_4C)))) return rc;
  if ((rc = block_bwd(h, 3, tp, ga, gb, B, grads, bb, st, at(COMIC_FM_MIXED_4B)))) return rc;
  if ((rc = block_bwd(h, 2, tp, gb, ga, B, grads, bb, st, at(COMIC_FM_MAXPOOL_4A_3X3)))) return rc;  // d(pool3) in ga
  if ((rc = maxpool_bwd(h, tp.y[1], ga, nullptr, gb, B, 28, 28, 480, 3, 2, st))) return rc;
  if ((rc = block_bwd(h, 1, tp, gb, ga, B, grads, bb, st))) return rc;
  if ((rc = block_bwd(h, 0, tp, ga, gb, B, grads, bb, st))) return rc;        // d(pool2) in gb
  // stem
  if ((rc = maxpool_bwd(h, tp.c2c, gb, nullptr, ga, B, 56, 56, 192, 3, 2, st))) return rc;   // d(Conv2d_2c out)
  if ((rc = relu_bn_bwd(h, ga, 192, 0, tp.c2c, 192, 0, 2, bb.dz, 192, 0, B * 56 * 56, grads->bn_beta[2], bb, st))) return rc;
  if ((rc = wgrad(h, tp.c2b, B, 56, 56, 64, 64, 3, 1, bb.dz, 192, 192, grads->conv_w[2], bb, st))) return rc;
  flip_transpose(h, h->w.conv_w[2], bb.wflip, 3, 64, 192, st);
  if ((rc = dgrad_conv(h, bb.dz, B, 56, 192, 3, bb.wflip, 64, gb, 64, bb, st))) return rc;   // d(Conv2d_2b out)
  if ((rc = relu_bn_bwd(h, gb, 64, 0, tp.c2b, 64, 0, 1, bb.dz, 64, 0, B * 56 * 56, grads->bn_beta[1], bb, st))) return rc;
  if ((rc = wgrad(h, tp.p1, B, 56, 56, 64, 64, 1, 1, bb.dz, 64, 64, grads->conv_w[1], bb, st))) return rc;
  flip_transpose(h, h->w.conv_w[1], bb.wflip, 1, 64, 64, st);
  if ((rc = dgrad_conv(h, bb.dz, B, 56, 64, 1, bb.wflip, 64, ga, 64, bb, st))) return rc;    // d(pool1)
  if ((rc = maxpool_bwd(h, tp.c1, ga, nullptr, gb, B, 112, 112, 64, 3, 2, st))) return rc;   // d(Conv2d_1a out)
  if ((rc = relu_bn_bwd(h, gb, 64, 0, tp.c1, 64, 0, 0, bb.dz, 64, 0, B * 112 * 112, grads->bn_beta[0], bb, st))) return rc;
  if ((rc = wgrad(h, images, B, 224, 224, 3, 3, cd[0].k, cd[0].stride, bb.dz, 64, 64, grads->conv_w[0], bb, st))) return rc;
  COMIC_CHECK_CUDA(cudaGetLastError());
  return COMIC_OK;
}

// After the optimiser changed conv kernels / betas in place: folded BN shifts, grouped panels, tensor-path panels.
extern "C" int comic_refresh_packed_cnn(comic_handle_t h, void* packed, size_t packed_bytes, void* stream) {
  COMIC_REQUIRE(h && h->bound && h->cnn_bound && packed, COMIC_E_BADARG, "refresh_packed_cnn: CNN not bound");
  (void)packed_bytes;
  Carver cv(packed);
  int rc = decoder_pack(h, cv, (cudaStream_t)stream, false);
  if (rc) return rc;
  return encoder_pack(h, cv, (cudaStream_t)stream, false);
}
