// encoder.cu -- InceptionV1 (GoogLeNet-BN) inference forward for sm_100a.
//
// Replaces the graph built by common/nets/inception_v1.py:29-339 under
// inception_arg_scope (common/nets/inception_utils.py:32-82), called from
// ModelBase._encoder (src/model_base.py:56-104) with is_training=False.
//
// Layout: activations NHWC fp32 in a caller-provided workspace, processed in
// image chunks so a chunk's activations stay L2-resident between layers.
// Every conv is an implicit GEMM (gemm_f32.cuh) whose epilogue applies the
// folded inference BN (scale = rsqrt(var+1e-3), shift = beta - mean*scale; no
// gamma) + ReLU and stores straight into the block's concat output at the
// branch's channel offset.  The three 1x1 convs that read a block's input
// (Branch_0, Branch_1/0a, Branch_2/0a) run as ONE GEMM over a packed
// [Cin, b0+b1a+b2a] weight panel with a 3-way routed epilogue.
#include "comic_internal.cuh"

namespace comic {

static const comic_conv_desc_t kConvs[COMIC_NUM_CONVS] = {
    {7, 2, 3, 64},   {1, 1, 64, 64},  {3, 1, 64, 192},
    // Mixed_3b
    {1, 1, 192, 64}, {1, 1, 192, 96}, {3, 1, 96, 128}, {1, 1, 192, 16}, {3, 1, 16, 32}, {1, 1, 192, 32},
    // Mixed_3c
    {1, 1, 256, 128}, {1, 1, 256, 128}, {3, 1, 128, 192}, {1, 1, 256, 32}, {3, 1, 32, 96}, {1, 1, 256, 64},
    // Mixed_4b
    {1, 1, 480, 192}, {1, 1, 480, 96}, {3, 1, 96, 208}, {1, 1, 480, 16}, {3, 1, 16, 48}, {1, 1, 480, 64},
    // Mixed_4c
    {1, 1, 512, 160}, {1, 1, 512, 112}, {3, 1, 112, 224}, {1, 1, 512, 24}, {3, 1, 24, 64}, {1, 1, 512, 64},
    // Mixed_4d
    {1, 1, 512, 128}, {1, 1, 512, 128}, {3, 1, 128, 256}, {1, 1, 512, 24}, {3, 1, 24, 64}, {1, 1, 512, 64},
    // Mixed_4e
    {1, 1, 512, 112}, {1, 1, 512, 144}, {3, 1, 144, 288}, {1, 1, 512, 32}, {3, 1, 32, 64}, {1, 1, 512, 64},
    // Mixed_4f
    {1, 1, 528, 256}, {1, 1, 528, 160}, {3, 1, 160, 320}, {1, 1, 528, 32}, {3, 1, 32, 128}, {1, 1, 528, 128},
    // Mixed_5b
    {1, 1, 832, 256}, {1, 1, 832, 160}, {3, 1, 160, 320}, {1, 1, 832, 32}, {3, 1, 32, 128}, {1, 1, 832, 128},
    // Mixed_5c
    {1, 1, 832, 384}, {1, 1, 832, 192}, {3, 1, 192, 384}, {1, 1, 832, 48}, {3, 1, 48, 128}, {1, 1, 832, 128},
};

static BlockDesc make_block(int first) {
  BlockDesc b;
  b.cin = kConvs[first].c_in;
  b.b0 = kConvs[first].c_out;
  b.b1a = kConvs[first + 1].c_out;
  b.b1b = kConvs[first + 2].c_out;
  b.b2a = kConvs[first + 3].c_out;
  b.b2b = kConvs[first + 4].c_out;
  b.b3 = kConvs[first + 5].c_out;
  for (int i = 0; i < 6; ++i) b.conv[i] = first + i;
  return b;
}

static BlockDesc kBlocks[kNumBlocks];
static bool kBlocksInit = false;

const BlockDesc* block_table() {
  if (!kBlocksInit) {
    for (int i = 0; i < kNumBlocks; ++i) kBlocks[i] = make_block(3 + 6 * i);
    kBlocksInit = true;
  }
  return kBlocks;
}

const comic_conv_desc_t* conv_table() { return kConvs; }

// --------------------------------------------------------------------------
// Bind-time packing kernels.
// --------------------------------------------------------------------------
__global__ void bn_fold_kernel(const float* __restrict__ beta, const float* __restrict__ mean,
                               const float* __restrict__ var, float* __restrict__ scale,
                               float* __restrict__ shift, int n, float eps) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    float s = 1.0f / sqrtf(var[i] + eps);
    scale[i] = s;
    shift[i] = beta[i] - mean[i] * s;
  }
}

__global__ void copy_cols_kernel(const float* __restrict__ src, int rows, int cols, float* __restrict__ dst,
                                 int ld, int coff) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < rows * cols) {
    int r = i / cols, c = i - r * cols;
    dst[(size_t)r * ld + coff + c] = src[i];
  }
}

__global__ void pack_stem_s2d_kernel(const float* __restrict__ W, uint16_t* __restrict__ hi, uint16_t* __restrict__ lo);

int encoder_pack(comic_handle_t h, Carver& cv, cudaStream_t st, bool dry) {
  const BlockDesc* blk = block_table();
  for (int i = 0; i < COMIC_NUM_CONVS; ++i) {
    h->pk.bn_scale[i] = cv.take<float>(kConvs[i].c_out);
    h->pk.bn_shift[i] = cv.take<float>(kConvs[i].c_out);
  }
  for (int b = 0; b < kNumBlocks; ++b) {
    int ng = blk[b].b0 + blk[b].b1a + blk[b].b2a;
    h->pk.grp_w[b] = cv.take<float>((size_t)blk[b].cin * ng);
    h->pk.grp_scale[b] = cv.take<float>(ng);
    h->pk.grp_shift[b] = cv.take<float>(ng);
  }
  // tensor-path panels: the stem conv reads an NHWC4-padded image (cin 3 -> 4);
  // Branch_0 / Branch_1a / Branch_2a only exist inside the grouped panels.
  for (int i = 0; i < COMIC_NUM_CONVS; ++i) {
    bool grouped = false;
    for (int b = 0; b < kNumBlocks; ++b)
      if (i == blk[b].conv[0] || i == blk[b].conv[1] || i == blk[b].conv[3]) grouped = true;
    if (grouped) continue;
    const comic_conv_desc_t& d = kConvs[i];
    int K = d.k * d.k * d.c_in;
    int cdst = (d.c_in == 3) ? 4 : d.c_in;
    int rc = pack_tc_weight(h, cv, dry ? nullptr : h->w.conv_w[i], K, d.c_out, d.c_out, d.c_in, cdst,
                            h->pk.tc_conv[i], st, dry);
    if (rc) return rc;
  }
  for (int b = 0; b < kNumBlocks; ++b) {
    h->pk.tc_grp[b].hi = cv.take<uint16_t>((size_t)round_up(blk[b].b0 + blk[b].b1a + blk[b].b2a, 16) *
                                        round_up(blk[b].cin, tc::BK));
    h->pk.tc_grp[b].lo = cv.take<uint16_t>((size_t)round_up(blk[b].b0 + blk[b].b1a + blk[b].b2a, 16) *
                                        round_up(blk[b].cin, tc::BK));
  }
  {
    tc::TcWeight& tw = h->pk.tc_stem_s2d;
    tw.N = 64; tw.K = 256; tw.Npad = 64; tw.Kpad = 256;
    tw.hi = cv.take<uint16_t>(64 * 256);
    tw.lo = cv.take<uint16_t>(64 * 256);
    tw.ready = false;
  }
  if (dry) return COMIC_OK;
  pack_stem_s2d_kernel<<<(64 * 256 + 255) / 256, 256, 0, st>>>(h->w.conv_w[0], h->pk.tc_stem_s2d.hi, h->pk.tc_stem_s2d.lo);
  COMIC_REQUIRE(tc::make_weight_maps(h->pk.tc_stem_s2d), COMIC_E_CUDA, "cuTensorMapEncodeTiled failed (stem panel)");
  for (int i = 0; i < COMIC_NUM_CONVS; ++i) {
    int n = kConvs[i].c_out;
    bn_fold_kernel<<<(n + 255) / 256, 256, 0, st>>>(h->w.bn_beta[i], h->w.bn_mean[i], h->w.bn_var[i],
                                                   h->pk.bn_scale[i], h->pk.bn_shift[i], n, 1e-3f);
  }
  for (int b = 0; b < kNumBlocks; ++b) {
    int ng = blk[b].b0 + blk[b].b1a + blk[b].b2a;
    int src_conv[3] = {blk[b].conv[0], blk[b].conv[1], blk[b].conv[3]};
    int coff = 0;
    for (int j = 0; j < 3; ++j) {
      int ci = src_conv[j];
      int n = kConvs[ci].c_out;
      int tot = blk[b].cin * n;
      copy_cols_kernel<<<(tot + 255) / 256, 256, 0, st>>>(h->w.conv_w[ci], blk[b].cin, n, h->pk.grp_w[b], ng, coff);
      copy_cols_kernel<<<(n + 255) / 256, 256, 0, st>>>(h->pk.bn_scale[ci], 1, n, h->pk.grp_scale[b], ng, coff);
      copy_cols_kernel<<<(n + 255) / 256, 256, 0, st>>>(h->pk.bn_shift[ci], 1, n, h->pk.grp_shift[b], ng, coff);
      coff += n;
    }
    // grouped panel for the tensor path (packed from the fp32 grouped panel above)
    tc::TcWeight& tw = h->pk.tc_grp[b];
    tw.N = ng; tw.K = blk[b].cin; tw.Npad = round_up(ng, 16); tw.Kpad = round_up(blk[b].cin, tc::BK);
    size_t n = (size_t)tw.Npad * tw.Kpad;
    tc::pack_bt_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(h->pk.grp_w[b], blk[b].cin, ng, ng, tw.hi, tw.lo,
                                                                   tw.Kpad, tw.Npad, 1, 1);
    COMIC_REQUIRE(tc::make_weight_maps(tw), COMIC_E_CUDA, "cuTensorMapEncodeTiled failed (grouped panel %d)", b);
  }
  COMIC_CHECK_CUDA(cudaGetLastError());
  return COMIC_OK;
}

// NHWC3 -> NHWC4 (zero 4th channel) so the stem conv's im2col rows are 16-byte vectors.
__global__ void pad_c3_c4_kernel(const float* __restrict__ x, float* __restrict__ y, size_t npix) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < npix) {
    float4 v = make_float4(x[i * 3 + 0], x[i * 3 + 1], x[i * 3 + 2], 0.f);
    reinterpret_cast<float4*>(y)[i] = v;
  }
}


// --------------------------------------------------------------------------
// Stem conv as a 4x4 stride-1 conv over the space-to-depth image (tensor path).
// Conv2d_1a_7x7 (stride 2, SAME: pad 2 before / 3 after, common/nets/inception_v1.py:70) reads input row
// 2*ho - 2 + kh = 2*(ho - 1 + (kh >> 1)) + (kh & 1): with X2[n, i, j, (a*2 + b)*3 + c] = x[n, 2i + a, 2j + b, c]
// it is   y[ho, wo] = sum_{di, dj < 4} sum_{ch < 12} X2[ho - 1 + di, wo - 1 + dj, ch] * W2[di, dj, ch]
// with W2[di, dj, (a*2 + b)*3 + c] = W[2di + a, 2dj + b, c] (zero where 2di + a or 2dj + b reaches 7): the same
// products, but 16-channel taps (12 + 4 zero) that the halo loader (gemm_tc.cuh AMODE 3) stages in shared memory
// instead of gathering 49 single-pixel taps per output.  X2 is stored directly as bf16 (hi, lo) planes.
// --------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
s2d_split_kernel(const float* __restrict__ x, uint16_t* __restrict__ hi, uint16_t* __restrict__ lo, size_t npix2) {
  size_t i = (size_t)blockIdx.x * 256 + threadIdx.x;      // (n, i2, j2) over [B, 112, 112]
  if (i >= npix2) return;
  const size_t j2 = i % 112, t = i / 112;
  const size_t i2 = t % 112, n = t / 112;
  const float* r0 = x + ((n * 224 + 2 * i2) * 224 + 2 * j2) * 3;      // x[n, 2i, 2j..2j+1, :] = 6 floats
  const float* r1 = r0 + 224 * 3;
  float v[16];
#pragma unroll
  for (int q = 0; q < 6; ++q) { v[q] = __ldg(r0 + q); v[6 + q] = __ldg(r1 + q); }
  v[12] = v[13] = v[14] = v[15] = 0.f;
  uint2 h[4], l[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) tc::split4(make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]), h[q], l[q]);
  uint4* ph = reinterpret_cast<uint4*>(hi + i * 16);
  uint4* pl = reinterpret_cast<uint4*>(lo + i * 16);
  ph[0] = make_uint4(h[0].x, h[0].y, h[1].x, h[1].y);
  ph[1] = make_uint4(h[2].x, h[2].y, h[3].x, h[3].y);
  pl[0] = make_uint4(l[0].x, l[0].y, l[1].x, l[1].y);
  pl[1] = make_uint4(l[2].x, l[2].y, l[3].x, l[3].y);
}

// W [7,7,3,64] HWIO -> B^T hi/lo panels [64, 256] (K-major) of W2 [4,4,16,64]
__global__ void pack_stem_s2d_kernel(const float* __restrict__ W, uint16_t* __restrict__ hi, uint16_t* __restrict__ lo) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 64 * 256) return;
  const int n = i / 256, kp = i % 256;
  const int di = kp / 64, dj = (kp / 16) % 4, ch = kp % 16;
  float v = 0.f;
  if (ch < 12) {
    const int a = ch / 6, b = (ch / 3) % 2, c = ch % 3;
    const int kh = 2 * di + a, kw = 2 * dj + b;
    if (kh < 7 && kw < 7) v = W[((kh * 7 + kw) * 3 + c) * 64 + n];
  }
  uint32_t h = tc::pack_bf16x2(v, 0.f) & 0xffffu;
  float hf = __uint_as_float(h << 16);
  uint32_t l = tc::pack_bf16x2(v - hf, 0.f) & 0xffffu;
  hi[i] = (uint16_t)h;
  lo[i] = (uint16_t)l;
}

// --------------------------------------------------------------------------
// Pooling kernels (NHWC, 4 channels per thread).
// slim.max_pool2d SAME: window clipped to the image (padding never wins).
// --------------------------------------------------------------------------
template <int K>
__global__ void __launch_bounds__(256)
maxpool_nhwc_kernel(const float* __restrict__ x, float* __restrict__ y, unsigned total, int H, int W, int C4,
                    int stride, int pad_t, int pad_l, int Ho, int Wo) {
  // one thread per (output pixel, 4 channels); all K*K taps are loaded before the max so the
  // loads are in flight together (the kernel is a pure L2/HBM stream)
  unsigned i = blockIdx.x * 256u + threadIdx.x;
  if (i >= total) return;
  unsigned c4 = i % (unsigned)C4, p = i / (unsigned)C4;
  unsigned wo = p % (unsigned)Wo, q = p / (unsigned)Wo;
  unsigned ho = q % (unsigned)Ho, b = q / (unsigned)Ho;
  const int h0 = (int)ho * stride - pad_t, w0 = (int)wo * stride - pad_l;
  const float4* xb = reinterpret_cast<const float4*>(x) + (size_t)b * H * W * C4 + c4;
  float4 v[K * K];
#pragma unroll
  for (int dh = 0; dh < K; ++dh) {
#pragma unroll
    for (int dw = 0; dw < K; ++dw) {
      const int hi = h0 + dh, wi = w0 + dw;
      const bool ok = hi >= 0 && hi < H && wi >= 0 && wi < W;
      v[dh * K + dw] = ok ? __ldg(xb + ((size_t)hi * W + wi) * C4)
                          : make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
    }
  }
  float4 m = v[0];
#pragma unroll
  for (int j = 1; j < K * K; ++j) {
    m.x = fmaxf(m.x, v[j].x); m.y = fmaxf(m.y, v[j].y); m.z = fmaxf(m.z, v[j].z); m.w = fmaxf(m.w, v[j].w);
  }
  reinterpret_cast<float4*>(y)[(size_t)p * C4 + c4] = m;
}


// 3x3 / stride 1 SAME max-pool (the inception blocks' Branch_3): one thread per (image, pair of output rows, 4
// channels) walks along the row keeping the column maxima of the last two columns, so an output costs 2 loads instead
// of 9.  The one-thread-per-output kernel above pulled 1.9x the tensor's bytes through L2 -> SM (14.9 GB per 512-image
// step against 7.9 GB of DRAM traffic, profiles/r01z_launch_summary_batch512.txt) and ran at 3 TB/s.
template <int ROWS>
__global__ void __launch_bounds__(256)
maxpool3s1_rows_kernel(const float* __restrict__ x, float* __restrict__ y, unsigned total, int H, int W, int C4, int HB) {
  const unsigned i = blockIdx.x * 256u + threadIdx.x;
  if (i >= total) return;
  const unsigned c4 = i % (unsigned)C4, q = i / (unsigned)C4;
  const int hb = (int)(q % (unsigned)HB);
  const unsigned b = q / (unsigned)HB;
  const int ho0 = hb * ROWS;
  const float4* xb = reinterpret_cast<const float4*>(x) + (size_t)b * H * W * C4 + c4;
  float4* yb = reinterpret_cast<float4*>(y) + (size_t)b * H * W * C4 + c4;
  const float4 ninf = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
  auto mx = [](const float4& a, const float4& c) {
    return make_float4(fmaxf(a.x, c.x), fmaxf(a.y, c.y), fmaxf(a.z, c.z), fmaxf(a.w, c.w));
  };
  bool ok[ROWS + 2];
#pragma unroll
  for (int j = 0; j < ROWS + 2; ++j) ok[j] = (ho0 - 1 + j) >= 0 && (ho0 - 1 + j) < H;
  float4 p1[ROWS], p2[ROWS];
#pragma unroll
  for (int o = 0; o < ROWS; ++o) { p1[o] = ninf; p2[o] = ninf; }
#pragma unroll 4
  for (int w = 0; w <= W; ++w) {
    float4 cm[ROWS];
    if (w < W) {
      float4 r[ROWS + 2];
#pragma unroll
      for (int j = 0; j < ROWS + 2; ++j)
        r[j] = ok[j] ? __ldg(xb + ((size_t)(ho0 - 1 + j) * W + w) * C4) : ninf;
#pragma unroll
      for (int o = 0; o < ROWS; ++o) cm[o] = mx(mx(r[o], r[o + 1]), r[o + 2]);
    } else {
#pragma unroll
      for (int o = 0; o < ROWS; ++o) cm[o] = ninf;
    }
    if (w >= 1) {
#pragma unroll
      for (int o = 0; o < ROWS; ++o)
        if (ho0 + o < H) yb[((size_t)(ho0 + o) * W + (w - 1)) * C4] = mx(mx(p2[o], p1[o]), cm[o]);
    }
#pragma unroll
    for (int o = 0; o < ROWS; ++o) { p2[o] = p1[o]; p1[o] = cm[o]; }
  }
}


// slim.avg_pool2d(net, [7,7], stride=1) VALID on a 7x7 map -> [B, C]
// (common/nets/inception_v1.py:326).
__global__ void avgpool_global_kernel(const float* __restrict__ x, float* __restrict__ y, int B, int HW, int C) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * C) return;
  int b = i / C, c = i - b * C;
  float s = 0.f;
  for (int p = 0; p < HW; ++p) s += x[((size_t)b * HW + p) * C + c];
  y[i] = s / (float)HW;
}

// Legacy head: LN(1024)+tanh (src/model_base.py:80-85); one CTA per row.
__global__ void ln_tanh_rows_kernel(const float* __restrict__ x, const float* __restrict__ gamma,
                                    const float* __restrict__ beta, float* __restrict__ y, int n, float eps) {
  __shared__ float red[32];
  int row = blockIdx.x;
  const float* xr = x + (size_t)row * n;
  float s = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) s += xr[i];
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  float tot = 0.f;
  for (int i = 0; i < (int)(blockDim.x >> 5); ++i) tot += red[i];
  float mean = tot / n;
  __syncthreads();
  float v = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) { float d = xr[i] - mean; v += d * d; }
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float vt = 0.f;
  for (int i = 0; i < (int)(blockDim.x >> 5); ++i) vt += red[i];
  float rstd = 1.0f / sqrtf(vt / n + eps);
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    float inv = rstd * gamma[i];
    y[(size_t)row * n + i] = tanhf(xr[i] * inv + (beta[i] - mean * inv));
  }
}

// --------------------------------------------------------------------------
// Forward plan.
// --------------------------------------------------------------------------
void same_pads(int n, int k, int s, int* out, int* before) {
  *out = (n + s - 1) / s;
  int pad = (*out - 1) * s + k - n;
  if (pad < 0) pad = 0;
  *before = pad / 2;
}

// The forward runs in three stages with their own image-chunk sizes: the stem (huge
// activations: 3.2 MB / image after Conv2d_1a) in small chunks, the 28x28 blocks in medium
// ones and the 14x14 / 7x7 blocks in large ones, so that every launch has several waves of
// 128-row tiles on the 148 SMs (a 64-image chunk gives a 14x14 layer 98 tiles: < 1 wave).
// Stage outputs (pool2 [B,28,28,192], pool3 [B,14,14,480]) are whole-batch buffers.
struct EncPlan {
  int cs, c3, c4;
  size_t ab, t1, t2, p, p2, p3, head;   // floats
};

static EncPlan enc_plan(comic_handle_t h, int B) {
  EncPlan pl;
  pl.cs = B < h->enc_chunk[0] ? B : h->enc_chunk[0];
  pl.c3 = B < h->enc_chunk[1] ? B : h->enc_chunk[1];
  pl.c4 = B < h->enc_chunk[2] ? B : h->enc_chunk[2];
  auto mx = [](size_t x, size_t y) { return x > y ? x : y; };
  // ping/pong: stem conv1 112x112x64 / conv2c 56x56x192; stage 3 28x28x480; stage 4 14x14x528 (832 goes to fm_out)
  pl.ab = mx(mx((size_t)pl.cs * 112 * 112 * 64, (size_t)pl.c3 * 28 * 28 * 480), (size_t)pl.c4 * 14 * 14 * 832);
  pl.t1 = mx((size_t)pl.c3 * 28 * 28 * 128, (size_t)pl.c4 * 14 * 14 * 192);
  pl.t2 = mx((size_t)pl.c3 * 28 * 28 * 32, (size_t)pl.c4 * 14 * 14 * 48);
  pl.p = mx((size_t)pl.c3 * 28 * 28 * 256, (size_t)pl.c4 * 14 * 14 * 832);
  pl.p2 = (size_t)B * 28 * 28 * 192;
  pl.p3 = (size_t)B * 14 * 14 * 480;
  pl.head = (size_t)pl.c4 * 1024;
  return pl;
}

int encoder_workspace_bytes(comic_handle_t h, int B, size_t* bytes) {
  EncPlan pl = enc_plan(h, B);
  Carver cv(nullptr);
  cv.take<float>(pl.ab); cv.take<float>(pl.ab); cv.take<float>(pl.t1); cv.take<float>(pl.t2); cv.take<float>(pl.p);
  cv.take<float>(pl.p2); cv.take<float>(pl.p3); cv.take<float>(pl.head);
  *bytes = cv.off;
  return COMIC_OK;
}

int run_conv(comic_handle_t h, const float* x, int B, int H, int W, int ldx, int ci, float* dst,
                    int ld_dst, int coff, int* Ho_out, int* Wo_out, cudaStream_t st) {
  const comic_conv_desc_t& d = kConvs[ci];
  AConv a;
  a.x = x; a.H = H; a.W = W; a.Cin = (d.c_in == 3 && ldx == 4) ? 4 : d.c_in; a.ldx = ldx;
  a.KH = d.k; a.KW = d.k; a.stride = d.stride;
  same_pads(H, d.k, d.stride, &a.Ho, &a.pad_t);
  same_pads(W, d.k, d.stride, &a.Wo, &a.pad_l);
  int M = B * a.Ho * a.Wo, N = d.c_out, K = d.k * d.k * d.c_in;
  Epi e{};
  e.bias = h->pk.bn_shift[ci];
  e.scale = h->pk.bn_scale[ci];
  e.relu = 1;
  e.nroute = 1;
  e.r[0] = Route{0, N, dst, ld_dst, coff};
  e.split_stride = 0;
  GemmPlan p = plan_gemm(M, N, K, h->num_sms, false);
  cudaError_t err;
  if (use_tc(h, h->pk.tc_conv[ci], M) && a.Cin % 4 == 0) {
    Prof pf(h, T_CONV, st);
    err = tc::launch_gemm_tc<1>(a, h->pk.tc_conv[ci], M, N, e, h->num_sms, st);
  } else {
    Prof pf(h, T_CONV, st);
    if (d.c_in % 4 == 0) err = launch_gemm<1, 4>(a, h->w.conv_w[ci], N, M, N, K, e, p, st);
    else err = launch_gemm<1, 1>(a, h->w.conv_w[ci], N, M, N, K, e, p, st);
  }
  COMIC_CHECK_CUDA(err);
  if (Ho_out) *Ho_out = a.Ho;
  if (Wo_out) *Wo_out = a.Wo;
  return COMIC_OK;
}

int run_maxpool(comic_handle_t h, const float* x, float* y, int B, int H, int W, int C, int k, int s,
                       int* Ho_out, int* Wo_out, cudaStream_t st) {
  int Ho, Wo, pt, pl;
  same_pads(H, k, s, &Ho, &pt);
  same_pads(W, k, s, &Wo, &pl);
  size_t total = (size_t)B * Ho * Wo * (C / 4);
  COMIC_REQUIRE(total < 0xffffffffull && C % 4 == 0 && (k == 2 || k == 3), COMIC_E_UNSUPPORTED,
                "maxpool: unsupported shape (total %zu, C %d, k %d)", total, C, k);
  unsigned grid = (unsigned)((total + 255) / 256);
  {
    Prof pf(h, T_POOL, st);
    if (k == 3 && s == 1) {
      const int HB = (H + 1) / 2;
      const size_t tot = (size_t)B * HB * (C / 4);
      maxpool3s1_rows_kernel<2><<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(x, y, (unsigned)tot, H, W, C / 4, HB);
    } else if (k == 3)
      maxpool_nhwc_kernel<3><<<grid, 256, 0, st>>>(x, y, (unsigned)total, H, W, C / 4, s, pt, pl, Ho, Wo);
    else
      maxpool_nhwc_kernel<2><<<grid, 256, 0, st>>>(x, y, (unsigned)total, H, W, C / 4, s, pt, pl, Ho, Wo);
  }
  COMIC_CHECK_CUDA(cudaGetLastError());
  if (Ho_out) *Ho_out = Ho;
  if (Wo_out) *Wo_out = Wo;
  return COMIC_OK;
}

void run_pad_c3_c4(comic_handle_t h, const float* img, float* dst, size_t npix, cudaStream_t st) {
  Prof pf(h, T_POOL, st);
  pad_c3_c4_kernel<<<(unsigned)((npix + 255) / 256), 256, 0, st>>>(img, dst, npix);
}

void run_avgpool_global(comic_handle_t h, const float* x, float* y, int B, int HW, int C, cudaStream_t st) {
  Prof pf(h, T_POOL, st);
  avgpool_global_kernel<<<(B * C + 255) / 256, 256, 0, st>>>(x, y, B, HW, C);
}

// One inception block: x [B,S,S,cin] -> y [B,S,S,cout].
int run_block(comic_handle_t h, int bi, const float* x, float* y, int B, int S, EncBufs& eb,
                     cudaStream_t st) {
  const BlockDesc& bd = block_table()[bi];
  int cout = bd.b0 + bd.b1b + bd.b2b + bd.b3;
  int M = B * S * S;
  // grouped 1x1: [b0 | b1a | b2a]
  {
    APlain a{};
    a.nseg = 1;
    a.seg[0] = ASeg{x, nullptr, bd.cin, bd.cin, M};
    int ng = bd.b0 + bd.b1a + bd.b2a;
    Epi e{};
    e.bias = h->pk.grp_shift[bi];
    e.scale = h->pk.grp_scale[bi];
    e.relu = 1;
    e.nroute = 3;
    e.r[0] = Route{0, bd.b0, y, cout, 0};
    e.r[1] = Route{bd.b0, bd.b0 + bd.b1a, eb.t1, bd.b1a, 0};
    e.r[2] = Route{bd.b0 + bd.b1a, ng, eb.t2, bd.b2a, 0};
    GemmPlan p = plan_gemm(M, ng, bd.cin, h->num_sms, false);
    cudaError_t err;
    {
      Prof pf(h, T_CONV, st);
      if (use_tc(h, h->pk.tc_grp[bi], M)) err = tc::launch_gemm_tc<0>(a, h->pk.tc_grp[bi], M, ng, e, h->num_sms, st);
      else err = launch_gemm<0, 4>(a, h->pk.grp_w[bi], ng, M, ng, bd.cin, e, p, st);
    }
    COMIC_CHECK_CUDA(err);
  }
  int rc;
  if ((rc = run_conv(h, eb.t1, B, S, S, bd.b1a, bd.conv[2], y, cout, bd.b0, nullptr, nullptr, st))) return rc;
  if ((rc = run_conv(h, eb.t2, B, S, S, bd.b2a, bd.conv[4], y, cout, bd.b0 + bd.b1b, nullptr, nullptr, st))) return rc;
  if ((rc = run_maxpool(h, x, eb.p, B, S, S, bd.cin, 3, 1, nullptr, nullptr, st))) return rc;
  if ((rc = run_conv(h, eb.p, B, S, S, bd.cin, bd.conv[5], y, cout, bd.b0 + bd.b1b + bd.b2b, nullptr, nullptr, st))) return rc;
  return COMIC_OK;
}


// Stem conv on the tensor path through the space-to-depth planes (see s2d_split_kernel): images [nb,224,224,3]
// -> Conv2d_1a_7x7 output dst [nb,112,112,64].  `scratch` holds the X2 planes: 2 * nb*112*112*16 bf16.
static int run_stem_s2d(comic_handle_t h, const float* img, int nb, float* scratch, float* dst, cudaStream_t st) {
  const size_t npix2 = (size_t)nb * 112 * 112;
  uint16_t* xh = reinterpret_cast<uint16_t*>(scratch);
  uint16_t* xl = xh + npix2 * 16;
  {
    Prof pf(h, T_POOL, st);
    s2d_split_kernel<<<(unsigned)((npix2 + 255) / 256), 256, 0, st>>>(img, xh, xl, npix2);
  }
  AHalo a;
  a.hi = xh; a.lo = xl; a.nimg = nb;
  Epi e{};
  e.bias = h->pk.bn_shift[0]; e.scale = h->pk.bn_scale[0]; e.relu = 1; e.nroute = 1;
  e.r[0] = Route{0, 64, dst, 64, 0};
  cudaError_t err;
  {
    Prof pf(h, T_CONV, st);
    err = tc::launch_stem_halo(a, h->pk.tc_stem_s2d, e, h->num_sms, st);
  }
  COMIC_CHECK_CUDA(err);
  return COMIC_OK;
}

int encoder_forward(comic_handle_t h, const float* images, int B, float* fm_out, float* im_embed_out,
                    float* mixed5c_out, void* ws, size_t ws_bytes, cudaStream_t st) {
  COMIC_REQUIRE(h->cnn_bound, COMIC_E_BADARG, "encode_fwd: CNN weights not bound");
  COMIC_REQUIRE(h->C == 832, COMIC_E_UNSUPPORTED, "encode_fwd: only cnn_fm_attention=Mixed_4f (C=832) is built");
  size_t need;
  encoder_workspace_bytes(h, B, &need);
  COMIC_REQUIRE(ws_bytes >= need, COMIC_E_WORKSPACE, "encode_fwd: workspace %zu < %zu", ws_bytes, need);
  const EncPlan pl = enc_plan(h, B);
  Carver cv(ws);
  EncBufs eb;
  eb.a = cv.take<float>(pl.ab); eb.b = cv.take<float>(pl.ab);
  eb.t1 = cv.take<float>(pl.t1); eb.t2 = cv.take<float>(pl.t2); eb.p = cv.take<float>(pl.p);
  float* pool2 = cv.take<float>(pl.p2);
  float* pool3 = cv.take<float>(pl.p3);
  float* head = cv.take<float>(pl.head);
  int rc;
  // ---- stem (inception_v1.py:70-93) -> pool2 [B,28,28,192]
  for (int b0 = 0; b0 < B; b0 += pl.cs) {
    int nb = (B - b0 < pl.cs) ? (B - b0) : pl.cs;
    const float* img = images + (size_t)b0 * 224 * 224 * 3;
    int Ho, Wo;
    if (use_tc(h, h->pk.tc_stem_s2d, nb * 112 * 112) && h->stem_s2d) {
      if ((rc = run_stem_s2d(h, img, nb, eb.b, eb.a, st))) return rc;
    } else if (use_tc(h, h->pk.tc_conv[0], nb * 112 * 112)) {
      size_t npix = (size_t)nb * 224 * 224;
      {
        Prof pf(h, T_POOL, st);
        pad_c3_c4_kernel<<<(unsigned)((npix + 255) / 256), 256, 0, st>>>(img, eb.b, npix);
      }
      if ((rc = run_conv(h, eb.b, nb, 224, 224, 4, 0, eb.a, 64, 0, &Ho, &Wo, st))) return rc;
    } else {
      if ((rc = run_conv(h, img, nb, 224, 224, 3, 0, eb.a, 64, 0, &Ho, &Wo, st))) return rc;    // 112x112x64
    }
    if ((rc = run_maxpool(h, eb.a, eb.b, nb, 112, 112, 64, 3, 2, &Ho, &Wo, st))) return rc;     // 56x56x64
    if ((rc = run_conv(h, eb.b, nb, 56, 56, 64, 1, eb.a, 64, 0, nullptr, nullptr, st))) return rc;
    if ((rc = run_conv(h, eb.a, nb, 56, 56, 64, 2, eb.b, 192, 0, nullptr, nullptr, st))) return rc;  // 56x56x192
    if ((rc = run_maxpool(h, eb.b, pool2 + (size_t)b0 * 28 * 28 * 192, nb, 56, 56, 192, 3, 2, nullptr, nullptr, st)))
      return rc;                                                                                // 28x28x192
  }
  // ---- Mixed_3b, 3c @28 -> pool3 [B,14,14,480]
  for (int b0 = 0; b0 < B; b0 += pl.c3) {
    int nb = (B - b0 < pl.c3) ? (B - b0) : pl.c3;
    if ((rc = run_block(h, 0, pool2 + (size_t)b0 * 28 * 28 * 192, eb.b, nb, 28, eb, st))) return rc;   // 256
    if ((rc = run_block(h, 1, eb.b, eb.a, nb, 28, eb, st))) return rc;                                   // 480
    if ((rc = run_maxpool(h, eb.a, pool3 + (size_t)b0 * 14 * 14 * 480, nb, 28, 28, 480, 3, 2, nullptr, nullptr, st)))
      return rc;                                                                                         // 14x14x480
  }
  // ---- Mixed_4b..4f @14, Mixed_5b, 5c @7, head
  for (int b0 = 0; b0 < B; b0 += pl.c4) {
    int nb = (B - b0 < pl.c4) ? (B - b0) : pl.c4;
    if ((rc = run_block(h, 2, pool3 + (size_t)b0 * 14 * 14 * 480, eb.a, nb, 14, eb, st))) return rc;   // 512
    if ((rc = run_block(h, 3, eb.a, eb.b, nb, 14, eb, st))) return rc;   // 512
    if ((rc = run_block(h, 4, eb.b, eb.a, nb, 14, eb, st))) return rc;   // 512
    if ((rc = run_block(h, 5, eb.a, eb.b, nb, 14, eb, st))) return rc;   // 528
    // Mixed_4f -> the attention feature map, written straight to fm_out [B,196,832]
    float* fm = fm_out + (size_t)b0 * 196 * 832;
    if ((rc = run_block(h, 6, eb.b, fm, nb, 14, eb, st))) return rc;
    if ((rc = run_maxpool(h, fm, eb.a, nb, 14, 14, 832, 2, 2, nullptr, nullptr, st))) return rc;    // 7x7x832
    if ((rc = run_block(h, 7, eb.a, eb.b, nb, 7, eb, st))) return rc;    // 832
    float* m5c = mixed5c_out ? mixed5c_out + (size_t)b0 * 49 * 1024 : eb.a;
    if ((rc = run_block(h, 8, eb.b, m5c, nb, 7, eb, st))) return rc;     // 1024
    float* emb = im_embed_out + (size_t)b0 * 1024;
    if (!h->cfg.legacy) {
      Prof pf(h, T_POOL, st);
      avgpool_global_kernel<<<(nb * 1024 + 255) / 256, 256, 0, st>>>(m5c, emb, nb, 49, 1024);
    } else {
      avgpool_global_kernel<<<(nb * 1024 + 255) / 256, 256, 0, st>>>(m5c, head, nb, 49, 1024);
      ln_tanh_rows_kernel<<<nb, 256, 0, st>>>(head, h->w.enc_ln_gamma, h->w.enc_ln_beta, eb.t1, 1024, 1e-12f);
      h->launches += 2;
      APlain a{};
      a.nseg = 1;
      a.seg[0] = ASeg{eb.t1, nullptr, 1024, 1024, nb};
      Epi e{};
      e.nroute = 1;
      e.r[0] = Route{0, 1024, emb, 1024, 0};
      GemmPlan p = plan_gemm(nb, 1024, 1024, h->num_sms, false);
      cudaError_t err;
      {
        Prof pf(h, T_MISC, st);
        err = launch_gemm<0, 4>(a, h->w.enc_embed_weight, 1024, nb, 1024, 1024, e, p, st);
      }
      COMIC_CHECK_CUDA(err);
    }
    COMIC_CHECK_CUDA(cudaGetLastError());
  }
  return COMIC_OK;
}

}  // namespace comic

// ---------------------------------------------------------------------------
// Evaluation pre-processing of common/inputs/preprocessing/inception_preprocessing_radix.py:
// convert_image_dtype(uint8 -> float32) (:271), resize_bilinear to 256 x 256 with TF r1.9's
// align_corners=False rule (source = destination * in / out, no half-pixel offset) (:272),
// resize_image_with_crop_or_pad to out_h x out_w (:230) and (x - 0.5) * 2 (:234-235), fused: only the
// cropped pixels are interpolated, one thread per output pixel (3 channels), uint8 in / fp32 NHWC out.
// ---------------------------------------------------------------------------
namespace comic {
// crop_yx == nullptr: evaluation (central crop / zero pad).  Otherwise training (preprocess_for_train,
// inception_preprocessing_radix.py:158-201): per image an optional left-right flip of the resized RS x RS image
// (flip[b] != 0) followed by the crop whose top-left corner is crop_yx[b] = (y0, x0); the random draws themselves are
// the caller's (TF's random streams cannot be reproduced).
__global__ void __launch_bounds__(256)
preprocess_eval_kernel(const uint8_t* __restrict__ img, int B, int H, int W, int RS, int out_h, int out_w,
                       float* __restrict__ out, const int* __restrict__ crop_yx = nullptr,
                       const uint8_t* __restrict__ flip = nullptr) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)B * out_h * out_w) return;
  const int x = (int)(i % out_w), y = (int)((i / out_w) % out_h), b = (int)(i / ((size_t)out_w * out_h));
  // crop_or_pad: crop offset = (RS - out) / 2 when out < RS, pad offset = (out - RS) / 2 otherwise
  int ry = (out_h <= RS) ? y + (RS - out_h) / 2 : y - (out_h - RS) / 2;
  int rx = (out_w <= RS) ? x + (RS - out_w) / 2 : x - (out_w - RS) / 2;
  if (crop_yx != nullptr) {
    ry = y + crop_yx[2 * b];
    rx = x + crop_yx[2 * b + 1];
    if (flip != nullptr && flip[b]) rx = RS - 1 - rx;           // the crop is taken from the flipped image
  }
  float v[3] = {0.f, 0.f, 0.f};                       // padding is 0 BEFORE the standardisation
  if (ry >= 0 && ry < RS && rx >= 0 && rx < RS) {
    const float sy = (float)H / (float)RS, sx = (float)W / (float)RS;
    const float fy = __fmul_rn((float)ry, sy), fx = __fmul_rn((float)rx, sx);
    const int y0 = (int)floorf(fy), x0 = (int)floorf(fx);
    const int y1 = min(y0 + 1, H - 1), x1 = min(x0 + 1, W - 1);
    const float ly = __fsub_rn(fy, (float)y0), lx = __fsub_rn(fx, (float)x0);
    const uint8_t* p = img + (size_t)b * H * W * 3;
    const float k = 1.0f / 255.0f;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float tl = (float)p[((size_t)y0 * W + x0) * 3 + c] * k, tr = (float)p[((size_t)y0 * W + x1) * 3 + c] * k;
      const float bl = (float)p[((size_t)y1 * W + x0) * 3 + c] * k, br = (float)p[((size_t)y1 * W + x1) * 3 + c] * k;
      // separate multiply and add (no FMA contraction): bit-identical to TF's / the oracle's lerp
      const float top = __fadd_rn(tl, __fmul_rn(__fsub_rn(tr, tl), lx)), bot = __fadd_rn(bl, __fmul_rn(__fsub_rn(br, bl), lx));
      v[c] = __fadd_rn(top, __fmul_rn(__fsub_rn(bot, top), ly));
    }
  }
  float* o = out + i * 3;
#pragma unroll
  for (int c = 0; c < 3; ++c) o[c] = __fmul_rn(__fsub_rn(v[c], 0.5f), 2.0f);
}
}  // namespace comic

extern "C" int comic_preprocess_eval(comic_handle_t h, const uint8_t* images, int B, int H, int W, int out_h,
                                     int out_w, float* out, void* stream) {
  COMIC_REQUIRE(h && images && out, COMIC_E_BADARG, "preprocess_eval: null argument");
  COMIC_REQUIRE(B > 0 && H > 0 && W > 0 && out_h > 0 && out_w > 0, COMIC_E_SHAPE,
                "preprocess_eval: bad shape B=%d H=%d W=%d out=%dx%d", B, H, W, out_h, out_w);
  const size_t n = (size_t)B * out_h * out_w;
  comic::preprocess_eval_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(images, B, H, W, 256,
                                                                                            out_h, out_w, out);
  h->launches++;
  COMIC_CHECK_CUDA(cudaGetLastError());
  return COMIC_OK;
}

extern "C" int comic_preprocess_train(comic_handle_t h, const uint8_t* images, int B, int H, int W, int out_h, int out_w,
                                      const int32_t* crop_yx, const uint8_t* flip, float* out, void* stream) {
  COMIC_REQUIRE(h && images && out && crop_yx, COMIC_E_BADARG, "preprocess_train: null argument");
  COMIC_REQUIRE(B > 0 && H > 0 && W > 0 && out_h > 0 && out_w > 0 && out_h <= 256 && out_w <= 256, COMIC_E_SHAPE,
                "preprocess_train: bad shape B=%d H=%d W=%d out=%dx%d (tf.random_crop needs out <= 256)", B, H, W, out_h,
                out_w);
  const size_t n = (size_t)B * out_h * out_w;
  comic::preprocess_eval_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(images, B, H, W, 256,
                                                                                            out_h, out_w, out, crop_yx, flip);
  h->launches++;
  COMIC_CHECK_CUDA(cudaGetLastError());
  return COMIC_OK;
}

extern "C" const comic_conv_desc_t* comic_conv_table(void) { return comic::conv_table(); }
