// gemm_tc.cuh -- persistent tcgen05 (5th-gen tensor core) GEMM / implicit-GEMM
// convolution for sm_100a with fp32-equivalent accuracy: "bf16x3" operand split.
//
//   C[M,N] = A[M,K] . B[K,N]      A, B, C fp32 in HBM
//   A = A_hi + A_lo, B = B_hi + B_lo   (hi = bf16(x), lo = bf16(x - hi): 16 mantissa bits)
//   C ~= A_hi.B_hi + A_lo.B_hi + A_hi.B_lo   (dropped terms ~2^-16 |a||b|)
// accumulated in fp32 in tensor memory with `tcgen05.mma.kind::f16`.  This keeps
// the reference's fp32 numerics (logits / attention maps within 1e-3, SURVEY.md
// §8; measured ~1e-5) at 3 bf16 MMAs per product instead of FFMA.
//
// Persistent CTAs (one per SM) walk a static tile schedule; 448 threads,
// warp-specialised:
//   warps 0-3    epilogue: tcgen05.ld of accumulator buffer (tile & 1) -> folded-BN
//                scale/shift, bias, ReLU -> routed fp32 stores; overlaps the next
//                tile's main loop (TMEM holds two 128 x BN fp32 accumulators).
//   warp 4       TMEM allocator + MMA issuer (one elected lane): 12 UMMAs
//                (128 x n x 16) per 64-wide K block, tcgen05.commit frees the stage.
//   warp 5       TMA producer for the pre-split, pre-transposed weight panels
//                B_hi / B_lo ([Npad, Kpad] bf16 K-major, packed at bind time).
//   warps 6-13   two A-loader groups that alternate K blocks: gather fp32 rows from
//                global (plain segments with row indirection = the beam-search
//                state gather, or NHWC im2col with TF SAME padding), split into
//                hi/lo bf16 in registers and store both tiles to shared memory in
//                the canonical K-major SWIZZLE_128B layout.
// mbarrier ring of STAGES shared-memory stages (full_a / full_b / empty) plus
// tmem_full / tmem_empty for the two accumulator buffers.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "gemm_f32.cuh"

namespace comic {
namespace tc {

constexpr int BM = 128;
constexpr int BK = 64;                      // bf16 elements = one 128-byte swizzle row
constexpr int A_TILE_BYTES = BM * BK * 2;   // 16 KB
constexpr int kEpiWarps = 8;                    // warps w and w + 4 share tensor-memory lane quadrant w & 3 and alternate 16-column chunks
constexpr int kMmaWarp = kEpiWarps;             // also allocates / frees tensor memory
constexpr int kTmaWarp = kEpiWarps + 1;
constexpr int kLoaderGroups = 2;                // must be <= the smallest STAGES: a group may run at most one
                                                // mbarrier phase ahead of the stage it refills (parity aliasing otherwise)
constexpr int kFirstLoaderWarp = kEpiWarps + 2;
constexpr int kThreads = (kFirstLoaderWarp + 4 * kLoaderGroups) * 32;   // 576

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t addr = smem_u32(bar);
  uint32_t done;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
  } while (!done);
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t smem_dst, const CUtensorMap* tm, uint64_t* bar, int c0,
                                            int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// (x, y) -> packed bf16x2 {lo half = bf16(x), hi half = bf16(y)}, round to nearest even.
__device__ __forceinline__ uint32_t pack_bf16x2(float x, float y) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(y), "f"(x));
  return r;
}
// Split four fp32 values into bf16 hi / lo pairs (8 bytes each).
__device__ __forceinline__ void split4(const float4& v, uint2& hi, uint2& lo) {
  hi.x = pack_bf16x2(v.x, v.y);
  hi.y = pack_bf16x2(v.z, v.w);
  float hx = __uint_as_float(hi.x << 16), hy = __uint_as_float(hi.x & 0xffff0000u);
  float hz = __uint_as_float(hi.y << 16), hw = __uint_as_float(hi.y & 0xffff0000u);
  lo.x = pack_bf16x2(v.x - hx, v.y - hy);
  lo.y = pack_bf16x2(v.z - hz, v.w - hw);
}

// K-major SWIZZLE_128B shared-memory operand descriptor (cute::UMMA::SmemDescriptor):
// start>>4 | LBO(1)<<16 | SBO(1024B>>4)<<32 | version 1 <<46 | layout SWIZZLE_128B(2)<<61.
__device__ __forceinline__ uint64_t make_desc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

// cute::UMMA::InstrDescriptor for kind::f16: c_format F32 (1) @4, a/b format BF16 (1)
// @7/@10, K-major A and B, N>>3 @17, M>>4 @24.
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void sts_v2(uint32_t addr, uint32_t a, uint32_t b) {
  asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(addr), "r"(a), "r"(b) : "memory");
}

// One im2col row of the tile (AMODE 1): pointer to channel 0 of the receptive field's top-left
// pixel (it may lie outside the image: only dereferenced for taps whose mask bit is set) and the
// validity of each of the KH*KW taps (TF SAME padding; rows beyond M have mask 0).
struct RowEntry {
  const void* ptr;
  unsigned long long mask;
};

// halo patch of the stem conv (AMODE 3): an 8 x 16 tile of outputs of the 4 x 4 stride-1 conv reads 11 x 19 input
// pixels of 16 channels; per plane 11 * 19 * 32 bytes, hi + lo, double buffered
constexpr int kHaloRows = 11, kHaloCols = 19;
constexpr int kHaloPlaneBytes = ((kHaloRows * kHaloCols * 32 + 127) / 128) * 128;   // 6784
constexpr int kHaloBytes = 2 * 2 * kHaloPlaneBytes;

template <int BN, int STAGES, int NKRES = 0, bool HALO = false>
struct SmemLayout {
  static constexpr int B_TILE_BYTES = BN * BK * 2;                // one weight tile (hi or lo)
  // NKRES > 0: the whole weight panel (<= NKRES K blocks, one N tile) is loaded ONCE per CTA and stays in shared
  // memory; the ring then stages only A (more stages), and the panel is not re-streamed for every M tile
  static constexpr int STAGE_BYTES = 2 * A_TILE_BYTES + (NKRES ? 0 : 2 * B_TILE_BYTES);
  static constexpr int PANEL_OFF = STAGES * STAGE_BYTES;
  static constexpr int TILES_BYTES = PANEL_OFF + NKRES * 2 * B_TILE_BYTES;
  static constexpr int ROWTAB_BYTES = BM * 3 * 8;                 // 3 segment row pointers or RowEntry
  static constexpr int BAR_BYTES = ((3 * STAGES + 4) * 8 + 8 + 15) & ~15;
  static constexpr int EPI_STRIDE = 20;                           // floats per staged row: 16 columns + 4 pad (16-byte rows,
                                                                  // conflict-free 128-bit row writes)
  static constexpr int EPI_BYTES = kEpiWarps * 32 * EPI_STRIDE * 4;   // per-warp 32 x 16 transpose buffer
  static constexpr int HALO_OFF = TILES_BYTES + kLoaderGroups * ROWTAB_BYTES + BAR_BYTES + EPI_BYTES;
  static constexpr int TOTAL = HALO_OFF + (HALO ? kHaloBytes : 0) + 1024;   // + alignment slack
  static constexpr int TMEM_COLS = (2 * BN <= 32) ? 32 : (2 * BN <= 64) ? 64 : (2 * BN <= 128) ? 128 : (2 * BN <= 256) ? 256 : 512;   // two accumulator buffers; allocations are powers of two
};

template <int BN, int STAGES, int AMODE, int NKRES = 0>
__device__ __forceinline__ void gemm_bf16x3_body(const typename AParam<AMODE>::type& a, const CUtensorMap* tm_hi,
                                                 const CUtensorMap* tm_lo, int M, int N, int K, const Epi& epi) {
  static_assert(AMODE != 4 || NKRES == 0, "TMA-staged A: plain kernel only");
  static_assert(AMODE != 3 || (NKRES > 0 && BN == 64), "halo loader: resident-panel stem kernel only");
  using L = SmemLayout<BN, STAGES, NKRES, AMODE == 3>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem = (smem_u32(smem_raw) + 1023u) & ~1023u;      // shared-window address of the tiles
  uint8_t* smem_g = smem_raw + (smem - smem_u32(smem_raw));
  uint8_t* rowtab0 = smem_g + L::TILES_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(rowtab0 + kLoaderGroups * L::ROWTAB_BYTES);
  uint64_t* full_a = bars;
  uint64_t* full_b = bars + STAGES;
  uint64_t* empty = bars + 2 * STAGES;
  uint64_t* tmem_full = bars + 3 * STAGES;        // [2]
  uint64_t* tmem_empty = bars + 3 * STAGES + 2;   // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * STAGES + 4);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int nk = (K + BK - 1) / BK;
  const int n_tiles = (N + BN - 1) / BN;
  const int m_tiles = (M + BM - 1) / BM;          // AMODE 3: M = nimg * 112 * 112 = nimg * 98 tiles of 8 x 16 outputs
  // split-K (launches of one or two M tiles, e.g. the decoder GEMMs at 33..128 rows, where a tile's K loop is a chain of
  // ~1.3 us operand-staging latencies): work item = (K range z, tile mn); the partial sums go to dst + z * split_stride
  // and are added in a fixed order by the consumer
  const int ksplit = (AMODE == 0 && NKRES == 0 && epi.ksplit > 1) ? epi.ksplit : 1;
  const int mn_tiles = m_tiles * n_tiles;
  const int total_tiles = mn_tiles * ksplit;
  const int first_tile = (int)blockIdx.x;
  const int tile_step = (int)gridDim.x;

  // ---- one-time setup ----
  if (tid == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_a[s], AMODE >= 3 ? 256 : 128);
      mbar_init(&full_b[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tmem_full[i], 1);
      mbar_init(&tmem_empty[i], kEpiWarps);
    }
    fence_barrier_init();
  }
  if (warp == kMmaWarp) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"((uint32_t)L::TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const bool stopped = epi.stop != nullptr && *epi.stop >= epi.stop_n;      // uniform over the grid

  if (stopped) {
    // every beam had finished before this step: nothing to compute
  } else if (warp < kEpiWarps) {
    // =====================  epilogue (this CTA's 128 rows)  =====================
    // The accumulator comes out of tensor memory one ROW per lane (32x32b); written like that, a
    // warp store touches 32 different rows (32 sectors per request).  Each 32 x 16 block is therefore
    // passed through a per-warp shared-memory buffer and stored with 4 lanes per row (8 rows x 64
    // contiguous bytes per request).  Folded BN / bias / ReLU are applied after the transpose, where a
    // lane owns 4 fixed columns (their scale / shift are loaded once per block).  Eight epilogue warps:
    // warp w reads lane quadrant w & 3 and the 16-column blocks with parity w >> 2 -- for the short-K
    // layers (1x1 convs: 3-8 K blocks per tile) the epilogue, not the main loop, sets the tile time.
    // Routing: column ranges are multiples of 8, so a 4-column group never straddles two routes.
    const int nr = epi.nroute;
    const int b1 = nr > 1 ? epi.r[1].n0 : 0x7fffffff;
    const int b2 = nr > 2 ? epi.r[2].n0 : 0x7fffffff;
    const int quad = warp & 3, half = warp >> 2;
    float* stage_buf = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(bars) + L::BAR_BYTES) + warp * 32 * L::EPI_STRIDE;
    const uint32_t stage_u32 = smem_u32(stage_buf);
    const int srow = lane >> 2, scol = (lane & 3) * 4;       // store phase: row within a group of 8, first column
    int iter = 0;
    for (int tile = first_tile; tile < total_tiles; tile += tile_step, ++iter) {
      const int kz = tile / mn_tiles, mn = tile - kz * mn_tiles;
      const int m0 = (mn / n_tiles) * BM;
      const int n0 = (mn % n_tiles) * BN;
      const int acc = iter & 1;
      const int n_umma = min(BN, ((N - n0) + 15) & ~15);
      mbar_wait(&tmem_full[acc], (uint32_t)((iter >> 1) & 1));
      tc_fence_after();
      const int mw = m0 + quad * 32;                           // first row of this warp
      // AMODE 3: tile = (image, 8-row band, 16-column band) of the 112 x 112 output map; tile row r = pixel (r >> 4, r & 15)
      const int t_img = AMODE == 3 ? tile / 98 : 0, t_rem = AMODE == 3 ? tile - t_img * 98 : 0;
      const int t_y0 = (t_rem / 7) * 8, t_x0 = (t_rem % 7) * 16;
      auto row_to_m = [&](int row) -> int {
        if constexpr (AMODE == 3) {
          const int r = quad * 32 + row;
          return (t_img * 112 + t_y0 + (r >> 4)) * 112 + t_x0 + (r & 15);
        } else {
          return mw + row;
        }
      };
#pragma unroll 1
      for (int c0 = half * 16; c0 < n_umma; c0 += 32) {
        uint32_t r[16];
        uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * BN + c0);
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, "
            "%14, %15}, [%16];"
            : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
              "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
            : "r"(taddr));
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int g = 0; g < 4; ++g)
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(stage_u32 + (uint32_t)(lane * L::EPI_STRIDE + g * 4) * 4u),
                       "r"(r[g * 4 + 0]), "r"(r[g * 4 + 1]), "r"(r[g * 4 + 2]), "r"(r[g * 4 + 3])
                       : "memory");
        __syncwarp();
        const int n = n0 + c0 + scol;
        if (n < N) {
          const int rt = n >= b2 ? 2 : (n >= b1 ? 1 : 0);
          float* const fdst = epi.r[rt].dst;
          const long long ld = epi.r[rt].ld;
          const long long cofs = (long long)epi.r[rt].coff - epi.r[rt].n0 + n + (long long)kz * epi.split_stride;
          const float4 sc = epi.scale ? ldg4(epi.scale + n) : make_float4(1.f, 1.f, 1.f, 1.f);
          const float4 bs = epi.bias ? ldg4(epi.bias + n) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int row = q * 8 + srow;
            const int m = row_to_m(row);
            if (m < M) {
              float4 v = *reinterpret_cast<const float4*>(stage_buf + row * L::EPI_STRIDE + scol);
              if (epi.scale) { v.x *= sc.x; v.y *= sc.y; v.z *= sc.z; v.w *= sc.w; }
              if (epi.bias) { v.x += bs.x; v.y += bs.y; v.z += bs.z; v.w += bs.w; }
              if (epi.relu) {
                v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f);
              }
              const long long o = (long long)m * ld + cofs;
              *reinterpret_cast<float4*>(fdst + o) = v;
            }
          }
        }
        __syncwarp();
      }
      // accumulator buffer drained -> the MMA warp may overwrite it
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[acc]);
    }
  } else if (warp == kMmaWarp) {
    // =====================  MMA issuer  =====================
    if (lane == 0) {
      int iter = 0;
      uint32_t it = 0;
      if constexpr (NKRES > 0) mbar_wait(&full_b[0], 0);      // resident weight panel landed
      for (int tile = first_tile; tile < total_tiles; tile += tile_step, ++iter) {
        const int kz = tile / mn_tiles, mn = tile - kz * mn_tiles;
        const int kt0 = (int)(((long long)kz * nk) / ksplit), kt1 = (int)(((long long)(kz + 1) * nk) / ksplit);
        const int n0 = (mn % n_tiles) * BN;
        const int acc = iter & 1;
        const int n_umma = min(BN, ((N - n0) + 15) & ~15);
        const uint32_t idesc = make_idesc_bf16(BM, n_umma);
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
        mbar_wait(&tmem_empty[acc], (uint32_t)(((iter >> 1) & 1) ^ 1));
        tc_fence_after();
        for (int kt = kt0; kt < kt1; ++kt, ++it) {
          const int s = it % STAGES;
          const uint32_t ph = (it / STAGES) & 1;
          if constexpr (AMODE != 4) mbar_wait(&full_a[s], ph);      // AMODE 4: A arrives with B on full_b
          if constexpr (NKRES == 0) mbar_wait(&full_b[s], ph);
          tc_fence_after();
          const uint32_t a_hi = smem + s * L::STAGE_BYTES;
          const uint32_t a_lo = a_hi + A_TILE_BYTES;
          const uint32_t b_hi = NKRES ? smem + L::PANEL_OFF + kt * 2 * L::B_TILE_BYTES : a_lo + A_TILE_BYTES;
          const uint32_t b_lo = b_hi + L::B_TILE_BYTES;
          const uint64_t dah = make_desc_sw128(a_hi), dal = make_desc_sw128(a_lo);
          const uint64_t dbh = make_desc_sw128(b_hi), dbl = make_desc_sw128(b_lo);
#pragma unroll
          for (int k16 = 0; k16 < BK / 16; ++k16) {
            const uint64_t adv = (uint64_t)((k16 * 16 * 2) >> 4);    // 32 bytes per K=16 step inside the swizzle row
            const uint32_t first = (kt > kt0 || k16 > 0) ? 1u : 0u;
            umma_bf16(d_tmem, dah + adv, dbh + adv, idesc, first);
            umma_bf16(d_tmem, dal + adv, dbh + adv, idesc, 1u);
            umma_bf16(d_tmem, dah + adv, dbl + adv, idesc, 1u);
          }
          umma_commit(&empty[s]);             // frees the stage when the MMAs above retire
        }
        umma_commit(&tmem_full[acc]);         // accumulator complete -> epilogue
      }
    }
    __syncwarp();
  } else if (warp == kTmaWarp) {
    // =====================  TMA producer (weight tiles)  =====================
    if constexpr (NKRES > 0) {
      if (lane == 0 && first_tile < total_tiles) {
        mbar_arrive_expect_tx(&full_b[0], (uint32_t)nk * 2u * L::B_TILE_BYTES);
        for (int kt = 0; kt < nk; ++kt) {
          const uint32_t b_hi = smem + L::PANEL_OFF + kt * 2 * L::B_TILE_BYTES;
          tma_load_2d(b_hi, tm_hi, &full_b[0], kt * BK, 0);
          tma_load_2d(b_hi + L::B_TILE_BYTES, tm_lo, &full_b[0], kt * BK, 0);
        }
      }
    } else
    if (lane == 0) {
      uint32_t it = 0;
      for (int tile = first_tile; tile < total_tiles; tile += tile_step) {
        const int kz = tile / mn_tiles, mn = tile - kz * mn_tiles;
        const int kt0 = (int)(((long long)kz * nk) / ksplit), kt1 = (int)(((long long)(kz + 1) * nk) / ksplit);
        const int n0 = (mn % n_tiles) * BN;
        for (int kt = kt0; kt < kt1; ++kt, ++it) {
          const int s = it % STAGES;
          const uint32_t ph = (it / STAGES) & 1;
          mbar_wait(&empty[s], ph ^ 1);
          const uint32_t b_hi = smem + s * L::STAGE_BYTES + 2 * A_TILE_BYTES;
          const uint32_t b_lo = b_hi + L::B_TILE_BYTES;
          if constexpr (AMODE == 4) {
            // both operands by TMA: 128 rows of the (hi, lo) A planes + the weight tile, one transaction
            const int m0 = (mn / n_tiles) * BM;
            const uint32_t a_hi = smem + s * L::STAGE_BYTES;
            mbar_arrive_expect_tx(&full_b[s], 2 * L::B_TILE_BYTES + 2 * A_TILE_BYTES);
            tma_load_2d(a_hi, &a.hi, &full_b[s], kt * BK, m0);
            tma_load_2d(a_hi + A_TILE_BYTES, &a.lo, &full_b[s], kt * BK, m0);
            tma_load_2d(b_hi, tm_hi, &full_b[s], kt * BK, n0);
            tma_load_2d(b_lo, tm_lo, &full_b[s], kt * BK, n0);
          } else {
            mbar_arrive_expect_tx(&full_b[s], 2 * L::B_TILE_BYTES);
            tma_load_2d(b_hi, tm_hi, &full_b[s], kt * BK, n0);
            tma_load_2d(b_lo, tm_lo, &full_b[s], kt * BK, n0);
          }
        }
      }
    }
    __syncwarp();
  } else {
    // =====================  A loaders  =====================
    if constexpr (AMODE == 4) {
      // the TMA warp stages A: nothing to do
    } else if constexpr (AMODE == 3) {
      // Stem conv from a shared-memory halo: per tile the 11 x 19 x 16-channel input patch (hi, lo) is fetched
      // ONCE with cp.async (the next tile's patch is in flight while this one is used); K block di (= tap row,
      // 4 taps x 16 channels = 64 contiguous values in the patch row) of output pixel (y, x) is the 128-byte run
      // starting at patch pixel (y + di, x), copied shared -> shared into the swizzled operand tile.
      const int lw = warp - kFirstLoaderWarp;                 // 0..7
      const int tg = lw * 32 + lane;                          // 0..255
      const int c8 = lane & 7, r4 = lane >> 3;
      uint8_t* halo_g = smem_g + L::HALO_OFF;
      const uint32_t halo = smem + L::HALO_OFF;
      auto fetch_halo = [&](int tile, int buf) {
        if (tile < total_tiles) {
          const int img = tile / 98, rem = tile - img * 98;
          const int y0 = (rem / 7) * 8 - 1, x0 = (rem % 7) * 16 - 1;
          // 209 pixels x 2 planes x 2 chunks of 16 bytes
          for (int i = tg; i < kHaloRows * kHaloCols * 4; i += 256) {
            const int plane = i & 1, ch = (i >> 1) & 1, px = i >> 2;
            const int hr = px / kHaloCols, hc = px - hr * kHaloCols;
            const int y = y0 + hr, x = x0 + hc;
            const bool ok = y >= 0 && y < 112 && x >= 0 && x < 112;
            const long long go = ok ? (((long long)img * 112 + y) * 112 + x) * 16 + ch * 8 : 0;
            const uint32_t so = halo + (uint32_t)((buf * 2 + plane) * kHaloPlaneBytes + px * 32 + ch * 16);
            const uint32_t nbytes = ok ? 16u : 0u;
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(so), "l"((plane ? a.lo : a.hi) + go), "r"(nbytes)
                         : "memory");
          }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
      };
      uint32_t it = 0;
      int tcount = 0;
      fetch_halo(first_tile, 0);
      for (int tile = first_tile; tile < total_tiles; tile += tile_step, ++tcount) {
        const int buf = tcount & 1;
        named_bar_sync(1, 256);                               // everyone is done reading buffer buf ^ 1 (previous tile)
        fetch_halo(tile + tile_step, buf ^ 1);
        asm volatile("cp.async.wait_group 1;" ::: "memory");   // this tile's patch (own copies) has landed
        named_bar_sync(1, 256);                               // ... and everyone else's
        const uint8_t* hb = halo_g + (size_t)(buf * 2) * kHaloPlaneBytes;
        for (int kt = 0; kt < nk; ++kt, ++it) {               // kt = tap row di
          const int s = it % STAGES;
          const uint32_t ph = (it / STAGES) & 1;
          const uint32_t a_hi = smem + s * L::STAGE_BYTES;
          mbar_wait(&empty[s], ph ^ 1);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int row = lw * 16 + i * 4 + r4;
            const int src = (((row >> 4) + kt) * kHaloCols + (row & 15)) * 32 + c8 * 16;
            const uint4 vh = *reinterpret_cast<const uint4*>(hb + src);
            const uint4 vl = *reinterpret_cast<const uint4*>(hb + kHaloPlaneBytes + src);
            const uint32_t so = (uint32_t)row * 128u + ((uint32_t)(c8 ^ (row & 7)) << 4);
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a_hi + so), "r"(vh.x), "r"(vh.y), "r"(vh.z), "r"(vh.w)
                         : "memory");
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a_hi + A_TILE_BYTES + so), "r"(vl.x), "r"(vl.y),
                         "r"(vl.z), "r"(vl.w)
                         : "memory");
          }
          fence_proxy_async();
          mbar_arrive(&full_a[s]);
        }
      }
      asm volatile("cp.async.wait_group 0;" ::: "memory");
    } else {
    const int grp = (warp - kFirstLoaderWarp) >> 2;         // loader group
    const int wg = (warp - kFirstLoaderWarp) & 3;           // warp inside the group
    const int tg = wg * 32 + lane;                          // thread inside the group
    uint8_t* rowtab = rowtab0 + grp * L::ROWTAB_BYTES;
    uint32_t it = 0;
    for (int tile = first_tile; tile < total_tiles; tile += tile_step) {
      const int kz = tile / mn_tiles, mn = tile - kz * mn_tiles;
      const int kt0 = (int)(((long long)kz * nk) / ksplit), kt1 = (int)(((long long)(kz + 1) * nk) / ksplit);
      const int m0 = (mn / n_tiles) * BM;
      // per-tile row table (this group's private copy)
      named_bar_sync(1 + grp, 128);
      {
        int m = m0 + tg;
        if constexpr (AMODE == 0) {
          const float** rp = reinterpret_cast<const float**>(rowtab);
#pragma unroll
          for (int s = 0; s < 3; ++s) {
            const float* p = nullptr;
            if (s < a.nseg && m < M) {
              int r = m;
              if (a.seg[s].idx) r = a.seg[s].idx[m];
              if (r >= 0 && r < a.seg[s].idx_limit) p = a.seg[s].ptr + (size_t)r * a.seg[s].ld;
            }
            rp[s * BM + tg] = p;
          }
        } else {   // AMODE 1: im2col row table
          RowEntry* re = reinterpret_cast<RowEntry*>(rowtab);
          RowEntry e;
          e.ptr = nullptr; e.mask = 0ull;
          if (m < M) {
            const int hw = a.Ho * a.Wo;
            const int b = m / hw, rem = m - b * hw;
            const int ho = rem / a.Wo, wo = rem - ho * a.Wo;
            const int hi0 = ho * a.stride - a.pad_t, wi0 = wo * a.stride - a.pad_l;
            e.ptr = a.x + (((long long)b * a.H + hi0) * a.W + wi0) * a.ldx;
            for (int kh = 0; kh < a.KH; ++kh)
              for (int kw = 0; kw < a.KW; ++kw) {
                const int hi = hi0 + kh, wi = wi0 + kw;
                if (hi >= 0 && hi < a.H && wi >= 0 && wi < a.W) e.mask |= 1ull << (kh * a.KW + kw);
              }
          }
          re[tg] = e;
        }
      }
      named_bar_sync(1 + grp, 128);
      for (int kt = kt0; kt < kt1; ++kt, ++it) {
        if ((int)(it % kLoaderGroups) != grp) continue;
        const int s = it % STAGES;
        const uint32_t ph = (it / STAGES) & 1;
        const uint32_t a_hi = smem + s * L::STAGE_BYTES;
        {
          const int chunk = lane & 15;                            // float4 chunk within the 64-float K row
          const int rsub = lane >> 4;                             // 2 rows per warp instruction
          float4 v[16];
          const int kk = kt * BK + chunk * 4;
          if constexpr (AMODE == 0) {
            const float* const* rp = reinterpret_cast<const float* const*>(rowtab);
            int seg = -1, col = kk;
            if (kk < K) {
#pragma unroll
              for (int sg = 0; sg < 3; ++sg) {
                if (seg < 0 && sg < a.nseg) {
                  if (col < a.seg[sg].ncols) seg = sg;
                  else col -= a.seg[sg].ncols;
                }
              }
            }
            const float* const* rps = rp + (seg >= 0 ? seg : 0) * BM + wg * 32 + rsub;
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float* p = (seg >= 0) ? rps[i * 2] : nullptr;
              v[i] = p ? ldg4(p + col) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
          } else {
            const RowEntry* re = reinterpret_cast<const RowEntry*>(rowtab) + wg * 32 + rsub;
            unsigned long long bit = 0ull;
            int tapoff = 0;
            if (kk < K) {
              const int tap = kk / a.Cin, ci = kk - tap * a.Cin;
              const int kh = tap / a.KW, kw = tap - kh * a.KW;
              bit = 1ull << tap;
              tapoff = (kh * a.W + kw) * a.ldx + ci;
            }
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const RowEntry e = re[i * 2];
              v[i] = (e.mask & bit) ? ldg4(static_cast<const float*>(e.ptr) + tapoff) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
          }
          mbar_wait(&empty[s], ph ^ 1);
          // K-major SWIZZLE_128B tile: row r at r*128 bytes, its 16-byte chunk c at ((c ^ (r & 7)) << 4).
          // row = wg*32 + i*2 + rsub: (row & 7) takes 4 values over i, rows 8 apart are 1024 bytes apart
          uint32_t sw[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const uint32_t r7 = (uint32_t)(j * 2 + rsub);
            sw[j] = a_hi + (uint32_t)(wg * 32 + j * 2 + rsub) * 128u + ((((uint32_t)chunk >> 1) ^ r7) << 4) +
                    (((uint32_t)chunk & 1u) << 3);
          }
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            uint2 h, l;
            split4(v[i], h, l);
            const uint32_t dst = sw[i & 3] + (uint32_t)(i >> 2) * 1024u;
            sts_v2(dst, h.x, h.y);
            sts_v2(dst + A_TILE_BYTES, l.x, l.y);
          }
          fence_proxy_async();          // generic-proxy stores -> visible to the tensor core (async proxy)
          mbar_arrive(&full_a[s]);
        }
      }
    }
    }
  }

  // ---- teardown ----
  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)L::TMEM_COLS)
                 : "memory");
}

template <int BN, int STAGES, int AMODE>
__global__ void __launch_bounds__(kThreads, 1)
gemm_bf16x3_kernel(const __grid_constant__ typename AParam<AMODE>::type a, const __grid_constant__ CUtensorMap tm_hi,
                   const __grid_constant__ CUtensorMap tm_lo, int M, int N, int K, const __grid_constant__ Epi epi) {
  gemm_bf16x3_body<BN, STAGES, AMODE>(a, &tm_hi, &tm_lo, M, N, K, epi);
}

// weights resident in shared memory (N <= 64, K <= NKRES * 64): see SmemLayout
template <int STAGES, int NKRES, int AMODE>
__global__ void __launch_bounds__(kThreads, 1)
gemm_bf16x3_bres_kernel(const __grid_constant__ typename AParam<AMODE>::type a, const __grid_constant__ CUtensorMap tm_hi,
                        const __grid_constant__ CUtensorMap tm_lo, int M, int N, int K, const __grid_constant__ Epi epi) {
  gemm_bf16x3_body<64, STAGES, AMODE, NKRES>(a, &tm_hi, &tm_lo, M, N, K, epi);
}

// ---------------------------------------------------------------------------
// Host side.
// ---------------------------------------------------------------------------
// A weight matrix packed for the tensor path: B^T split into bf16 hi / lo, [Npad, Kpad]
// row-major (K-major), zero padded; one tensor map per BN option.
struct TcWeight {
  uint16_t* hi = nullptr;
  uint16_t* lo = nullptr;
  int N = 0, K = 0, Npad = 0, Kpad = 0;   // K = extent of the A operand's K index space
  CUtensorMap tm_hi[5], tm_lo[5];   // BN = 64, 128, 256, 176, 192
  bool ready = false;
};

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

inline bool make_weight_maps(TcWeight& w) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return false;
  const int bns[5] = {64, 128, 256, 176, 192};
  for (int i = 0; i < 5; ++i) {
    cuuint64_t dims[2] = {(cuuint64_t)w.Kpad, (cuuint64_t)w.Npad};
    cuuint64_t strides[1] = {(cuuint64_t)w.Kpad * sizeof(uint16_t)};
    cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)bns[i]};
    cuuint32_t estr[2] = {1, 1};
    CUresult r1 = enc(&w.tm_hi[i], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, w.hi, dims, strides, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    CUresult r2 = enc(&w.tm_lo[i], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, w.lo, dims, strides, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r1 != CUDA_SUCCESS || r2 != CUDA_SUCCESS) return false;
  }
  w.ready = true;
  return true;
}

// B^T bf16 hi/lo packing: src W[k][n] (row stride ldw); optional channel padding of an
// HWIO conv kernel (cin_src -> cin_dst, e.g. 3 -> 4 for the NHWC4 stem input).
static __global__ void pack_bt_kernel(const float* __restrict__ W, int K, int N, int ldw, uint16_t* __restrict__ hi,
                                      uint16_t* __restrict__ lo, int Kpad, int Npad, int cin_src, int cin_dst) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (size_t)Npad * Kpad) return;
  int n = (int)(i / Kpad), kp = (int)(i % Kpad);
  float v = 0.f;
  if (n < N) {
    int k = kp;
    bool ok = kp < K;
    if (cin_src != cin_dst) {
      int tap = kp / cin_dst, ci = kp - tap * cin_dst;
      ok = ci < cin_src && tap < K / cin_src;
      k = tap * cin_src + ci;
    }
    if (ok) v = W[(size_t)k * ldw + n];
  }
  uint32_t h = pack_bf16x2(v, 0.f) & 0xffffu;
  float hf = __uint_as_float(h << 16);
  uint32_t l = pack_bf16x2(v - hf, 0.f) & 0xffffu;
  hi[i] = (uint16_t)h;
  lo[i] = (uint16_t)l;
}

template <int BN, int STAGES, int AMODE>
inline cudaError_t launch_one(const typename AParam<AMODE>::type& a, const TcWeight& w, int bn_idx, int M, int N,
                              const Epi& epi, int num_sms, cudaStream_t st) {
  using L = SmemLayout<BN, STAGES>;
  static PerDeviceOnce once;
  {
    cudaError_t e = once([&] { return cudaFuncSetAttribute(gemm_bf16x3_kernel<BN, STAGES, AMODE>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, L::TOTAL); });
    if (e != cudaSuccess) return e;
  }
  int tiles = ((N + BN - 1) / BN) * ((M + BM - 1) / BM) * ((AMODE == 0 && epi.ksplit > 1) ? epi.ksplit : 1);
  int grid = tiles < num_sms ? tiles : num_sms;
  gemm_bf16x3_kernel<BN, STAGES, AMODE><<<grid, kThreads, L::TOTAL, st>>>(a, w.tm_hi[bn_idx], w.tm_lo[bn_idx], M,
                                                                          N, w.K, epi);
  return cudaGetLastError();
}

// N tile = shared-memory / TMEM allocation; the UMMA N is the exact remainder per tile.
// A launch that cannot fill the SMs with 256-wide tiles takes 128-wide ones when those still fit in one wave
// (e.g. the [logits | query] GEMM at 1,536 rows: 48 -> 84 tiles, each half as long).
// A launch that is less than one wave of 256-wide tiles (the decoder GEMMs at 1,536 rows: 96 and 36 tiles on 148 SMs) is
// tile-quantisation bound -- with three MMAs per operand pair a 128 x 256 x 64 block is 0.83 us of tensor time -- so it takes
// the width that minimises waves x (tile width + fixed cost): 176 for the gate GEMM (12 x 12 = 144 tiles), 64 for
// [logits | query] (144 tiles).  small_ok: the caller's kernel family has the 176 / 64 instantiations.
inline int pick_bn(int M, int N, int num_sms, bool small_ok = false) {
  if (N <= 64) return 64;
  if (N <= 128) return 128;
  const int mt = (M + BM - 1) / BM;
  const int t256 = mt * ((N + 255) / 256), t128 = mt * ((N + 127) / 128);
  if (small_ok && t256 < num_sms) {
    const int cand[4] = {256, 176, 128, 64};
    int best = 256;
    long best_cost = -1;
    for (int i = 0; i < 4; ++i) {
      const int bn = cand[i];
      const int tiles = mt * ((N + bn - 1) / bn);
      const long cost = (long)((tiles + num_sms - 1) / num_sms) * (bn + 48);
      if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = bn; }
    }
    return best;
  }
  if (t256 < num_sms && t128 <= num_sms) return 128;
  return 256;
}

template <int STAGES, int NKRES, int AMODE>
inline cudaError_t launch_bres(const typename AParam<AMODE>::type& a, const TcWeight& w, int M, int N, const Epi& epi,
                               int num_sms, cudaStream_t st) {
  using L = SmemLayout<64, STAGES, NKRES>;
  static_assert(L::TOTAL <= 232448, "resident-panel kernel exceeds the shared memory of an SM");
  static PerDeviceOnce once;
  {
    cudaError_t e = once([&] { return cudaFuncSetAttribute(gemm_bf16x3_bres_kernel<STAGES, NKRES, AMODE>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, L::TOTAL); });
    if (e != cudaSuccess) return e;
  }
  int tiles = (M + BM - 1) / BM;
  int grid = tiles < num_sms ? tiles : num_sms;
  gemm_bf16x3_bres_kernel<STAGES, NKRES, AMODE><<<grid, kThreads, L::TOTAL, st>>>(a, w.tm_hi[0], w.tm_lo[0], M, N, w.K, epi);
  return cudaGetLastError();
}

// Stem conv (AMODE 3): a: space-to-depth planes; w: the W2 panel [64, 256]; output rows M = nimg * 12544.
inline cudaError_t launch_stem_halo(const AHalo& a, const TcWeight& w, const Epi& epi, int num_sms, cudaStream_t st) {
  using L = SmemLayout<64, 3, 4, true>;
  static_assert(L::TOTAL <= 232448, "halo stem kernel exceeds the shared memory of an SM");
  static PerDeviceOnce once;
  {
    cudaError_t e = once([&] { return cudaFuncSetAttribute(gemm_bf16x3_bres_kernel<3, 4, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, L::TOTAL); });
    if (e != cudaSuccess) return e;
  }
  const int tiles = a.nimg * 98;
  const int grid = tiles < num_sms ? tiles : num_sms;
  gemm_bf16x3_bres_kernel<3, 4, 3><<<grid, kThreads, L::TOTAL, st>>>(a, w.tm_hi[0], w.tm_lo[0], a.nimg * 12544, 64, 256, epi);
  return cudaGetLastError();
}

// Tensor maps of a bf16 (hi, lo) A operand [rows, K] (row stride K elements; K % 8 == 0), box = one 128 x 64 A tile.
inline bool make_a_maps(ATma& a, const uint16_t* hi, const uint16_t* lo, int rows, int K) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return false;
  cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)K * sizeof(uint16_t)};
  cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)BM};
  cuuint32_t estr[2] = {1, 1};
  CUresult r1 = enc(&a.hi, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<uint16_t*>(hi), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  CUresult r2 = enc(&a.lo, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<uint16_t*>(lo), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r1 == CUDA_SUCCESS && r2 == CUDA_SUCCESS;
}

template <int AMODE>
inline cudaError_t launch_gemm_tc(const typename AParam<AMODE>::type& a, const TcWeight& w, int M, int N,
                                  const Epi& epi, int num_sms, cudaStream_t st) {
  int bn = pick_bn(M, N, num_sms, AMODE == 0 || AMODE == 4);
  if constexpr (AMODE == 0) {
    if (epi.ksplit > 1) return launch_one<128, 3, 0>(a, w, 1, M, N, epi, num_sms, st);    // tc_ksplit() assumed 128-wide tiles
  }
  if constexpr (AMODE == 0 || AMODE == 4) {
    if (bn == 176) return launch_one<176, 2, AMODE>(a, w, 3, M, N, epi, num_sms, st);
  }
  if constexpr (AMODE == 1) {
    // convolutions a little wider than one 256-column tile (Mixed_4e / 4f 3x3: N = 288 / 320): two tiles of 176 + rest
    // instead of 256 + a 32..64-column tile that pays a full pass over the im2col operand for a sliver of MMA work
    if (N > 256 && N <= 352 && w.K >= 512) return launch_one<176, 2, 1>(a, w, 3, M, N, epi, num_sms, st);
    // 3x3 convolutions with exactly 192 outputs and one 64-channel block per tap (Conv2d_2c): a 192-column tile leaves
    // 40 KB less shared memory allocated, the L1 carve-out grows from 28 to 60 KB and the horizontally neighbouring taps of
    // consecutive K blocks (same pixels shifted by one, 32 KB apart) hit L1 instead of L2
    if (N == 192 && a.KH == 3 && a.Cin == 64) return launch_one<192, 2, 1>(a, w, 4, M, N, epi, num_sms, st);
    // narrow convs (N <= 64): the whole weight panel fits beside the A ring -> load it once per CTA
    if (bn == 64 && (M + BM - 1) / BM >= 2 * num_sms) {
      const int nkb = (w.K + BK - 1) / BK;
      if (nkb <= 4) return launch_bres<4, 4, 1>(a, w, M, N, epi, num_sms, st);
      if (nkb <= 6) return launch_bres<3, 6, 1>(a, w, M, N, epi, num_sms, st);
      if (nkb <= 8) return launch_bres<2, 8, 1>(a, w, M, N, epi, num_sms, st);
    }
  }
  if (bn == 64) return launch_one<64, 4, AMODE>(a, w, 0, M, N, epi, num_sms, st);
  if (bn == 128) return launch_one<128, 3, AMODE>(a, w, 1, M, N, epi, num_sms, st);
  return launch_one<256, 2, AMODE>(a, w, 2, M, N, epi, num_sms, st);
}

}  // namespace tc
}  // namespace comic
