// api.cu -- handle lifecycle, weight binding and the remaining C-ABI entry
// points of libcomic_b200.so (see include/comic_b200.h).
#include <stdarg.h>
#include <string.h>

#include <new>

#include "comic_internal.cuh"

namespace comic {

static thread_local char g_err[1024] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

}  // namespace comic

using namespace comic;

extern "C" const char* comic_last_error(void) { return g_err; }
extern "C" const char* comic_version(void) { return "comic_b200 0.2 (sm_100a; fp32 FFMA + tcgen05 bf16x3)"; }

extern "C" int comic_create(const comic_cfg_t* cfg, comic_handle_t* out) {
  COMIC_REQUIRE(cfg && out, COMIC_E_BADARG, "create: null argument");
  COMIC_REQUIRE(cfg->rnn_size > 0 && cfg->rnn_size % 128 == 0, COMIC_E_UNSUPPORTED,
                "create: rnn_size %d must be a positive multiple of 128", cfg->rnn_size);
  COMIC_REQUIRE(cfg->word_size > 0 && cfg->word_size % 4 == 0, COMIC_E_UNSUPPORTED, "create: word_size %% 4 != 0");
  COMIC_REQUIRE(cfg->num_heads > 0 && cfg->rnn_size % cfg->num_heads == 0 &&
                    (cfg->rnn_size / cfg->num_heads) % 4 == 0,
                COMIC_E_UNSUPPORTED, "create: heads %d incompatible with rnn_size %d", cfg->num_heads, cfg->rnn_size);
  COMIC_REQUIRE(cfg->fm_channels > 0 && cfg->fm_channels % 4 == 0 && cfg->fm_positions > 0, COMIC_E_SHAPE,
                "create: bad feature map %d x %d", cfg->fm_positions, cfg->fm_channels);
  COMIC_REQUIRE(cfg->vocab > 1 && cfg->eos_id >= 0 && cfg->eos_id < cfg->vocab, COMIC_E_SHAPE, "create: bad vocab / eos");
  COMIC_REQUIRE(cfg->fm_projection >= 0 && cfg->fm_projection <= 2, COMIC_E_BADARG, "create: fm_projection");
  COMIC_REQUIRE(cfg->alignment == 0 || cfg->alignment == 1, COMIC_E_BADARG,
                "create: Invalid alignment method.");   // src/model_base.py:133-138
  COMIC_REQUIRE(cfg->prob_fn == 0 || cfg->prob_fn == 1, COMIC_E_BADARG, "create: Invalid alignment method.");
  COMIC_REQUIRE(cfg->embed_size % 4 == 0, COMIC_E_SHAPE, "create: embed_size %% 4 != 0");
  comic_handle_s* h = new (std::nothrow) comic_handle_s();
  COMIC_REQUIRE(h, COMIC_E_BADARG, "create: out of host memory");
  h->cfg = *cfg;
  COMIC_CHECK_CUDA(cudaGetDevice(&h->dev));
  cudaDeviceProp prop;
  COMIC_CHECK_CUDA(cudaGetDeviceProperties(&prop, h->dev));
  h->num_sms = prop.multiProcessorCount;
  h->R = cfg->rnn_size; h->W = cfg->word_size; h->H = cfg->num_heads;
  h->C = cfg->fm_channels; h->M = cfg->fm_positions; h->E = cfg->embed_size; h->V = cfg->vocab;
  h->Vp = round_up(h->V, 4);
  h->VAL = (cfg->fm_projection == 0) ? h->C : h->R;
  h->A = (cfg->fm_projection == 0 && !cfg->context_layer) ? h->C : h->R;   // src/model_base.py:611-615
  h->LQ = h->Vp + h->R;
  h->KX = h->W + h->A + h->R;
  if (h->VAL % h->H != 0) {
    delete h;
    set_error("create: value width %d not divisible by heads %d", h->VAL, h->H);
    return COMIC_E_SHAPE;
  }
  memset(&h->w, 0, sizeof(h->w));
  int rc = decoder_configure();
  if (rc) { delete h; return rc; }
  if (cudaMallocHost(&h->attn2_host, 16 * sizeof(float)) != cudaSuccess) {   // see attn2_prepare (decoder.cu)
    h->attn2_host = nullptr;
    (void)cudaGetLastError();
  }
  *out = h;
  return COMIC_OK;
}

extern "C" int comic_destroy(comic_handle_t h) {
  if (h && h->prof_ev) {
    for (int i = 0; i < 2 * kMaxProfEvents; ++i) cudaEventDestroy(h->prof_ev[i]);
    delete[] h->prof_ev;
    delete[] h->prof_tag;
  }
  if (h && h->attn2_host) cudaFreeHost(h->attn2_host);
  delete h;
  return COMIC_OK;
}

extern "C" int comic_profile_enable(comic_handle_t h, uint32_t tag_mask) {
  COMIC_REQUIRE(h, COMIC_E_BADARG, "profile_enable: null handle");
  if (tag_mask && !h->prof_ev) {
    h->prof_ev = new cudaEvent_t[2 * kMaxProfEvents];
    h->prof_tag = new int[kMaxProfEvents];
    for (int i = 0; i < 2 * kMaxProfEvents; ++i) COMIC_CHECK_CUDA(cudaEventCreate(&h->prof_ev[i]));
  }
  h->prof_mask = tag_mask;
  h->prof_used = 0;
  return COMIC_OK;
}

extern "C" int comic_profile_read(comic_handle_t h, int tag, double* total_ms, int64_t* count) {
  COMIC_REQUIRE(h && total_ms && count, COMIC_E_BADARG, "profile_read: null argument");
  double tot = 0.0;
  int64_t n = 0;
  for (int i = 0; i < h->prof_used; ++i) {
    if (h->prof_tag[i] != tag) continue;
    COMIC_CHECK_CUDA(cudaEventSynchronize(h->prof_ev[2 * i + 1]));
    float ms = 0.f;
    COMIC_CHECK_CUDA(cudaEventElapsedTime(&ms, h->prof_ev[2 * i], h->prof_ev[2 * i + 1]));
    tot += ms;
    ++n;
  }
  *total_ms = tot;
  *count = n;
  return COMIC_OK;
}

namespace comic {
int pack_tc_weight(comic_handle_t h, Carver& cv, const float* W, int K, int N, int ldw, int cin_src, int cin_dst,
                   tc::TcWeight& out, cudaStream_t st, bool dry) {
  (void)h;
  int ntaps = K / cin_src;
  int Kd = (cin_src == cin_dst) ? K : ntaps * cin_dst;
  out.N = N;
  out.K = Kd;
  out.Npad = round_up(N, 16);
  out.Kpad = round_up(Kd, tc::BK);
  size_t n = (size_t)out.Npad * out.Kpad;
  out.hi = cv.take<uint16_t>(n);
  out.lo = cv.take<uint16_t>(n);
  out.ready = false;
  if (dry) return COMIC_OK;
  tc::pack_bt_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(W, K, N, ldw, out.hi, out.lo, out.Kpad, out.Npad,
                                                                 cin_src, cin_dst);
  COMIC_CHECK_CUDA(cudaGetLastError());
  COMIC_REQUIRE(tc::make_weight_maps(out), COMIC_E_CUDA, "cuTensorMapEncodeTiled failed for a %d x %d weight", N, Kd);
  return COMIC_OK;
}
}  // namespace comic

extern "C" int comic_set_precision(comic_handle_t h, int mode) {
  COMIC_REQUIRE(h && mode >= 0 && mode <= 2, COMIC_E_BADARG, "set_precision: mode must be 0 (f32), 1 (split tensor) or 2 (fast)");
  h->precision = mode;
  return COMIC_OK;
}

extern "C" int comic_set_option(comic_handle_t h, int option, int value) {
  COMIC_REQUIRE(h, COMIC_E_BADARG, "set_option: null handle");
  switch (option) {
    case COMIC_OPT_FUSED_ATTN_MIN_IMAGES: h->fused_min_images = value; return COMIC_OK;
    case COMIC_OPT_PERSISTENT_MAX_ROWS: h->persist_max_rows = value; return COMIC_OK;
    case COMIC_OPT_PERSISTENT_TRACE: h->persist_trace = value; return COMIC_OK;
    case COMIC_OPT_PERSISTENT_WATCHDOG_MS:
      if (value < 0) break;
      h->persist_watchdog_ms = value;
      return COMIC_OK;
    case COMIC_OPT_STEM_S2D:
      COMIC_REQUIRE(value == 0 || value == 2, COMIC_E_BADARG, "set_option: stem_s2d must be 0 (7x7 gather) or 2 (halo)");
      h->stem_s2d = value;
      return COMIC_OK;
    case COMIC_OPT_TC_MIN_ROWS: h->tc_min_rows = value; return COMIC_OK;
    case COMIC_OPT_TC_SPLITK: h->tc_splitk = value; return COMIC_OK;
    case COMIC_OPT_ATTN2: h->attn2 = value; return COMIC_OK;
    case COMIC_OPT_TMA_A: h->tma_a = value; return COMIC_OK;
    case COMIC_OPT_ENC_CHUNK_STEM:
    case COMIC_OPT_ENC_CHUNK_28:
    case COMIC_OPT_ENC_CHUNK_14:
      COMIC_REQUIRE(value >= 1, COMIC_E_BADARG, "set_option: encoder chunk must be >= 1");
      h->enc_chunk[option - COMIC_OPT_ENC_CHUNK_STEM] = value;
      return COMIC_OK;
    default: break;
  }
  set_error("set_option: unknown option %d", option);
  return COMIC_E_BADARG;
}

extern "C" int comic_decode_trace(comic_handle_t h, int64_t* out, int max_steps, int* steps, void* stream) {
  COMIC_REQUIRE(h && out && steps, COMIC_E_BADARG, "decode_trace: null argument");
  int n = h->last_trace_steps < max_steps ? h->last_trace_steps : max_steps;
  *steps = n;
  if (n <= 0 || !h->last_trace) { *steps = 0; return COMIC_OK; }
  COMIC_CHECK_CUDA(cudaMemcpyAsync(out, h->last_trace, (size_t)n * 32 * sizeof(int64_t), cudaMemcpyDeviceToHost,
                                   (cudaStream_t)stream));
  COMIC_CHECK_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
  return COMIC_OK;
}

extern "C" int comic_packed_bytes(comic_handle_t h, size_t* bytes) {
  COMIC_REQUIRE(h && bytes, COMIC_E_BADARG, "packed_bytes: null argument");
  Carver cv(nullptr);
  comic::Packed keep = h->pk;
  h->sized = true;
  decoder_pack(h, cv, 0, true);
  encoder_pack(h, cv, 0, true);
  h->pk = keep;
  *bytes = cv.off + 256;
  return COMIC_OK;
}

extern "C" int comic_set_rnn_cell(comic_handle_t h, int cell) {
  COMIC_REQUIRE(h, COMIC_E_BADARG, "set_rnn_cell: null handle");
  COMIC_REQUIRE(cell == COMIC_CELL_LSTM || cell == COMIC_CELL_GRU, COMIC_E_UNSUPPORTED,
                "set_rnn_cell: cell %d is not built (0 LSTM, 1 GRU)", cell);
  COMIC_REQUIRE(!h->bound && !h->sized, COMIC_E_BADARG,
                "set_rnn_cell: call it before any size query or binding (packed and workspace layouts depend on the cell)");
  h->cell = cell;
  return COMIC_OK;
}

extern "C" int comic_set_fm_endpoint(comic_handle_t h, int endpoint) {
  COMIC_REQUIRE(h, COMIC_E_BADARG, "set_fm_endpoint: null handle");
  COMIC_REQUIRE(endpoint >= 0 && endpoint < kNumFmTaps, COMIC_E_UNSUPPORTED,
                "set_fm_endpoint: end point %d is not built (0..8: MaxPool_4a_3x3, Mixed_4b..4f, MaxPool_5a_2x2, Mixed_5b, "
                "Mixed_5c)", endpoint);
  COMIC_REQUIRE(!h->bound && !h->sized, COMIC_E_BADARG,
                "set_fm_endpoint: call it before any size query or binding (workspace layouts depend on the end point)");
  const int C = kFmTapC[endpoint], S = kFmTapS[endpoint];
  COMIC_REQUIRE(h->C == C && h->M == S * S, COMIC_E_SHAPE,
                "set_fm_endpoint: end point %d is [%d x %d, %d] but the config has fm_positions %d, fm_channels %d", endpoint,
                S, S, C, h->M, h->C);
  h->fm_tap = endpoint;
  return COMIC_OK;
}

extern "C" int comic_bind_gru_candidate(comic_handle_t h, const float* kernel, const float* bias) {
  COMIC_REQUIRE(h && kernel && bias, COMIC_E_BADARG, "bind_gru_candidate: null argument");
  COMIC_REQUIRE(h->cell == COMIC_CELL_GRU, COMIC_E_BADARG, "bind_gru_candidate: the handle's cell is not GRU");
  h->gru_cand_kernel = kernel;
  h->gru_cand_bias = bias;
  h->bound = false;   // the packed panels were built from the previous candidate: decoding waits for comic_bind_weights
  return COMIC_OK;
}

extern "C" int comic_bind_weights(comic_handle_t h, const comic_weights_t* w, int with_cnn, void* packed,
                                  size_t packed_bytes, void* stream) {
  COMIC_REQUIRE(h && w && packed, COMIC_E_BADARG, "bind_weights: null argument");
  size_t need;
  comic_packed_bytes(h, &need);
  COMIC_REQUIRE(packed_bytes >= need, COMIC_E_WORKSPACE, "bind_weights: packed buffer %zu < %zu", packed_bytes, need);
  COMIC_REQUIRE(w->lstm_kernel && w->lstm_bias && w->init_weight && w->memory_kernel && w->query_kernel &&
                    w->out_kernel && w->out_bias && w->embedding_map,
                COMIC_E_BADARG, "bind_weights: missing decoder tensor");
  if (h->cfg.alignment == 0)
    COMIC_REQUIRE(w->attention_v && w->ln_gamma && w->ln_beta && w->temperature, COMIC_E_BADARG,
                  "bind_weights: missing add_LN attention tensor");
  if (h->cell == COMIC_CELL_GRU)
    COMIC_REQUIRE(h->gru_cand_kernel && h->gru_cand_bias, COMIC_E_BADARG,
                  "bind_weights: GRU cell without candidate/{kernel, bias} (comic_bind_gru_candidate)");
  if (h->cfg.fm_projection == 2) COMIC_REQUIRE(w->value_kernel, COMIC_E_BADARG, "bind_weights: missing value_layer");
  if (h->cfg.context_layer) COMIC_REQUIRE(w->a_layer, COMIC_E_BADARG, "bind_weights: missing a_layer");
  if (with_cnn) {
    for (int i = 0; i < COMIC_NUM_CONVS; ++i)
      COMIC_REQUIRE(w->conv_w[i] && w->bn_beta[i] && w->bn_mean[i] && w->bn_var[i], COMIC_E_BADARG,
                    "bind_weights: missing CNN tensor %d", i);
    if (h->cfg.legacy)
      COMIC_REQUIRE(w->enc_ln_gamma && w->enc_ln_beta && w->enc_embed_weight, COMIC_E_BADARG,
                    "bind_weights: missing legacy encoder head");
  }
  h->w = *w;
  cudaStream_t st = (cudaStream_t)stream;
  Carver cv(packed);
  int rc = decoder_pack(h, cv, st, false);
  if (rc) return rc;
  rc = encoder_pack(h, cv, st, !with_cnn);
  if (rc) return rc;
  h->bound = true;
  h->attn2_state = 0;
  h->cnn_bound = with_cnn != 0;
  return COMIC_OK;
}

extern "C" int comic_workspace_bytes(comic_handle_t h, int mode, int B, int k, int T, size_t* bytes) {
  COMIC_REQUIRE(h && bytes, COMIC_E_BADARG, "workspace_bytes: null argument");
  COMIC_REQUIRE(B > 0 && k > 0 && T >= 0, COMIC_E_SHAPE, "workspace_bytes: bad B=%d k=%d T=%d", B, k, T);
  h->sized = true;
  if (mode == 0) return encoder_workspace_bytes(h, B, bytes);
  if (mode == 5) {   // gemm_f32 tensor-path scratch: B = N, k = K of the GEMM (B^T hi/lo pack)
    *bytes = 2 * (size_t)round_up(B, 16) * round_up(k, tc::BK) * sizeof(float) + 2048;
    return COMIC_OK;
  }
  return decoder_workspace_bytes(h, mode, B, k, T, bytes);
}

extern "C" int comic_encode_fwd(comic_handle_t h, const float* images, int B, float* fm_out, float* im_embed_out,
                                float* mixed5c_out, void* ws, size_t ws_bytes, void* stream) {
  COMIC_REQUIRE(h && images && fm_out && im_embed_out && ws, COMIC_E_BADARG, "encode_fwd: null argument");
  COMIC_REQUIRE(B > 0, COMIC_E_SHAPE, "encode_fwd: bad batch %d", B);
  return encoder_forward(h, images, B, fm_out, im_embed_out, mixed5c_out, ws, ws_bytes, (cudaStream_t)stream);
}

extern "C" int comic_gemm_f32(comic_handle_t h, const float* A, int lda, const float* Bm, int ldb, const float* bias,
                              float* C, int ldc, int M, int N, int K, void* ws, size_t ws_bytes, void* stream) {
  COMIC_REQUIRE(h && A && Bm && C, COMIC_E_BADARG, "gemm_f32: null argument");
  COMIC_REQUIRE(M > 0 && N > 0 && K > 0, COMIC_E_SHAPE, "gemm_f32: bad shape");
  COMIC_REQUIRE(N % 4 == 0 && ldb % 4 == 0 && ldc % 4 == 0, COMIC_E_UNSUPPORTED, "gemm_f32: N, ldb, ldc must be multiples of 4");
  APlain a{};
  a.nseg = 1;
  a.seg[0] = ASeg{A, nullptr, lda, K, M};
  Epi e{};
  e.bias = bias;
  e.nroute = 1;
  e.r[0] = Route{0, N, C, ldc, 0};
  e.stop_n = 0x7fffffff;
  GemmPlan p = plan_gemm(M, N, K, h->num_sms, false);
  cudaError_t err;
  if (h->precision >= 1 && M >= 128 && K % 4 == 0 && lda % 4 == 0) {
    // tensor path: pack B on the fly into the caller's workspace
    size_t need = 2 * (size_t)round_up(N, 16) * round_up(K, tc::BK) * sizeof(float) + 1024;
    COMIC_REQUIRE(ws && ws_bytes >= need, COMIC_E_WORKSPACE, "gemm_f32: tensor path needs %zu workspace bytes", need);
    Carver cv(ws);
    tc::TcWeight tw;
    int rc = pack_tc_weight(h, cv, Bm, K, N, ldb, 1, 1, tw, (cudaStream_t)stream, false);
    if (rc) return rc;
    err = tc::launch_gemm_tc<0>(a, tw, M, N, e, h->num_sms, (cudaStream_t)stream);
    h->launches += 2;
    COMIC_CHECK_CUDA(err);
    return COMIC_OK;
  }
  if (K % 4 == 0 && lda % 4 == 0) err = launch_gemm<0, 4>(a, Bm, ldb, M, N, K, e, p, (cudaStream_t)stream);
  else err = launch_gemm<0, 1>(a, Bm, ldb, M, N, K, e, p, (cudaStream_t)stream);
  h->launches++;
  COMIC_CHECK_CUDA(err);
  return COMIC_OK;
}

extern "C" int comic_launch_count(comic_handle_t h, int64_t* count) {
  COMIC_REQUIRE(h && count, COMIC_E_BADARG, "launch_count: null argument");
  *count = h->launches;
  return COMIC_OK;
}
