/*
 * comic_b200.h -- C ABI of libcomic_b200.so, the B200 (sm_100a) engine behind the
 * COMIC caption-decoding hot path.
 *
 * The reference (jiahuei/COMIC-Compact-Image-Captioning-with-Attention) has no
 * FFI: its boundary is the Python call surface that the session loops drive
 * (SURVEY.md §8b).  Each entry point below names the reference call it replaces
 * (file:line under the reference tree).  The Python shim in
 * comic-compact-image-captioning-with-attention_b200/ binds these with ctypes
 * and re-exposes the reference's own signatures (rops.*, CaptionModel).
 *
 * Conventions
 *   - every function returns 0 on success or a negative COMIC_E_* code;
 *     comic_last_error() returns a thread-local message for the last failure;
 *   - all tensor arguments are DEVICE pointers unless named host_*; row-major,
 *     fp32 unless stated; ids/parents int32, lengths int64, flags uint8;
 *   - the caller (PyTorch's allocator in the shim) owns every device buffer,
 *     including `packed` weights and per-call `ws` workspaces; the library never
 *     allocates or frees device memory and never synchronises the stream;
 *   - a handle is bound to one device; calls on one handle are not re-entrant;
 *     distinct handles are independent (one per GPU / process);
 *   - `stream` is a cudaStream_t passed as void*.
 */
#ifndef COMIC_B200_H_
#define COMIC_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define COMIC_OK             0
#define COMIC_E_BADARG      -1
#define COMIC_E_SHAPE       -2
#define COMIC_E_CUDA        -3
#define COMIC_E_UNSUPPORTED -4
#define COMIC_E_WORKSPACE   -5

#define COMIC_NUM_CONVS 57   /* common/nets/inception_v1.py:70-261 */

typedef struct comic_handle_s* comic_handle_t;

/* Model description = the config.pkl fields that shape the graph
 * (src/model_base.py:40-46, 109-184, 606-689). */
typedef struct {
  int32_t rnn_size;        /* R: c.rnn_size (512) */
  int32_t word_size;       /* W: c.rnn_word_size (256) */
  int32_t num_heads;       /* H: c.attn_num_heads */
  int32_t fm_channels;     /* C: channels of c.cnn_fm_attention (832 for Mixed_4f; see comic_set_fm_endpoint) */
  int32_t fm_positions;    /* M: 196 for a 14x14 end point, 49 for a 7x7 one */
  int32_t embed_size;      /* E: 1024 (im_embed) */
  int32_t vocab;           /* V: softmax size (radix_base+2 | len(itow)) */
  int32_t fm_projection;   /* c.cnn_fm_projection: 0 none, 1 tied, 2 independent */
  int32_t context_layer;   /* c.attn_context_layer */
  int32_t init_method;     /* c.rnn_init_method: 0 first_input, 1 project_hidden */
  int32_t alignment;       /* c.attn_alignment_method: 0 add_LN, 1 dot */
  int32_t prob_fn;         /* c.attn_probability_fn: 0 softmax, 1 sigmoid(_signorm) */
  int32_t embed_lookup;    /* 0: one_hot x matmul (radix/char; id outside [0,V) -> zero row);
                              1: embedding_lookup (word)  (src/model_base.py:557-594) */
  int32_t legacy;          /* c.legacy: LN+tanh+linear encoder head (src/model_base.py:80-91) */
  int32_t go_id, eos_id;   /* src/model_base.py:701-706 */
} comic_cfg_t;

/* Device pointers to the reference's variables, TF shapes (SURVEY.md §8a). */
typedef struct {
  const float* lstm_kernel;      /* [W+A+R, 4R] gate order i,j,f,o; GRU cell: gates/kernel [W+A+R, 2R], r then u */
  const float* lstm_bias;        /* [4R]; GRU cell: gates/bias [2R] */
  const float* init_weight;      /* first_input: [E, W+A]; project_hidden: [E, R] */
  const float* memory_kernel;    /* [C, R] */
  const float* value_kernel;     /* [C, R] (independent) or NULL */
  const float* query_kernel;     /* [R, R] */
  const float* attention_v;      /* [R] */
  const float* ln_gamma;         /* [R] */
  const float* ln_beta;          /* [R] */
  const float* temperature;      /* [1] */
  const float* a_layer;          /* [VAL, R] or NULL */
  const float* out_kernel;       /* [R, V] */
  const float* out_bias;         /* [V] */
  const float* embedding_map;    /* [V, W] */
  const float* enc_ln_gamma;     /* legacy [E] or NULL */
  const float* enc_ln_beta;      /* legacy [E] or NULL */
  const float* enc_embed_weight; /* legacy [E, E] or NULL */
  /* InceptionV1, conv order = comic_conv_table() */
  const float* conv_w[COMIC_NUM_CONVS];    /* HWIO */
  const float* bn_beta[COMIC_NUM_CONVS];
  const float* bn_mean[COMIC_NUM_CONVS];
  const float* bn_var[COMIC_NUM_CONVS];
} comic_weights_t;

typedef struct { int32_t k, stride, c_in, c_out; } comic_conv_desc_t;

const char* comic_last_error(void);
const char* comic_version(void);

/* The 57 (k, stride, c_in, c_out) conv descriptors in weight order. */
const comic_conv_desc_t* comic_conv_table(void);

/* Replaces graph construction: CaptionModel.__init__ src/model.py:23-73. */
int comic_create(const comic_cfg_t* cfg, comic_handle_t* out);
int comic_destroy(comic_handle_t h);

/* Bytes of the engine-layout weight pack ([W_o|W_q] panel, folded BN
 * scale/shift, grouped 1x1 conv panels). */
int comic_packed_bytes(comic_handle_t h, size_t* bytes);
/* Replaces ModelBase.restore_model src/model_base.py:422-490 (variables ->
 * engine).  `with_cnn` = 0 binds the decoder only. */
int comic_bind_weights(comic_handle_t h, const comic_weights_t* w, int with_cnn,
                       void* packed, size_t packed_bytes, void* stream);

/* Recurrent cell of the decoder (c.rnn_name, src/model_base.py:622-629).  Call after comic_create and before
 * comic_packed_bytes / comic_workspace_bytes / comic_bind_weights: the packed weights and the decode workspaces are
 * laid out for the cell.  Any other value returns COMIC_E_UNSUPPORTED.
 *   LSTM: BasicLSTMCell (default).
 *   GRU:  TF r1.9 GRUCell, state h only:
 *           [r, u] = sigmoid([x, h] . gates/kernel + gates/bias)
 *           c      = tanh([x, r*h] . candidate/kernel + candidate/bias)
 *           h'     = u*h + (1-u)*c
 *         The c0 / c_in / c_out arguments of comic_rnn_init, comic_decode_step, comic_decode_greedy and
 *         comic_decode_beam may be NULL and are neither read nor written.  Decodes take the per-step path (no
 *         persistent loop).  Training writes the candidate gradients to comic_decoder_grads_t.cand_kernel / cand_bias. */
#define COMIC_CELL_LSTM 0
#define COMIC_CELL_GRU  1
int comic_set_rnn_cell(comic_handle_t h, int cell);
/* GRU cell: candidate/kernel [W+A+R, R] and candidate/bias [R], bound by pointer (the weights are read in place by
 * every bind / comic_refresh_packed).  Call before comic_bind_weights, which refuses a GRU handle without them; a call
 * after binding unbinds the weights until the next comic_bind_weights.  comic_set_rnn_cell returns COMIC_E_BADARG once
 * a size (packed, workspace, train workspace) was queried or weights were bound;
 * comic_weights_t.lstm_kernel / lstm_bias carry gates/kernel / gates/bias. */
int comic_bind_gru_candidate(comic_handle_t h, const float* kernel, const float* bias);

/* InceptionV1 end point the decoder attends over (c.cnn_fm_attention, src/model_base.py:94-104): the tensor
 * comic_encode_fwd / comic_encode_train_fwd write to fm_out and comic_encode_bwd takes dfm at.  Call after comic_create
 * and before comic_packed_bytes / comic_workspace_bytes / comic_bind_weights (COMIC_E_BADARG afterwards).  The
 * config's fm_channels / fm_positions must be the end point's (C, S*S), else COMIC_E_SHAPE; any other id returns
 * COMIC_E_UNSUPPORTED (the 28x28 and earlier end points are not built).  Default COMIC_FM_MIXED_4F.
 *   id                       S x S    C
 *   COMIC_FM_MAXPOOL_4A_3X3  14x14   480
 *   COMIC_FM_MIXED_4B..4D    14x14   512
 *   COMIC_FM_MIXED_4E        14x14   528
 *   COMIC_FM_MIXED_4F        14x14   832
 *   COMIC_FM_MAXPOOL_5A_2X2   7x7    832
 *   COMIC_FM_MIXED_5B         7x7    832
 *   COMIC_FM_MIXED_5C         7x7   1024 */
#define COMIC_FM_MAXPOOL_4A_3X3 0
#define COMIC_FM_MIXED_4B       1
#define COMIC_FM_MIXED_4C       2
#define COMIC_FM_MIXED_4D       3
#define COMIC_FM_MIXED_4E       4
#define COMIC_FM_MIXED_4F       5
#define COMIC_FM_MAXPOOL_5A_2X2 6
#define COMIC_FM_MIXED_5B       7
#define COMIC_FM_MIXED_5C       8
int comic_set_fm_endpoint(comic_handle_t h, int endpoint);

/* Arithmetic modes (all within the 1e-3 parity bound of the reference's fp32 graph):
 *   0  fp32 FFMA everywhere (the reference's fp32 arithmetic up to summation order);
 *   1  tcgen05 tensor cores with an error-compensated operand split and fp32
 *      accumulation for GEMMs / convolutions with >= 128 rows (fp32-equivalent,
 *      ~1e-6 relative); tanh = 1 - 2/(2^(2y log2 e) + 1) via ex2/rcp (default);
 *   2  as 1, but the attention LN-tanh uses the single-MUFU tanh.approx.f32
 *      (|err| <= 2^-11 per element, ~1e-5 on attention maps).
 * Small-row GEMMs (M < 128, e.g. batch-8 decode) always use the FFMA kernel. */
int comic_set_precision(comic_handle_t h, int mode);

/* Engine tunables (no reference counterpart).  Ids 6-8, 10, 13, 14, 16 and 17 are retired and refused. */
#define COMIC_OPT_FUSED_ATTN_MIN_IMAGES 0   /* one-CTA-per-image fused attention from this batch on (default 48) */
#define COMIC_OPT_ENC_CHUNK_STEM 1          /* images per encoder chunk, stem convs (default 256) */
#define COMIC_OPT_ENC_CHUNK_28 2            /* ... Mixed_3b/3c (default 512) */
#define COMIC_OPT_ENC_CHUNK_14 3            /* ... Mixed_4b..5c (default 512); set before comic_workspace_bytes */
#define COMIC_OPT_PERSISTENT_MAX_ROWS 4      /* decode loops with batch*beam <= this run as ONE cooperative kernel
                                             * (default 32, the kernel's limit; 0 = always one launch per step op) */
#define COMIC_OPT_PERSISTENT_TRACE 5         /* 1: the persistent loop records per-phase clock stamps (diagnostics) */
#define COMIC_OPT_STEM_S2D 9                 /* tensor-path stem conv: 2 (default) = 4x4 stride-1 conv over the space-to-depth
                                             * image stored as bf16 planes, each 8x16-pixel tile's im2col rows built from a
                                             * shared-memory halo patch (one L2 read per input element per tile instead of
                                             * 16); 0 = 7x7/2 gather from NHWC4 fp32; other values are refused */
#define COMIC_OPT_ATTN2 12                   /* 1 (default): large-batch decode steps use the streaming attention kernel
                                                (TMA-staged key slices, one HBM pass per step) where it applies: tied
                                                values, add_LN, softmax, rnn_size 512, 8 heads, beam <= 3; 0: never */
#define COMIC_OPT_TMA_A 15                   /* bit 0: [logits | query] GEMM, bit 1: gate GEMM -- on the tensor path the GEMM reads its A
                                               operand as bf16 (hi, lo) planes through TMA (h' planes are written by the LSTM kernel;
                                               x = [emb ; ctx ; h] is gathered and split once per step by a small kernel) instead of
                                               gathering and splitting fp32 rows in every N tile's loader warps.  Default 1. */
#define COMIC_OPT_PERSISTENT_WATCHDOG_MS 18   /* how long a CTA of the persistent decode loop may spin at a grid barrier before the
                                               launch is declared dead (T_out = -1); default 2000, 0 = never (time-sliced GPUs,
                                               debuggers) */
#define COMIC_OPT_TC_SPLITK 19                /* bit 0: gate GEMM, bit 1: [logits | query] GEMM (default 3): tensor-path decoder GEMMs with at most 128 rows (batch 25 x beam 3 = 75,
                                               the reference's default inference shape) cut their K loop into up to 8 ranges,
                                               one CTA each; the partial sums are added in a fixed order by the consumer */
#define COMIC_OPT_TC_MIN_ROWS 11             /* GEMMs / convs with at least this many rows run on the tensor path when
                                             * precision >= 1 (default 64) */
int comic_set_option(comic_handle_t h, int option, int value);

/* Diagnostics: clock64 stamps of the last persistent decode call, [steps][2][16] int64 (CTA 0 and the first
 * selection CTA); slot order in time: 0 step start, 9 row pointers, 10 x slice loaded, 11 partial gates, 12 barrier,
 * 1 LSTM cell, 2 barrier, 3 logits|query, 4 barrier, 5 scores, 6 barrier, 7 softmax+context, 8 barrier.
 * Valid until the workspace of that call is reused.  Synchronises the stream.  *steps = 0 when tracing was off or
 * the per-step path ran. */
int comic_decode_trace(comic_handle_t h, int64_t* out, int max_steps, int* steps, void* stream);

/* mode: 0 encode, 1 decode_greedy, 2 decode_beam, 3 decode_step, 4 rnn_init,
 * 5 gemm_f32 (B = N, k = K of the GEMM). */
int comic_workspace_bytes(comic_handle_t h, int mode, int B, int k, int T, size_t* bytes);

/* E1+E2: ModelBase._encoder src/model_base.py:56-104 (InceptionV1 forward,
 * common/nets/inception_v1.py:29-339).  images [B,224,224,3] NHWC in [-1,1];
 * fm_out [B,M,C] = the end point of comic_set_fm_endpoint; im_embed_out [B,1024]; mixed5c_out optional
 * [B,7,7,1024] (at COMIC_FM_MIXED_5C it may be fm_out itself: the two are the same tensor). */
int comic_encode_fwd(comic_handle_t h, const float* images, int B, float* fm_out,
                     float* im_embed_out, float* mixed5c_out, void* ws, size_t ws_bytes,
                     void* stream);

/* Evaluation pre-processing, common/inputs/preprocessing/inception_preprocessing_radix.py:229-235, 270-273
 * (convert_image_dtype -> resize_bilinear 256x256, align_corners=False -> central crop / zero pad to
 * out_h x out_w -> (x - 0.5) * 2), fused.  images uint8 [B,H,W,3] (decoded RGB, one size per call);
 * out fp32 [B,out_h,out_w,3] = the `images` argument of comic_encode_fwd.  A batch of images of mixed sizes takes
 * comic_preprocess_ragged instead. */
int comic_preprocess_eval(comic_handle_t h, const uint8_t* images, int B, int H, int W, int out_h, int out_w,
                          float* out, void* stream);

/* Training-time pre-processing (inception_preprocessing_radix.py:158-201 `preprocess_for_train`, after the shared
 * convert_image_dtype + resize_bilinear(256, 256) of :270-273): optional left-right flip of the resized image
 * (flip[b] != 0; NULL = never), crop of out_h x out_w at crop_yx[b] = (y0, x0) with 0 <= y0 <= 256 - out_h, same for x
 * (tf.random_crop), (x - 0.5) * 2.  The random draws are the caller's.  images uint8 [B,H,W,3] device, out fp32
 * [B,out_h,out_w,3] device. */
int comic_preprocess_train(comic_handle_t h, const uint8_t* images, int B, int H, int W, int out_h, int out_w,
                           const int32_t* crop_yx, const uint8_t* flip, float* out, void* stream);

/* The same pre-processing for a batch of decoded RGB images of mixed sizes, in one launch whose grid depends on B and
 * out_h x out_w only.  Image b is hw[b] = (h, w) uint8 [h,w,3] at bytes + offsets[b].  crop_yx == NULL: evaluation
 * (as comic_preprocess_eval, flip must be NULL); otherwise training (as comic_preprocess_train, with its out <= 256
 * rule).  bytes, offsets (int64 [B]), hw (int32 [B,2]), crop_yx, flip and out are device pointers; the library cannot
 * read the tables without a synchronise, so the caller guarantees h, w >= 1 and that every image lies inside the
 * buffer.  Each image gives the bits comic_preprocess_eval / comic_preprocess_train give it alone. */
int comic_preprocess_ragged(comic_handle_t h, const uint8_t* bytes, int B, const int64_t* offsets, const int32_t* hw,
                            int out_h, int out_w, const int32_t* crop_yx, const uint8_t* flip, float* out,
                            void* stream);

/* D0: MultiHeadAttV3.__init__ common/ops_rnn.py:441-477: keys = fm.W_k once per
 * IMAGE (the reference does it per tiled beam row); values_out only for
 * `independent`. fm [B,M,C]; keys_out [B,M,R]; values_out [B,M,R] or NULL. */
int comic_project_fm(comic_handle_t h, const float* fm, int B, float* keys_out,
                     float* values_out, void* stream);

/* D1: ModelBase._get_rnn_init src/model_base.py:651-689. im_embed [B,E] ->
 * c0,h0 [B,R]. in_mask optional [B,W+A] 0/1 dropout mask (train), keep prob in_keep. */
int comic_rnn_init(comic_handle_t h, const float* im_embed, int B, float* c0, float* h0,
                   const float* in_mask, float in_keep, void* ws, size_t ws_bytes, void* stream);

/* D3-D7: one MultiHeadAttentionWrapperV3.call + output layer
 * (common/ops_rnn.py:660-755, src/model_base.py:541-543) on N = B*k rows whose
 * memory is keys/values of image n / k.  For unit parity.
 *   tokens [N] i32; c_in,h_in [N,R]; ctx_in [N,A];
 *   outputs: c_out,h_out [N,R]; ctx_out [N,A]; align_out [N,H*M]; logits_out [N,V].
 *   Optional 0/1 dropout masks (NULL = off): in_mask [N,W+A], out_mask [N,R],
 *   att_mask [N,H*M] with keep probabilities. */
int comic_decode_step(comic_handle_t h, const float* keys, const float* values, int B, int k,
                      const int32_t* tokens, const float* c_in, const float* h_in,
                      const float* ctx_in, float* c_out, float* h_out, float* ctx_out,
                      float* align_out, float* logits_out,
                      const float* in_mask, const float* out_mask, const float* att_mask,
                      float in_keep, float out_keep, float att_keep,
                      void* ws, size_t ws_bytes, void* stream);

/* B2: rops.rnn_decoder_search(greedy_search=True) common/ops_rnn.py:115-180.
 *   ids_out [max_it,B] i32; logits_out [max_it,B,V] or NULL;
 *   attn_out [B,H,max_it,M] or NULL (layout of _decoder_post_process
 *   src/model_base.py:307-313); T_out device int32[1] = executed steps. */
int comic_decode_greedy(comic_handle_t h, const float* keys, const float* values,
                        const float* c0, const float* h0, int B, int max_it,
                        int32_t* ids_out, float* logits_out, float* attn_out, int32_t* T_out,
                        void* ws, size_t ws_bytes, void* stream);

/* B1+B3: rops.rnn_decoder_beam_search common/ops_rnn.py:49-112 (TF r1.9
 * BeamSearchDecoder + dynamic_decode + finalize) on B images x k beams.
 * c0,h0 are per IMAGE [B,R] (tile_batch is implicit).
 *   pred_ids_out   [max_it,B,k] i32  gather_tree'd ids (FinalBeamSearchDecoderOutput.predicted_ids)
 *   step_ids_out   [max_it,B,k] i32  raw per-step word ids (optional)
 *   parent_ids_out [max_it,B,k] i32  backpointers
 *   scores_out     [max_it,B,k] f32  per-step top-k scores
 *   lengths_out    [B,k] i64
 *   attn_top_out   [B,H,max_it,M] f32 or NULL: reordered alignment history, top beam
 *                  (src/model_base.py:296-313)
 *   T_out          device int32[1]: executed steps; rows t >= T are EOS / 0. */
int comic_decode_beam(comic_handle_t h, const float* keys, const float* values,
                      const float* c0, const float* h0, int B, int k, float length_penalty_weight,
                      int max_it, int32_t* pred_ids_out, int32_t* step_ids_out,
                      int32_t* parent_ids_out, float* scores_out, int64_t* lengths_out,
                      float* attn_top_out, int32_t* T_out, void* ws, size_t ws_bytes, void* stream);

/* K10 alone: TF r1.9 `_beam_search_step` (called through common/ops_rnn.py:88-104)
 * on given logits [B,k,V] (row stride ld_logits) and beam state; updates
 * log_probs [B,k], finished [B,k] u8, lengths [B,k] i64 in place and writes
 * scores/word/parent [B,k]. */
int comic_beam_step(comic_handle_t h, const float* logits, int ld_logits, int B, int k, int V,
                    int eos_id, float length_penalty_weight, float* log_probs,
                    uint8_t* finished, int64_t* lengths, float* scores_out,
                    int32_t* word_out, int32_t* parent_out, void* stream);

/* K11: TF r1.9 beam_search_ops.gather_tree. step_ids,parent_ids,out [T,B,k] i32;
 * max_seq_len [B] i32. */
int comic_gather_tree(comic_handle_t h, const int32_t* step_ids, const int32_t* parent_ids,
                      const int32_t* max_seq_len, int T, int B, int k, int end_token,
                      int32_t* out, void* stream);

/* The dense kernel on its own (unit parity / roofline): C[M,N] = A[M,K].B[K,N]
 * (+bias[N]); row-major fp32, lda/ldb/ldc in elements; N, ldb, ldc % 4 == 0. */
int comic_gemm_f32(comic_handle_t h, const float* A, int lda, const float* Bm, int ldb,
                   const float* bias, float* C, int ldc, int M, int N, int K,
                   void* ws, size_t ws_bytes, void* stream);


/* ------------------------------------------------------------------------- *
 * Training: train_mode = decoder | scst (frozen CNN) and cnn_finetune (encoder
 * forward-with-tape + backward, further down).
 * ------------------------------------------------------------------------- */

/* Explicit 0/1 dropout masks (NULL member = that dropout off) + keep probabilities:
 * DropoutWrapper input/output dropout (src/model_base.py:637-647) and the
 * attention-map dropout (common/ops_rnn.py:696-701).  Generate them with
 * comic_dropout_masks (Philox4x32-10) or inject them for parity tests. */
typedef struct {
  const float* init_in;   /* [B, W+A]      input mask of the rnn-init LSTM step */
  const float* inp;       /* [T_run, B, W+A] */
  const float* out;       /* [T_run, B, R] */
  const float* att;       /* [T_run, B, H*M] */
  float in_keep, out_keep, att_keep;
} comic_train_masks_t;

/* Device pointers receiving the gradient of each decoder variable (same shapes as
 * comic_weights_t; normally views into one flat buffer that is all-reduced). */
typedef struct {
  float* lstm_kernel; float* lstm_bias; float* init_weight; float* memory_kernel; float* value_kernel;
  float* query_kernel; float* attention_v; float* ln_gamma; float* ln_beta; float* temperature;
  float* out_kernel; float* out_bias; float* embedding_map;
  float* a_layer;                /* [VAL, R] (attn_context_layer, common/ops_rnn.py:734-739) or NULL */
  float* cand_kernel;            /* GRU cell: candidate/kernel [W+A+R, R] (lstm_kernel / lstm_bias receive gates/{kernel,
                                    bias}); NULL for the LSTM */
  float* cand_bias;              /* GRU cell: candidate/bias [R] */
} comic_decoder_grads_t;

int comic_train_workspace_bytes(comic_handle_t h, int B, int T_run, size_t* bytes);

/* 0/1 keep masks: out[i] = uniform(seed, stream_id, i) < keep. */
int comic_dropout_masks(comic_handle_t h, float* out, size_t n, float keep, uint64_t seed, uint64_t stream_id,
                        void* stream);

/* T1+T3: rops.rnn_decoder_training (common/ops_rnn.py:183-243, TrainingHelper,
 * impute_finished=True) + ModelBase._train_caption_model (src/model_base.py:325-383)
 * forward AND backward on B rows (one image per row; SCST callers repeat images).
 *   fm [B,M,C], im_embed [B,E]          encoder outputs (frozen CNN)
 *   inputs_tm, targets_tm [T,B] i32     time-major decoder inputs / targets (_process_inputs :501-528)
 *   coef_tm [T,B] f32                   weight / normaliser per token: XE: mask/(sum mask + 1e-12);
 *                                       SCST: reward_b/B * mask/(sum_t mask + 1e-12)  (:337-347)
 *   lens [B] i32, T_run = max(lens)     executed steps (dynamic_decode stops when all rows finished)
 *   loss_out [4] device                 [unused, xe, map, unused]  (reg: comic_l2_regularise)
 *   logits_out [B,T,V] or NULL, attn_out [B,H,T_run,M] or NULL
 *   grads                               overwritten with dLoss/dvariable (xe + map terms)          */
int comic_train_fwd_bwd(comic_handle_t h, const float* fm, const float* im_embed, int B,
                        const int32_t* inputs_tm, const int32_t* targets_tm, const float* coef_tm,
                        const int32_t* lens, int T, int T_run, const comic_train_masks_t* masks,
                        float map_loss_scale, float* loss_out, float* logits_out, float* attn_out,
                        const comic_decoder_grads_t* grads, void* ws, size_t ws_bytes, void* stream);

/* cnn_finetune, decoder side: gradient of the loss with respect to the encoder outputs.  Call right
 * after comic_train_fwd_bwd with the SAME B, T_run and workspace (it reads the key / value / init-input
 * gradients that call left there):
 *   dfm_out [B,M,C]     = dkeys . W_k^T (+ dvalues . W_v^T | + dvalues for cnn_fm_projection none)
 *   dim_embed_out [B,E] = dx0 . W_I^T   (first_input rnn init, src/model_base.py:675-686)            */
int comic_train_encoder_grads(comic_handle_t h, int B, int T_run, float* dfm_out, float* dim_embed_out,
                              void* ws, size_t ws_bytes, void* stream);

/* --legacy models in train_mode=decoder (the only mode the reference trains them in, src/train.py:242, 253): the image
 * embedding is im_embed = tanh(LN(pool)) . W with pool = mean over the 7x7 positions of Mixed_5c (src/model_base.py:80-91),
 * and LN_tanh/{gamma, beta} and im_embed/weight are trainable (they are not under freeze_scopes = Model/encoder/cnn).
 * Given mixed5c [B,7,7,1024] (comic_encode_fwd's optional output) and d loss / d im_embed [B,1024]
 * (comic_train_encoder_grads), writes d gamma [1024], d beta [1024], d weight [1024,1024]. */
int comic_legacy_head_bwd_bytes(comic_handle_t h, int B, size_t* bytes);
int comic_legacy_head_bwd(comic_handle_t h, const float* mixed5c, int B, const float* d_im_embed, float* d_gamma,
                          float* d_beta, float* d_weight, void* ws, size_t ws_bytes, void* stream);

/* Gradient buffers of the trainable CNN variables (src/train.py:241-250: cnn_finetune clears
 * freeze_scopes; BN runs with is_training=False, src/model_base.py:71-77, so only the conv
 * kernels [HWIO] and the BN betas train).  Order = comic_conv_table(). */
typedef struct {
  float* conv_w[COMIC_NUM_CONVS];
  float* bn_beta[COMIC_NUM_CONVS];
} comic_cnn_grads_t;

/* Bytes of the activation tape (every conv / pool output of the InceptionV1 forward) and of the
 * scratch workspace shared by comic_encode_train_fwd and comic_encode_bwd for B images. */
int comic_encode_train_bytes(comic_handle_t h, int B, size_t* tape_bytes, size_t* ws_bytes);

/* E1+E2 forward that keeps the tape: same outputs as comic_encode_fwd (fm_out [B,M,C] = the end point). */
int comic_encode_train_fwd(comic_handle_t h, const float* images, int B, float* fm_out, float* im_embed_out,
                           void* tape, size_t tape_bytes, void* ws, size_t ws_bytes, void* stream);

/* Backward of the InceptionV1 graph (TF autodiff of common/nets/inception_v1.py:29-339 under
 * create_train_op, src/model_base.py:387-401) from dfm [B,M,C] (at the end point) and dim_embed [B,1024]:
 * overwrites every grads->conv_w[i] / bn_beta[i].  Max-pool gradients go to the first maximum
 * of each window; all reductions have a fixed order (bit-reproducible). */
int comic_encode_bwd(comic_handle_t h, const float* images, int B, const float* dfm, const float* dim_embed,
                     const void* tape, size_t tape_bytes, const comic_cnn_grads_t* grads, void* ws,
                     size_t ws_bytes, void* stream);

/* ModelBase._loss_regularisation (src/model_base.py:408-417) on a flat parameter buffer:
 * grads += decay * params (grads may be NULL); reg_out[0] = decay/2 * sum params^2.  ws >= 4 KB. */
int comic_l2_regularise(comic_handle_t h, const float* params, float* grads, size_t n, float decay,
                        float* reg_out, void* ws, size_t ws_bytes, void* stream);

/* tf.train.AdamOptimizer dense update (src/model_base.py:852-861), step >= 1:
 * lr_t = lr sqrt(1-b2^t)/(1-b1^t); m,v moving averages; params -= lr_t m/(sqrt(v)+eps).
 * grad_scale multiplies the gradient first (1/world_size after a sum all-reduce). */
int comic_adam_step(comic_handle_t h, float* params, const float* grads, float* m, float* v, size_t n,
                    float lr, float beta1, float beta2, float eps, int step, float grad_scale, void* stream);

/* tf.train.MomentumOptimizer(momentum, use_nesterov=False) dense update, `--optimiser sgd` (src/model_base.py:868-880):
 * accum = momentum * accum + grad * grad_scale; params -= lr * accum. */
int comic_momentum_step(comic_handle_t h, float* params, const float* grads, float* accum, size_t n, float lr,
                        float momentum, float grad_scale, void* stream);

/* slim.learning.create_train_op(clip_gradient_norm = max_norm) (src/model_base.py:394-401): each variable's gradient
 * (a slice [offsets[i], offsets[i] + sizes[i]) of the flat buffer; device arrays) is clipped by its own l2 norm. */
int comic_clip_by_norm(comic_handle_t h, float* grads, const int64_t* offsets, const int64_t* sizes, int nvars,
                       float max_norm, void* stream);

/* After the optimiser changed the variables in place: rebuild the decoder's packed copies. */
int comic_refresh_packed(comic_handle_t h, void* packed, size_t packed_bytes, void* stream);
/* Same, decoder AND CNN (folded BN shifts, grouped 1x1 panels, tensor-path panels). */
int comic_refresh_packed_cnn(comic_handle_t h, void* packed, size_t packed_bytes, void* stream);

/* Number of kernels this handle has launched since creation (bench.py's gpu_launches). */
int comic_launch_count(comic_handle_t h, int64_t* count);

/* Per-kernel-class device timing for the roofline report (no reference
 * counterpart; the reference only logs wall-clock, src/infer_fn.py:176-184).
 * Kernel classes (bit i of tag_mask): 0 conv implicit-GEMM, 1 pooling, 2 key
 * projection, 3 rnn init, 4 gate GEMM, 5 LSTM pointwise, 6 logits|query GEMM,
 * 7 attention scores, 8 attention softmax+context, 9 beam step, 10 finalise,
 * 11 misc.  While a class is enabled every launch of it is bracketed by CUDA
 * events on the launching stream; comic_profile_read synchronises those events
 * and returns the summed duration and the launch count.  enable(0) switches
 * timing off; enable() always resets the counters. */
int comic_profile_enable(comic_handle_t h, uint32_t tag_mask);
int comic_profile_read(comic_handle_t h, int tag, double* total_ms, int64_t* count);

#ifdef __cplusplus
}
#endif
#endif /* COMIC_B200_H_ */
