/*
 * nrms_b200.h -- C-ABI of the B200-native NRMS hot path (libnrms_b200.so).
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch types.  Every entry
 * point replaces the PyTorch op sequence of one reference function (file:line relative
 * to the reference tree, Maguire1999/NewsRecommendationSystem):
 *
 *   nrms_news_encoder_fwd/bwd   NewsEncoder.forward            src/model/NRMS/news_encoder.py:27-48
 *   nrms_user_encoder_fwd/bwd   UserEncoder.forward            src/model/NRMS/user_encoder.py:15-26
 *       (both = MultiHeadSelfAttention.forward  src/model/general/attention/multihead_self.py:46-76,
 *               ScaledDotProductAttention.forward :15-23,
 *               AdditiveAttention.forward        src/model/general/attention/additive.py:27-53)
 *   nrms_score_fwd/bwd          DotProductClickPredictor.forward  src/model/general/click_predictor/dot_product.py:8-19
 *   nrms_score_csr              the per-impression get_prediction loop   src/evaluate.py:245-260
 *   nrms_ce_loss_fwd_bwd        CrossEntropyLoss(y_pred, zeros)    src/train.py:126,205-206
 *   nrms_adam_step              torch.optim.Adam(lr=1e-4).step()   src/train.py:127-128,233 (AdamW: decoupled=1)
 *   nrms_rank_metrics           calculate_single_user_metric + nanmean  src/evaluate.py:24-42,160-168,270-272
 *   nrms_news_encoder_rows_fwd/bwd  NewsEncoder over an index-only minibatch    src/dataset.py:17-85, src/train.py:118-124
 *   nrms_text_encoder_fwd/bwd   NewsEncoder.forward / Exp1 TextEncoder at any text length 1..64
 *                               src/model/NRMS/news_encoder.py:27-48, src/model/Exp1/news_encoder.py:10-34
 *   nrms_recommend_user         the single-user path of the demo            src/recommend.py:245-341
 *   nrms_mhsa_fwd/bwd, nrms_mhsa_masked_fwd  MultiHeadSelfAttention.forward(Q, length=...)  multihead_self.py:46-76
 *   nrms_mha_fwd/bwd            MultiHeadSelfAttention.forward(Q, K, V, length) at 1..64 queries / keys  (same lines)
 *   nrms_additive_fwd/bwd       AdditiveAttention.forward at 1..64 candidates  src/model/general/attention/additive.py:27-53
 *   nrms_element_encoder_fwd/bwd, nrms_add_position_fwd/bwd
 *                               model/Exp1                                  src/model/Exp1/news_encoder.py:37-111,
 *                                                                           src/model/Exp1/user_encoder.py:15-31
 *
 * Conventions
 *   - All pointers are DEVICE pointers unless the name ends in _host.  Buffers are
 *     caller-owned (torch-allocated); the library never frees or keeps a pointer after
 *     the call returns.  All fp32 row pointers must be 16-byte aligned.
 *   - Calls are asynchronous on `stream` (a cudaStream_t passed as void*); no call syncs.
 *   - Return value: 0 = ok, nonzero = error (NRMS_E_*); text via nrms_last_error()
 *     (thread-local).  No exception crosses the ABI.  There is no CPU fallback.
 *   - Model dimensions are compile-time: D=300, H=15 (d_k=d_v=20), query dim 200
 *     (src/config.py:14-45).  Text length L is 20 (titles) or 50 (abstracts) in nrms_news_encoder_*, and any 1..64
 *     (config.num_words_title / num_words_abstract) in nrms_text_encoder_*; the user encoder's history length S
 *     (config.num_clicked_news_a_user) is any 1..64, with fused kernels at 20 and 50.
 *   - Packed weights: wqkv = rows [W_Q; W_K; W_V] -> [900,300] (nn.Linear "out,in" layout),
 *     bqkv [900], wa [200,300], ba [200], qa [200].
 */
#ifndef NRMS_B200_H
#define NRMS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NRMS_D 300
#define NRMS_H 15
#define NRMS_DH 20
#define NRMS_QD 200
#define NRMS_CE 100 /* category_embedding_dim (model/Exp1 element encoders, src/config.py:34) */

enum {
  NRMS_OK = 0,
  NRMS_E_INVALID = 1,     /* bad argument / null pointer / misaligned */
  NRMS_E_UNSUPPORTED = 2, /* shape not supported by the compiled kernels */
  NRMS_E_WORKSPACE = 3,   /* workspace / stash too small */
  NRMS_E_CUDA = 4         /* CUDA runtime error (launch failure etc.) */
};

/* arithmetic mode of the dense contractions */
enum {
  NRMS_MODE_FP32 = 0, /* CUDA-core FFMA everywhere: reference-exact fp32 (up to summation order) */
  NRMS_MODE_TF32 = 1  /* tcgen05 kind::tf32 projections (operands rounded to TF32, fp32 accumulate in TMEM) */
};

const char* nrms_last_error(void);
int nrms_abi_version(void);
/* number of CUDA kernels this library has launched in this process (bench.py's gpu_launches) */
int64_t nrms_launch_count(void);

/* Tuning / A-B switches of the tensor-mode inference encoders.
 * "user_table_attn" / "news_table_attn" (default 1): indexed calls whose gathered rows outnumber the rows of their source
 *  table "table_ratio":1 (default 4) project the TABLE once (q|k|v rows in fp16, one kind::f16 GEMM) and run the attention
 *  on gathered rows (K1g, k1g_table_attn.cu) instead of projecting every gathered row (K1 v6, tc_fused7.cu); 0 = always
 *  the per-sequence projection.
 * "fused_pool" (default 0): table path with the additive pooling inside the attention kernel (K1f, k1f_attn_pool.cu: the
 *  context rows never leave the SM; measured slower than K1g + K2, see DESIGN.md).
 * "attn_safe_softmax" (default -1): -1 = the attention kernels choose between 2^s and the row-shifted form
 *  2^(s - max) / (Z + 1e-8 * 2^-max) from a bound on the scores, 0 / 1 force one form (tests).
 * "train_attn_mma" (default 1): tensor-mode training attention of the news encoder, over titles (L = 20) and 50-token
 *  texts (L = 50), on mma.sync TF32 tiles (attn_mma.cu); 0 = the CUDA-core kernels of the FP32 mode.  The user
 *  encoder's S = 50 training attention stays on the CUDA-core kernel either way; its other history lengths (not 20)
 *  run the attention of nrms_mha_* in the call's mode.
 * "k1f_debug": component-removal timing masks of K1f (garbage results; profiles/k1f_probe.py). */
int nrms_set_option(const char* key, int value);
/* "time_k1" = 1 brackets every fused K1 launch with CUDA events on the launching stream (clears the previous
 * record); nrms_get_stat("<kind>_ms" | "<kind>_launches" | "<kind>_sequences") reads the totals back (syncs on the
 * recorded events) for kind = k1 (user encoder, per-user projection), k1n (news encoder, per-title projection), k1g (user
 * encoder, table attention), k1gn (news encoder, table attention).  Used by bench.py for the roofline of the dominant
 * kernel.  Unknown key: -1. */
double nrms_get_stat(const char* key);

/* ---- sizes ------------------------------------------------------------------------- */
/* Bytes of the saved-for-backward stash of one encoder call over n_seq sequences of length S
 * (X, QKV, C, T, w).  The same stash is written by *_fwd (when non-NULL) and read by *_bwd. */
size_t nrms_encoder_stash_bytes(int64_t n_seq, int S);
/* Scratch bytes for one encoder fwd / bwd call (mode-dependent).  n_src_rows: rows of the gather source of the
 * call (num_words for the news encoder, n_rows of the table for the indexed user encoder, 0 for dense input) --
 * the tensor-mode inference path keeps an fp16 copy of that source in the workspace. */
size_t nrms_encoder_fwd_workspace_bytes(int64_t n_seq, int S, int mode, int training, int64_t n_src_rows);
size_t nrms_encoder_bwd_workspace_bytes(int64_t n_seq, int S, int mode);

/* ---- encoders ---------------------------------------------------------------------- */
/* News encoder forward: tokens int64 [n_titles, L] -> out fp32 [n_titles, 300].
 * emb: [num_words, 300].  stash: NULL for inference, else nrms_encoder_stash_bytes bytes.
 * dropout_p in [0,1): 0 = eval mode.  (seed, offset) key the in-kernel Philox stream.
 * L = 20 (title, config.num_words_title) or 50 (a 50-token text such as Exp1's abstract), for training (stash != NULL)
 * and inference alike; any other L returns NRMS_E_UNSUPPORTED before any CUDA call. */
int nrms_news_encoder_fwd(const int64_t* tokens, int64_t n_titles, int L,
                          const float* emb, int64_t num_words,
                          const float* wqkv, const float* bqkv,
                          const float* wa, const float* ba, const float* qa,
                          float* out, void* stash,
                          void* workspace, size_t workspace_bytes,
                          float dropout_p, uint64_t seed, uint64_t offset,
                          int mode, void* stream);

/* Inference-only, tensor-mode form of the news encoder over int32 token ids (the pre-tokenised evaluate table: half the
 * host-to-device bytes of the int64 LongTensor the reference's DataLoader ships, src/evaluate.py:51-78).  Workspace:
 * nrms_encoder_fwd_workspace_bytes(n_titles, L, NRMS_MODE_TF32, 0, num_words). */
int nrms_news_encoder_i32_fwd(const int32_t* tokens, int64_t n_titles, int L,
                              const float* emb, int64_t num_words,
                              const float* wqkv, const float* bqkv,
                              const float* wa, const float* ba, const float* qa,
                              float* out, void* workspace, size_t workspace_bytes, void* stream);

/* News encoder backward (L = 20 or 50, as the forward that wrote the stash).  d_out [n_titles,300].  Gradients are
 * ACCUMULATED (+=) into
 * d_emb [num_words,300] (row 0 = padding_idx is never touched), d_wqkv [900,300],
 * d_bqkv [900], d_wa [200,300], d_ba [200], d_qa [200]. */
int nrms_news_encoder_bwd(const float* d_out, const int64_t* tokens, int64_t n_titles, int L,
                          int64_t num_words,
                          const float* wqkv, const float* wa, const float* qa,
                          const void* stash,
                          float* d_emb, float* d_wqkv, float* d_bqkv,
                          float* d_wa, float* d_ba, float* d_qa,
                          void* workspace, size_t workspace_bytes,
                          float dropout_p, uint64_t seed, uint64_t offset,
                          int mode, void* stream);

/* User encoder forward.  Input rows are either dense x [n_users, S, 300] (rows == NULL, n_rows ignored) or
 * gathered from a table: x = table [n_rows,300], rows int32 [n_users, S] with values in [0, n_rows)
 * (evaluate.py:220-224; the PADDED_NEWS zero vector is a zero row of the table).
 * S = 1..64 for every user-encoder entry point (forward, backward, LayerNorm and fp16-table forms); S outside that range
 * returns NRMS_E_UNSUPPORTED before any CUDA call.  S = 20 and 50 run the compiled kernels (in tensor-mode inference the
 * fused K1 / K2 paths); other lengths run the projection GEMM, the run-time-length attention of nrms_mha_* and the
 * additive block, chunked in inference. */
int nrms_user_encoder_fwd(const float* x, int64_t n_rows, const int32_t* rows, int64_t n_users, int S,
                          const float* wqkv, const float* bqkv,
                          const float* wa, const float* ba, const float* qa,
                          float* out, void* stash,
                          void* workspace, size_t workspace_bytes,
                          int mode, void* stream);

/* Tensor-mode, inference-only form of the indexed user encoder whose table is already held as fp16 rows: table16 =
 * [n_rows + 1][320] halfs in nrms_pack_rows_f16's layout (300 values, 1.0 in column 300, zero tail; last row all zero).
 * This is what evaluate keeps between its stages (src/evaluate.py:193-233): the news stage packs its vectors once, the
 * all-gather moves 640-byte rows, and both the user encoder and nrms_score_csr_f16 read the same copy.  At S other than
 * 20 and 50 the gathered rows are widened to fp32 and run through the tensor-mode encoder a chunk of users at a time. */
size_t nrms_user_encoder_table16_workspace_bytes(int64_t n_users, int S, int64_t n_rows);
int nrms_user_encoder_table16_fwd(const void* table16, int64_t n_rows, const int32_t* rows, int64_t n_users, int S,
                                  const float* wqkv, const float* bqkv,
                                  const float* wa, const float* ba, const float* qa,
                                  float* out, void* workspace, size_t workspace_bytes, void* stream);

/* User encoder backward (dense input only, S = 1..64 as the forward that wrote the stash).  d_x [n_users,S,300] is
 * OVERWRITTEN; weight gradients are accumulated (+=). */
int nrms_user_encoder_bwd(const float* d_out, int64_t n_users, int S,
                          const float* wqkv, const float* wa, const float* qa,
                          const void* stash,
                          float* d_x, float* d_wqkv, float* d_bqkv,
                          float* d_wa, float* d_ba, float* d_qa,
                          void* workspace, size_t workspace_bytes,
                          int mode, void* stream);

/* Standalone L0 blocks (inside the encoders they are fused; both have a backward below):
 *   nrms_mhsa_fwd      MultiHeadSelfAttention.forward(Q) with K=V=Q, length=None   multihead_self.py:46-76
 *                      x [n_seq,S,300] -> ctx [n_seq,S,300]; workspace >= n_seq*S*900*4 bytes
 *   nrms_additive_fwd  AdditiveAttention.forward                                   additive.py:27-53
 *                      c [n_seq,S,300] -> out [n_seq,300];   workspace >= n_seq*S*(200+1)*4 + 256 bytes */
int nrms_mhsa_fwd(const float* x, int64_t n_seq, int S, const float* wqkv, const float* bqkv, float* ctx,
                  void* workspace, size_t workspace_bytes, int mode, void* stream);
/* The `length` branch of MultiHeadSelfAttention.forward (multihead_self.py:60-68 builds attn_mask[b,h,i,j] =
 * j < length[b]; :18-19 multiplies exp(scores) by it): lengths int32 [n_seq]; keys at positions >= length add nothing
 * to the sum or the context of ANY query row (rows past the length are still computed, as in the reference). */
int nrms_mhsa_masked_fwd(const float* x, const int32_t* lengths, int64_t n_seq, int S, const float* wqkv,
                         const float* bqkv, float* ctx, void* workspace, size_t workspace_bytes, int mode, void* stream);
int nrms_additive_fwd(const float* c, int64_t n_seq, int S, const float* wa, const float* ba, const float* qa,
                      float* out, void* workspace, size_t workspace_bytes, int mode, void* stream);

/* MultiHeadSelfAttention backward for the standalone block (K=V=Q), with or without the `length` mask.
 * fwd_workspace = the workspace nrms_mhsa_fwd / nrms_mhsa_masked_fwd filled (QKV [n_seq*S, 900] at its start), lengths
 * the same int32 [n_seq] the forward took (NULL = no mask).  Masked keys get exactly zero dK / dV; length <= 0 leaves the
 * whole sequence out.  d_x [n_seq,S,300] is OVERWRITTEN (NULL: not computed); d_wqkv [900,300] and d_bqkv [900] are
 * accumulated into.  Tensor mode runs the attention on mma.sync TF32 tiles (nrms_set_option("train_attn_mma", 0): the
 * CUDA-core kernels of FP32 mode) and the weight and input contractions on tcgen05. */
size_t nrms_mhsa_bwd_workspace_bytes(int64_t n_seq, int S, int mode);
int nrms_mhsa_bwd(const float* d_ctx, const float* x, const int32_t* lengths, int64_t n_seq, int S, const float* wqkv,
                  const void* fwd_workspace, float* d_x, float* d_wqkv, float* d_bqkv, void* workspace,
                  size_t workspace_bytes, int mode, void* stream);

/* MultiHeadSelfAttention.forward(Q, K, V, length) at any 1 <= Sq, Sk <= 64: cross-attention (K and / or V other inputs
 * than Q) and self-attention at lengths other than 20 and 50.  xq [n_seq,Sq,300], xk and xv [n_seq,Sk,300]; pass the
 * same pointer for the same input (K = Q, K = V, ...): each input is projected onto the rows of wqkv it needs, once
 * when its roles' rows are adjacent (Q = V with K another input takes two 300-row projections).  Distinct inputs must
 * be distinct pointers: two pointers that are equal are one input.  ctx [n_seq,Sq,300].  lengths (int32 [n_seq], NULL = no mask) is the reference's `length`: with Sq == Sk the
 * keys j < length[b] are kept; with Sq == 1 < Sk the reference's [B,H,1,1] mask broadcasts, so all keys are kept iff
 * length[b] >= 1; any other Sq != Sk with lengths -> NRMS_E_UNSUPPORTED.  length <= 0 gives a zero context.
 * Tensor mode: projections on tcgen05, attention on mma.sync TF32 tiles; FP32 mode: CUDA cores throughout.
 * The forward workspace keeps the projections; it is what nrms_mha_bwd reads (the same inputs, shapes and lengths).
 * Backward: d_xq / d_xk / d_xv are OVERWRITTEN (NULL: not computed).  When two inputs are the same pointer their gradient
 * pointers must be equal or NULL, and that buffer receives the sum; gradients of distinct inputs must be distinct
 * buffers, and none may be an input (NRMS_E_INVALID).  d_wqkv [900,300] and d_bqkv [900] are accumulated into.
 * Masked keys get exactly zero dK / dV rows.  Arguments are checked before any CUDA call: Sq or Sk outside 1..64 ->
 * NRMS_E_UNSUPPORTED, null or misaligned pointers (the workspace included) -> NRMS_E_INVALID, a null or short
 * workspace -> NRMS_E_WORKSPACE. */
size_t nrms_mha_fwd_workspace_bytes(int64_t n_seq, int Sq, int Sk);
int nrms_mha_fwd(const float* xq, const float* xk, const float* xv, int64_t n_seq, int Sq, int Sk, const int32_t* lengths,
                 const float* wqkv, const float* bqkv, float* ctx, void* workspace, size_t workspace_bytes, int mode,
                 void* stream);
size_t nrms_mha_bwd_workspace_bytes(int64_t n_seq, int Sq, int Sk, int mode);
int nrms_mha_bwd(const float* d_ctx, const float* xq, const float* xk, const float* xv, int64_t n_seq, int Sq, int Sk,
                 const int32_t* lengths, const float* wqkv, const void* fwd_workspace, float* d_xq, float* d_xk,
                 float* d_xv, float* d_wqkv, float* d_bqkv, void* workspace, size_t workspace_bytes, int mode,
                 void* stream);

/* AdditiveAttention backward for the standalone block.  nrms_additive_fwd accepts 1 <= S <= 64 (2..4: the final attention
 * over the element vectors of model/Exp1, src/model/Exp1/news_encoder.py:104-110).  S < 20 runs its linear map on the
 * CUDA cores in either mode.  fwd_workspace = the workspace the forward call filled (tanh activations | softmax weights).  d_c [n_seq,S,300]
 * is OVERWRITTEN; d_wa [200,300], d_ba [200], d_qa [200] are accumulated into. */
size_t nrms_additive_bwd_workspace_bytes(int64_t n_seq, int S, int mode);
int nrms_additive_bwd(const float* d_out, const float* c, int64_t n_seq, int S, const float* wa, const float* qa,
                      const void* fwd_workspace, float* d_c, float* d_wa, float* d_ba, float* d_qa, void* workspace,
                      size_t workspace_bytes, int mode, void* stream);

/* ---- index-only training minibatch (SURVEY 8 f2) ----------------------------------------
 * The reference DataLoader ships 1+K+50 token tensors per step (src/dataset.py:17-85, src/train.py:118-124); here the
 * pre-tokenised news table int64 [n_news, L] lives on the device and a minibatch is news-row indices: title t of the call
 * is row news_rows[t] (int64, in [0, n_news)) of token_table, gathered inside the embedding gather / gradient scatter
 * kernels.  Training form only (stash required); ln_* NULL = plain NRMS, else the config-5 variant.  L = 20 or 50.
 * Stash / workspace sizes and the gradient contract are those of nrms_news_encoder_fwd / _bwd. */
int nrms_news_encoder_rows_fwd(const int64_t* token_table, int64_t n_news, const int64_t* news_rows, int64_t n_titles,
                               int L, const float* emb, int64_t num_words, const float* wqkv, const float* bqkv,
                               const float* ln_gamma, const float* ln_beta, const float* wa, const float* ba,
                               const float* qa, float* out, void* stash, float dropout_p, uint64_t seed, uint64_t offset,
                               int mode, void* stream);
int nrms_news_encoder_rows_bwd(const float* d_out, const int64_t* token_table, int64_t n_news, const int64_t* news_rows,
                               int64_t n_titles, int L, int64_t num_words, const float* wqkv, const float* ln_gamma,
                               const float* wa, const float* qa, const void* stash, float* d_emb, float* d_wqkv,
                               float* d_bqkv, float* d_ln_gamma, float* d_ln_beta, float* d_wa, float* d_ba, float* d_qa,
                               void* workspace, size_t workspace_bytes, float dropout_p, uint64_t seed, uint64_t offset,
                               int mode, void* stream);

/* ---- text encoder at any length 1..64 --------------------------------------------------------
 * The news encoder (src/model/NRMS/news_encoder.py:27-48; Exp1's TextEncoder, src/model/Exp1/news_encoder.py:10-34) at
 * any title / abstract length L = 1..64: the reference pads and truncates every text to BaseConfig.num_words_title /
 * num_words_abstract (src/data_preprocess.py:115,132-139), so L is a setting.  One pair for every form:
 *   - news_rows NULL: dense tokens int64 [n_token_rows, L], text t = row t (n_token_rows >= n_texts);
 *     news_rows non-NULL: index-only minibatch (as nrms_news_encoder_rows_*), text t = row news_rows[t] of the
 *     [n_token_rows, L] table -- training only (stash required);
 *   - ln_gamma / ln_beta both NULL (reference NRMS) or both given (config-5 LayerNorm); the backward takes ln_gamma and
 *     d_ln_gamma / d_ln_beta;
 *   - stash non-NULL: training (nrms_encoder_stash_bytes / nrms_encoder_ln_stash_bytes); NULL: inference, with
 *     workspace = nrms_encoder_fwd_workspace_bytes(n_texts, L, mode, 0, num_words).  The backward's workspace is
 *     nrms_encoder_bwd_workspace_bytes(n_texts, L, mode).
 * Both dropout sites (:38-45) draw the Philox stream of nrms_news_encoder_fwd: element e of the [rows, 300] activation
 * keeps counter e / 4 + offset, so a text's masks depend only on its row, and a chunked inference pass equals a single
 * one.  L outside 1..64 returns NRMS_E_UNSUPPORTED before any pointer check and before any CUDA call; then each form is
 * checked as its nrms_news_encoder_* counterpart.  L = 20 and 50 run exactly what nrms_news_encoder_* run; other lengths
 * run the attention of nrms_mha_* with dropout #2 applied inside it, and the run-time-length additive kernels (inference
 * takes the chunked path: the fused inference kernels are compiled for 20 and 50 only).  Gradients are ACCUMULATED as in
 * nrms_news_encoder_bwd. */
int nrms_text_encoder_fwd(const int64_t* tokens, int64_t n_token_rows, const int64_t* news_rows, int64_t n_texts, int L,
                          const float* emb, int64_t num_words, const float* wqkv, const float* bqkv,
                          const float* ln_gamma, const float* ln_beta, const float* wa, const float* ba, const float* qa,
                          float* out, void* stash, void* workspace, size_t workspace_bytes, float dropout_p,
                          uint64_t seed, uint64_t offset, int mode, void* stream);
int nrms_text_encoder_bwd(const float* d_out, const int64_t* tokens, int64_t n_token_rows, const int64_t* news_rows,
                          int64_t n_texts, int L, int64_t num_words, const float* wqkv, const float* ln_gamma,
                          const float* wa, const float* qa, const void* stash, float* d_emb, float* d_wqkv,
                          float* d_bqkv, float* d_ln_gamma, float* d_ln_beta, float* d_wa, float* d_ba, float* d_qa,
                          void* workspace, size_t workspace_bytes, float dropout_p, uint64_t seed, uint64_t offset,
                          int mode, void* stream);

/* ---- model/Exp1 blocks (SURVEY 8 f3) ------------------------------------------------------
 * ElementEncoder.forward = relu(linear(embedding(element)))  (src/model/Exp1/news_encoder.py:37-44):
 * idx int64 [n] in [0, num_categories), emb [num_categories, 100], w [300, 100], b [300] -> out [n, 300].
 * `table` ([num_categories, 300], nrms_element_encoder_table_bytes) receives relu(W emb^T + b) for every category -- the
 * linear layer runs over the vocabulary once, the per-element work is a row gather -- and is what the backward reads.
 * Backward accumulates into d_emb (row 0 = padding_idx untouched), d_w, d_b; workspace = table bytes. */
size_t nrms_element_encoder_table_bytes(int64_t num_categories);
int nrms_element_encoder_fwd(const int64_t* idx, int64_t n, const float* emb, int64_t num_categories, const float* w,
                             const float* b, float* out, void* table, void* stream);
int nrms_element_encoder_bwd(const float* d_out, const int64_t* idx, int64_t n, const float* emb, int64_t num_categories,
                             const float* w, const void* table, float* d_emb, float* d_w, float* d_b, void* workspace,
                             size_t workspace_bytes, void* stream);
/* out[u,i,:] = x[u,i,:] + pos[i,:]  (user_vector + position_embedding, src/model/Exp1/user_encoder.py:25-26);
 * backward: d_pos [S,300] += sum_u d_out[u,:,:]  (d_x = d_out). */
int nrms_add_position_fwd(const float* x, const float* pos, int64_t n_users, int S, float* out, void* stream);
size_t nrms_add_position_bwd_workspace_bytes(int S);
int nrms_add_position_bwd(const float* d_out, int64_t n_users, int S, float* d_pos, void* workspace,
                          size_t workspace_bytes, void* stream);
/* dst[r*dst_stride .. +width) = src[r*src_stride .. +width): torch.stack(all_vectors, dim=1) and its backward
 * (src/model/Exp1/news_encoder.py:109); strides and width in floats, multiples of 4. */
int nrms_copy_rows_strided(const float* src, int64_t src_stride, float* dst, int64_t dst_stride, int64_t n, int width,
                           void* stream);

/* ---- single-user latency path (SURVEY 8 f4; src/recommend.py:245-341) ---------------------
 * One user, two cluster launches: user_vec [300] = UserEncoder(table[hist_rows[0..50)]), scores[c] = table[cand_rows[c]] .
 * user_vec, order = candidate positions by descending score (equal scores in ascending position, -0 == +0; NaN scores
 * after every number, -inf included, in ascending position: np.argsort(-y) of recommend.py:339 on a stable sort).
 * table fp32 [n_rows, 300] (the news2vector cache, PADDED_NEWS = a zero row);
 * hist_rows int32 [50] and cand_rows int32 [C] are DEVICE arrays with values in [0, n_rows) (an out-of-range value
 * reads row n_rows - 1).  order may be NULL (scores only); with order, C <= 4096.  FP32 arithmetic. */
size_t nrms_recommend_workspace_bytes(void);
int nrms_recommend_user(const float* table, int64_t n_rows, const int32_t* hist_rows, const int32_t* cand_rows, int C,
                        const float* wqkv, const float* bqkv, const float* wa, const float* ba, const float* qa,
                        float* user_vec, float* scores, int32_t* order, void* workspace, size_t workspace_bytes,
                        void* stream);

/* ---- top-k news of the whole table per user ------------------------------------------
 * The ranking of src/recommend.py:338-340 (np.argsort(-y) over the candidates the caller passes) generalised to every
 * row of the news table: for each user u, top_rows[u, 0..k) are the k rows of [0, n_news) with the highest score
 * table[row] . user_vec[u], and top_scores[u, j] is that score.
 *   - Order: score descending, equal scores by row ascending (the rule of nrms_recommend_user), so the result is unique
 *     and does not depend on the launch configuration.  -0 and +0 are equal scores.  A NaN score ranks below every number
 *     and is never returned.  When fewer than k rows remain, the tail is row -1, score -inf.  1 <= k <= 256.
 *   - mode NRMS_MODE_TF32: `table` is the fp16 copy in nrms_pack_rows_f16's layout (rows of 320 halfs); user_vec is rounded
 *     to fp16 and the dot products run on the tensor cores (tcgen05 kind::f16, fp32 accumulation).
 *     mode NRMS_MODE_FP32: `table` is fp32 [>= n_news, 300]; CUDA-core fp32 dot products.
 *     Only rows [0, n_news) are candidates: rows past it (evaluate's PADDED_NEWS replicas, the closing zero row of the fp16
 *     copy) are never read as candidates.
 *   - user_vec fp32 [n_users, 300].  exclude_rows int32 [n_users, n_exclude] (n_exclude <= 64) or NULL: those rows are
 *     never returned for that user -- the intended input is the history rows [n_users, 50].  Entries outside [0, n_news)
 *     are ignored (the pads), duplicates are harmless.
 *   - Outputs top_scores fp32 [n_users, k], top_rows int32 [n_users, k].
 *   - Asynchronous, no host sync, no allocation.  The workspace (nrms_topk_workspace_bytes; 0 for arguments the call
 *     rejects) grows with n_users * (k + n_exclude) and the number of news splits, never with n_users * n_news.
 *   - Arguments are checked before any CUDA call: k out of range or n_exclude > 64 -> NRMS_E_UNSUPPORTED; null or
 *     misaligned pointers (table / user_vec 16 bytes, workspace 256 bytes) -> NRMS_E_INVALID. */
size_t nrms_topk_workspace_bytes(int64_t n_users, int64_t n_news, int k, int n_exclude, int mode);
int nrms_topk_news(const void* table, int64_t n_news, const float* user_vec, int64_t n_users,
                   const int32_t* exclude_rows, int n_exclude, int k,
                   float* top_scores, int32_t* top_rows,
                   void* workspace, size_t workspace_bytes, int mode, void* stream);

/* ---- click predictor --------------------------------------------------------------- */
/* scores[b,c] = cand[b,c,:] . user[b,:]     cand [B,C,X], user [B,X] */
int nrms_score_fwd(const float* cand, const float* user, int64_t B, int C, int X,
                   float* scores, void* stream);
/* d_cand [B,C,X] and d_user [B,X] are overwritten. */
int nrms_score_bwd(const float* d_scores, const float* cand, const float* user,
                   int64_t B, int C, int X, float* d_cand, float* d_user, void* stream);
/* CSR form used by evaluate: impression i owns candidates [offsets[i], offsets[i+1]);
 * scores[k] = table[cand_rows[k], :] . user_vec[i, :]   (X = 300). */
int nrms_score_csr(const float* table, const int32_t* cand_rows, const int64_t* offsets,
                   const float* user_vec, int64_t n_impressions, float* scores, void* stream);
/* Tensor-mode scoring: the candidate rows are read from an fp16 copy of the table (half the bytes per candidate, fp32
 * accumulation).  nrms_pack_rows_f16 writes that copy: dst16 = (n_rows + 1) * 640 bytes, rows of 320 halfs. */
int nrms_pack_rows_f16(const float* src, int64_t n_rows, void* dst16, void* stream);
int nrms_score_csr_f16(const void* table16, const int32_t* cand_rows, const int64_t* offsets,
                       const float* user_vec, int64_t n_impressions, float* scores, void* stream);

/* ---- loss / optimizer --------------------------------------------------------------- */
/* loss = mean_b( -log_softmax(logits[b,:])[0] ); d_logits = d(loss)/d(logits) * grad_scale. */
int nrms_ce_loss_fwd_bwd(const float* logits, int64_t B, int C, float grad_scale,
                         float* loss, float* d_logits, void* stream);
/* One Adam/AdamW update over n contiguous elements.  step is 1-based.  grad_scale multiplies
 * g first (1/world_size for data-parallel averaging).  decoupled=1 -> AdamW. */
int nrms_adam_step(float* p, const float* g, float* m, float* v, int64_t n,
                   float lr, float beta1, float beta2, float eps, float weight_decay,
                   int decoupled, int64_t step, float grad_scale, void* stream);

/* ---- evaluate helpers ---------------------------------------------------------------- */
/* Row gather: dst[i,:] = src[rows[i],:] (width floats per row, width % 4 == 0). */
int nrms_gather_rows(const float* src, const int64_t* rows, int64_t n, int width,
                     float* dst, void* stream);
/* Per-impression AUC / MRR / nDCG@5 / nDCG@10 (fp64) on CSR (labels int8 in {0,1});
 * single-class impressions give NaN x4.  per_impression [n,4] (required when n > 0);
 * sums_counts [8] = {sum auc, mrr, ndcg5, ndcg10, count auc, mrr, ndcg5, ndcg10} over non-NaN
 * rows (nanmean numerators/denominators), overwritten. */
int nrms_rank_metrics(const float* scores, const int8_t* labels, const int64_t* offsets,
                      int64_t n_impressions, double* per_impression, double* sums_counts,
                      void* stream);

/* ---- generic dense contraction (exposed for tests / profiling) ---------------------- */
/* C[M,N] = A[M,K] * B[N,K]^T (+ bias[N] if non-NULL); row-major, lda/ldb/ldc in floats. */
int nrms_gemm_nt(const float* A, int64_t lda, const float* B, int64_t ldb, const float* bias,
                 float* C, int64_t ldc, int64_t M, int N, int K, int mode, void* stream);

/* ---- config-5 variant: LayerNorm(300) between the self-attention context and the additive block ------------
 * The reference tree has no code for its "+LN +AdamW +cosine" row (README.md:105-112); the definition used here is
 * builder-defined (DESIGN.md section 1): c = LayerNorm(dropout(MHSA(x))) with torch semantics (biased variance,
 * eps 1e-5, affine weight/bias [300]) in BOTH encoders, then AdditiveAttention(c).  Same contracts as the entry
 * points above; the stash of a training forward is nrms_encoder_ln_stash_bytes bytes.  d_ln_gamma / d_ln_beta are
 * accumulated into (zero them first), like the other gradient outputs. */
size_t nrms_encoder_ln_stash_bytes(int64_t n_seq, int S);
int nrms_news_encoder_ln_fwd(const int64_t* tokens, int64_t n_titles, int L,
                             const float* emb, int64_t num_words,
                             const float* wqkv, const float* bqkv,
                             const float* ln_gamma, const float* ln_beta,
                             const float* wa, const float* ba, const float* qa,
                             float* out, void* stash,
                             void* workspace, size_t workspace_bytes,
                             float dropout_p, uint64_t seed, uint64_t offset,
                             int mode, void* stream);
int nrms_news_encoder_ln_bwd(const float* d_out, const int64_t* tokens, int64_t n_titles, int L, int64_t num_words,
                             const float* wqkv, const float* ln_gamma, const float* wa, const float* qa,
                             const void* stash,
                             float* d_emb, float* d_wqkv, float* d_bqkv, float* d_ln_gamma, float* d_ln_beta,
                             float* d_wa, float* d_ba, float* d_qa,
                             void* workspace, size_t workspace_bytes,
                             float dropout_p, uint64_t seed, uint64_t offset,
                             int mode, void* stream);
int nrms_user_encoder_ln_fwd(const float* x, int64_t n_rows, const int32_t* rows_idx, int64_t n_users, int S,
                             const float* wqkv, const float* bqkv,
                             const float* ln_gamma, const float* ln_beta,
                             const float* wa, const float* ba, const float* qa,
                             float* out, void* stash,
                             void* workspace, size_t workspace_bytes,
                             int mode, void* stream);
int nrms_user_encoder_ln_bwd(const float* d_out, int64_t n_users, int S,
                             const float* wqkv, const float* ln_gamma, const float* wa, const float* qa,
                             const void* stash,
                             float* d_x, float* d_wqkv, float* d_bqkv, float* d_ln_gamma, float* d_ln_beta,
                             float* d_wa, float* d_ba, float* d_qa,
                             void* workspace, size_t workspace_bytes,
                             int mode, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NRMS_B200_H */
