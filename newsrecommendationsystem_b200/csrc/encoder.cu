// Host side of the encoder entry points (C-ABI): argument checks, stash/workspace carving and
// the launch sequence.  Kernels live in encoder_kernels.cuh / sgemm.cuh / tc_gemm.cuh.
#include <string.h>
#include "common.cuh"
#include "encoder_kernels.cuh"
#include "sgemm.cuh"
#include "tc_api.cuh"

namespace nrms {

// ---- stash layout: X [rows,300] | QKV [rows,900] | C [rows,300] | T [rows,200] | w [rows] ----
// LayerNorm variant (config 5): + CN [rows,300] (normalised context, the additive block's input) | stats [rows,2]
struct Stash {
  float *x, *qkv, *c, *t, *w, *cn, *stats;
  size_t bytes;
};
// optional LayerNorm between the self-attention context and the additive block (nullptr = reference NRMS)
struct LnArgs {
  const float* gamma;
  const float* beta;
  float* d_gamma;
  float* d_beta;
};
constexpr float LN_EPS = 1e-5f;    // torch.nn.LayerNorm default
static Stash carve_stash(void* base, int64_t rows, bool ln = false) {
  Stash s;
  char* p = reinterpret_cast<char*>(base);
  size_t off = 0;
  auto take = [&](size_t nfloat) {
    float* r = reinterpret_cast<float*>(p + off);
    off += align_up(nfloat * sizeof(float), 256);
    return r;
  };
  s.x = take((size_t)rows * D);
  s.qkv = take((size_t)rows * D3);
  s.c = take((size_t)rows * D);
  s.t = take((size_t)rows * QD);
  s.w = take((size_t)rows);
  s.cn = ln ? take((size_t)rows * D) : nullptr;
  s.stats = ln ? take((size_t)rows * 2) : nullptr;
  s.bytes = off;
  return s;
}

static bool g_train_attn_mma = true;   // nrms_set_option("train_attn_mma"): tensor-mode news-encoder training attention
                                       // (titles and 50-token texts) on mma.sync tiles
constexpr int64_t INFER_CHUNK_ROWS = 2048 * 20;  // rows processed per pass in inference (reference batch 2048 titles)
constexpr int REDUCE_BLOCKS = 296;

// Tensor mode adds the transposed operand copies of the weight-gradient GEMMs (see encoder_core_bwd):
// t1 [900, ldr] | t2 [300, ldr] (ldr = rows rounded up to 4) | wt [300, 900].
struct BwdWs {
  float *d_c, *d_u, *d_qkv, *d_x, *partial, *t1, *t2, *wt;
  int64_t ldr;
  size_t bytes;
};
static BwdWs carve_bwd(void* base, int64_t rows, bool need_dx, int mode) {
  BwdWs s;
  char* p = reinterpret_cast<char*>(base);
  size_t off = 0;
  auto take = [&](size_t nfloat) {
    float* r = reinterpret_cast<float*>(p + off);
    off += align_up(nfloat * sizeof(float), 256);
    return r;
  };
  s.d_c = take((size_t)rows * D);
  s.d_u = take((size_t)rows * QD);
  s.d_qkv = take((size_t)rows * D3);
  s.d_x = need_dx ? take((size_t)rows * D) : nullptr;
  s.partial = take((size_t)REDUCE_BLOCKS * D3);
  s.ldr = (rows + 3) / 4 * 4;
  s.t1 = s.t2 = s.wt = nullptr;
  if (mode == NRMS_MODE_TF32) {
    s.t1 = take((size_t)s.ldr * D3);
    s.t2 = take((size_t)s.ldr * D);
    s.wt = take((size_t)D3 * D);
  }
  s.bytes = off;
  return s;
}

template <int S, int HC>
static cudaError_t launch_attention_fwd(const float* qkv, float* ctx, int64_t n_seq, float p, uint64_t seed,
                                        uint64_t offset, cudaStream_t st, const int32_t* lengths = nullptr) {
  constexpr int threads = ((S * HC + 31) / 32) * 32;
  const size_t smem = 2 * S * HC * DH * sizeof(float);
  static bool configured[64] = {false};
  if (cudaError_t e = set_max_dynamic_smem(attention_fwd_kernel<S, HC>, (int)smem, configured)) return e;
  int64_t gx = n_seq < (int64_t)num_sms() * 8 ? n_seq : (int64_t)num_sms() * 8;
  dim3 grid((unsigned)gx, H / HC);
  const float scale = p > 0.f ? 1.f / (1.f - p) : 1.f;
  attention_fwd_kernel<S, HC><<<grid, threads, smem, st>>>(qkv, ctx, n_seq, p, scale, seed, offset, lengths);
  count_launch();
  return cudaGetLastError();
}

template <int S, int HC, bool MASKED = false>
static cudaError_t launch_attention_bwd(const float* qkv, const float* d_ctx, float* d_qkv, int64_t n_seq, float p,
                                        uint64_t seed, uint64_t offset, cudaStream_t st, const int32_t* lengths = nullptr) {
  constexpr int threads = ((S * HC + 31) / 32) * 32;
  const size_t smem = (4 * S * HC * DH + 2 * HC * S * (S + 1)) * sizeof(float);
  static bool configured[64] = {false};
  if (cudaError_t e = set_max_dynamic_smem(attention_bwd_kernel<S, HC, MASKED>, (int)smem, configured)) return e;
  int64_t gx = n_seq < (int64_t)num_sms() * 4 ? n_seq : (int64_t)num_sms() * 4;
  dim3 grid((unsigned)gx, H / HC);
  const float scale = p > 0.f ? 1.f / (1.f - p) : 1.f;
  attention_bwd_kernel<S, HC, MASKED><<<grid, threads, smem, st>>>(qkv, d_ctx, d_qkv, n_seq, p, scale, seed, offset, lengths);
  count_launch();
  return cudaGetLastError();
}

static int gemm_nt_bias(const float* A, int64_t lda, const float* B, int64_t ldb, const float* bias, float* C,
                        int64_t ldc, int64_t M, int N, int K, int mode, cudaStream_t st) {
  if (mode == NRMS_MODE_TF32) return tc_gemm_nt(A, lda, B, ldb, bias, C, ldc, M, N, K, st);
  cudaError_t e = sgemm_launch<0, 0, EPI_STORE>(A, lda, B, ldb, bias, C, ldc, M, N, K, 1, st);
  if (e != cudaSuccess) return cuda_fail(e, "sgemm_nt");
  return NRMS_OK;
}

// additive pooling kernels: compiled for 20 (titles), 50 (history / abstracts) and 2..4 (the final attention over the
// element vectors of model/Exp1, reference src/model/Exp1/news_encoder.py:106-110); every other length up to 64 (user
// histories of another num_clicked_news_a_user, standalone blocks) takes the run-time-length kernels
static bool additive_len_ok(int S) { return S >= 1 && S <= ADD_MAXS; }
static cudaError_t launch_additive_fwd(const float* cin, float* t, const float* qa, float* wv, float* out, int64_t n_seq,
                                       int S, cudaStream_t st) {
  const unsigned gx = (unsigned)(n_seq < (int64_t)num_sms() * 8 ? n_seq : (int64_t)num_sms() * 8);
  switch (S) {
    case 20: additive_fwd_kernel<20><<<gx, 256, 0, st>>>(cin, t, qa, wv, out, n_seq); break;
    case 50: additive_fwd_kernel<50><<<gx, 256, 0, st>>>(cin, t, qa, wv, out, n_seq); break;
    case 2: additive_fwd_kernel<2><<<gx, 256, 0, st>>>(cin, t, qa, wv, out, n_seq); break;
    case 3: additive_fwd_kernel<3><<<gx, 256, 0, st>>>(cin, t, qa, wv, out, n_seq); break;
    case 4: additive_fwd_kernel<4><<<gx, 256, 0, st>>>(cin, t, qa, wv, out, n_seq); break;
    default: additive_fwd_rt_kernel<<<gx, 256, 0, st>>>(cin, t, qa, wv, out, n_seq, S); break;
  }
  count_launch();
  return cudaGetLastError();
}
static cudaError_t launch_additive_bwd(const float* d_out, const float* cin, const float* t, const float* wv,
                                       const float* qa, float* d_c, float* d_u, float* partial, int64_t n_seq, int S,
                                       int nb, cudaStream_t st) {
  switch (S) {
    case 20: additive_bwd_kernel<20><<<nb, 256, 0, st>>>(d_out, cin, t, wv, qa, d_c, d_u, partial, n_seq); break;
    case 50: additive_bwd_kernel<50><<<nb, 256, 0, st>>>(d_out, cin, t, wv, qa, d_c, d_u, partial, n_seq); break;
    case 2: additive_bwd_kernel<2><<<nb, 256, 0, st>>>(d_out, cin, t, wv, qa, d_c, d_u, partial, n_seq); break;
    case 3: additive_bwd_kernel<3><<<nb, 256, 0, st>>>(d_out, cin, t, wv, qa, d_c, d_u, partial, n_seq); break;
    case 4: additive_bwd_kernel<4><<<nb, 256, 0, st>>>(d_out, cin, t, wv, qa, d_c, d_u, partial, n_seq); break;
    default: additive_bwd_rt_kernel<<<nb, 256, 0, st>>>(d_out, cin, t, wv, qa, d_c, d_u, partial, n_seq, S); break;
  }
  count_launch();
  return cudaGetLastError();
}

// Forward over `n_seq` sequences whose input rows X are already materialised in st.x.  text_train: the news encoder's
// training form -- in tensor mode its 50-token texts take the mma.sync attention; every other S = 50 caller (the user
// encoder, inference) keeps the CUDA-core kernel.
static int encoder_core_fwd(const Stash& s, int64_t n_seq, int S, const float* wqkv, const float* bqkv,
                            const float* wa, const float* ba, const float* qa, float* out, float p2,
                            uint64_t seed, uint64_t offset, int64_t row_base, int mode, cudaStream_t st,
                            const LnArgs* ln = nullptr, bool text_train = false) {
  const int64_t rows = n_seq * S;
  int rc = gemm_nt_bias(s.x, D, wqkv, D, bqkv, s.qkv, D3, rows, D3, D, mode, st);
  if (rc) return rc;
  // dropout #2 mask indices are global row indices: offset the Philox counter by row_base*D/4
  const uint64_t off2 = offset + (uint64_t)row_base * D / 4;
  cudaError_t e;
  if (S == 20 && mode == NRMS_MODE_TF32 && g_train_attn_mma) {
    // tensor mode, titles: exp-softmax attention on mma.sync TF32 tiles (attn_mma.cu)
    if (int rc2 = attn_mma_fwd(s.qkv, s.c, n_seq, p2, seed, off2, st)) return rc2;
    e = cudaSuccess;
  } else if (S == 50 && text_train && mode == NRMS_MODE_TF32 && g_train_attn_mma) {
    if (int rc2 = attn_mma50_fwd(s.qkv, s.c, n_seq, p2, seed, off2, st)) return rc2;
    e = cudaSuccess;
  } else if (S == 20) e = launch_attention_fwd<20, 15>(s.qkv, s.c, n_seq, p2, seed, off2, st);
  else if (S == 50) e = launch_attention_fwd<50, 5>(s.qkv, s.c, n_seq, p2, seed, off2, st);
  else {
    // every other length (1..64: user histories, texts of nrms_text_encoder_*): the run-time-length attention of
    // attn_cross.cu over the stash's q|k|v rows, in the call's mode, with dropout #2 when p2 > 0
    const MhaOperands op{s.qkv, s.qkv + D, s.qkv + 2 * D, D3, D3, D3};
    if (int rc2 = mha_attn_fwd(op, s.c, n_seq, S, S, nullptr, mode, st, p2, seed, off2)) return rc2;
    e = cudaSuccess;
  }
  if (e != cudaSuccess) return cuda_fail(e, "attention_fwd");
  const float* cin = s.c;
  if (ln) {
    int64_t lb = (rows + 7) / 8;
    if (lb > (int64_t)num_sms() * 8) lb = (int64_t)num_sms() * 8;
    layernorm_fwd_kernel<<<(unsigned)lb, 256, 0, st>>>(s.c, ln->gamma, ln->beta, s.cn, s.stats, rows, LN_EPS);
    NRMS_LAUNCH_CHECK("layernorm_fwd");
    cin = s.cn;
  }
  rc = gemm_nt_bias(cin, D, wa, D, ba, s.t, QD, rows, QD, D, mode, st);
  if (rc) return rc;
  if (cudaError_t e2 = launch_additive_fwd(cin, s.t, qa, s.w, out, n_seq, S, st)) return cuda_fail(e2, "additive_fwd");
  return NRMS_OK;
}

// Backward of the additive block (additive.py:27-53) over n_seq sequences of S rows: cin = its input rows, t / wv = the
// tanh activations and softmax weights its forward saved.  d_c [rows,300] is OVERWRITTEN with dL/d(cin); d_wa, d_ba,
// d_qa are accumulated into.  Tensor mode (S = 20 / 50 only) needs the transposed operand copies t1 / t2 / wt.
struct AddBwdWs {
  float *d_u, *partial, *t1, *t2, *wt;
  int64_t ldr;
};
static int additive_block_bwd(const float* d_out, const float* cin, const float* t, const float* wv, const float* wa,
                              const float* qa, float* d_c, const AddBwdWs& w, int64_t n_seq, int S, float* d_wa,
                              float* d_ba, float* d_qa, bool tc, cudaStream_t st) {
  const int64_t rows = n_seq * S;
  // 4 CTAs per SM; the partial buffer (REDUCE_BLOCKS x 900 floats) holds two 200-wide blocks per CTA
  constexpr int ADD_BWD_BLOCKS = 592;
  static_assert(2 * ADD_BWD_BLOCKS * QD <= REDUCE_BLOCKS * D3, "partial buffer too small");
  int nb = (int)(n_seq < ADD_BWD_BLOCKS ? n_seq : ADD_BWD_BLOCKS);
  if (cudaError_t e2 = launch_additive_bwd(d_out, cin, t, wv, qa, d_c, w.d_u, w.partial, n_seq, S, nb, st))
    return cuda_fail(e2, "additive_bwd");
  launch_partial_reduce_accum(w.partial, nb, QD, QD, d_qa, st);
  NRMS_LAUNCH_CHECK("dqa_reduce");
  // d_ba = colsum(dU): per-thread sums inside additive_bwd_kernel, second block of the partial buffer
  launch_partial_reduce_accum(w.partial + (size_t)nb * QD, nb, QD, QD, d_ba, st);
  NRMS_LAUNCH_CHECK("dba_reduce");
  int splits = (int)((rows + 4095) / 4096);
  if (splits > 64) splits = 64;
  if (tc) {
    // d_wa[200,300] += dU^T C
    if (int rc = transpose_f32(w.d_u, QD, w.t1, w.ldr, rows, QD, st)) return rc;
    if (int rc = transpose_f32(cin, D, w.t2, w.ldr, rows, D, st)) return rc;
    if (int rc = tc_gemm_nt_ex(w.t1, w.ldr, w.t2, w.ldr, nullptr, d_wa, D, QD, D, (int)rows,
                               tc_gemm_auto_splits(QD, D, (int)rows), TC_EPI_ATOMIC, st)) return rc;
    // d_c += dU * Wa
    if (int rc = transpose_f32(wa, D, w.wt, QD, QD, D, st)) return rc;
    if (int rc = tc_gemm_nt_ex(w.d_u, QD, w.wt, QD, nullptr, d_c, D, rows, D, QD, 1, TC_EPI_ACCUM, st)) return rc;
  } else {
    // d_wa[200,300] += dU^T C   (reduction over rows, split-K + fp32 atomics)
    cudaError_t e = sgemm_launch<1, 1, EPI_ATOMIC>(w.d_u, QD, cin, D, nullptr, d_wa, D, QD, D, rows, splits, st);
    if (e != cudaSuccess) return cuda_fail(e, "sgemm dWa");
    // d_c += dU * Wa   ([rows,200] x [200,300])
    e = sgemm_launch<0, 1, EPI_ACCUM>(w.d_u, QD, wa, D, nullptr, d_c, D, rows, D, QD, 1, st);
    if (e != cudaSuccess) return cuda_fail(e, "sgemm dC");
  }
  return NRMS_OK;
}

// Backward of the q|k|v projection QKV = X Wqkv^T + bqkv from dQKV [rows,900], shared by the encoders and the
// standalone attention block: d_bqkv += colsum(dQKV), d_wqkv += dQKV^T X, d_x = dQKV Wqkv (skipped when d_x is
// null).  Tensor mode takes the transposed operands from t1 / t2 / wt (t1 = dQKV^T already when dqkv_t_written).
// ncols < 900: the projection onto a contiguous slice of rows of Wqkv (wqkv, d_wqkv and d_bqkv point at the slice, dQKV
// is [rows, ncols]) -- the standalone block projects each input onto the rows it needs (nrms_mha_bwd).  accum_dx: d_x +=
// instead of d_x = (the second projection of an input the block projects twice).
struct QkvBwdWs {
  float *d_qkv, *partial, *t1, *t2, *wt;
  int64_t ldr;
};
static int qkv_proj_bwd(const QkvBwdWs& w, const float* x, const float* wqkv, int64_t rows, float* d_x, float* d_wqkv,
                        float* d_bqkv, bool tc, bool dqkv_t_written, cudaStream_t st, int ncols = D3,
                        bool accum_dx = false) {
  int cb = (int)(rows < REDUCE_BLOCKS ? rows : REDUCE_BLOCKS);
  int splits = (int)((rows + 4095) / 4096);
  if (splits > 64) splits = 64;
  // d_bqkv = colsum(dQKV)
  colsum_partial_kernel<<<cb, 256, 0, st>>>(w.d_qkv, rows, ncols, w.partial);
  NRMS_LAUNCH_CHECK("colsum_dqkv");
  launch_partial_reduce_accum(w.partial, cb, ncols, ncols, d_bqkv, st);
  NRMS_LAUNCH_CHECK("dbqkv_reduce");
  if (tc) {
    // d_wqkv[900,300] += dQKV^T X
    if (!dqkv_t_written)
      if (int rc = transpose_f32(w.d_qkv, ncols, w.t1, w.ldr, rows, ncols, st)) return rc;
    if (int rc = transpose_f32(x, D, w.t2, w.ldr, rows, D, st)) return rc;
    if (int rc = tc_gemm_nt_ex(w.t1, w.ldr, w.t2, w.ldr, nullptr, d_wqkv, D, ncols, D, (int)rows,
                               tc_gemm_auto_splits(ncols, D, (int)rows), TC_EPI_ATOMIC, st)) return rc;
    if (!d_x) return NRMS_OK;
    // d_x = dQKV * Wqkv
    if (int rc = transpose_f32(wqkv, D, w.wt, ncols, ncols, D, st)) return rc;
    if (int rc = tc_gemm_nt_ex(w.d_qkv, ncols, w.wt, ncols, nullptr, d_x, D, rows, D, ncols, 1,
                               accum_dx ? TC_EPI_ACCUM : TC_EPI_STORE, st)) return rc;
  } else {
    // d_wqkv[900,300] += dQKV^T X
    cudaError_t e = sgemm_launch<1, 1, EPI_ATOMIC>(w.d_qkv, ncols, x, D, nullptr, d_wqkv, D, ncols, D, rows, splits, st);
    if (e != cudaSuccess) return cuda_fail(e, "sgemm dWqkv");
    if (!d_x) return NRMS_OK;
    // d_x = dQKV * Wqkv   ([rows,900] x [900,300])
    e = accum_dx ? sgemm_launch<0, 1, EPI_ACCUM>(w.d_qkv, ncols, wqkv, D, nullptr, d_x, D, rows, D, ncols, 1, st)
                 : sgemm_launch<0, 1, EPI_STORE>(w.d_qkv, ncols, wqkv, D, nullptr, d_x, D, rows, D, ncols, 1, st);
    if (e != cudaSuccess) return cuda_fail(e, "sgemm dX");
  }
  return NRMS_OK;
}

// Backward over the whole stash.  d_x (rows x 300) receives dL/dX.  text_train: as in encoder_core_fwd.
static int encoder_core_bwd(const Stash& s, const BwdWs& w, const float* d_out, int64_t n_seq, int S,
                            const float* wqkv, const float* wa, const float* qa, float* d_x, float* d_wqkv,
                            float* d_bqkv, float* d_wa, float* d_ba, float* d_qa, float p2, uint64_t seed,
                            uint64_t offset, int mode, cudaStream_t st, const LnArgs* ln = nullptr,
                            bool text_train = false) {
  // FP32 mode: every contraction on the CUDA cores (reference-exact up to summation order).  Tensor mode: the four
  // GEMMs run on tcgen05 (TF32 operands rounded by the TMA unit, fp32 accumulation) through the K-major NT kernel:
  //   dC  += dU   Wa        = NT(dU   [rows,200], Wa^T   [300,200])
  //   dX   = dQKV Wqkv      = NT(dQKV [rows,900], Wqkv^T [300,900])
  //   dWa   += dU^T   C     = NT(dU^T   [200,rows], C^T [300,rows])      split along K = rows, atomic epilogue
  //   dWqkv += dQKV^T X     = NT(dQKV^T [900,rows], X^T [300,rows])
  // so the row-major activations are transposed once per use (1.2 KB/row of extra traffic, a fraction of what the
  // fp32 SGEMMs cost: measured 6.3 ms -> see profiles/).
  const bool tc = (mode == NRMS_MODE_TF32);
  const int64_t rows = n_seq * S;
  const float* cin = ln ? s.cn : s.c;        // input of the additive block
  {
    const AddBwdWs aw{w.d_u, w.partial, w.t1, w.t2, w.wt, w.ldr};
    if (int rc = additive_block_bwd(d_out, cin, s.t, s.w, wa, qa, w.d_c, aw, n_seq, S, d_wa, d_ba, d_qa, tc, st)) return rc;
  }
  cudaError_t e;
  if (ln) {   // d_c holds dL/dCN: through the LayerNorm, in place; d_gamma / d_beta via per-block partial sums
    int lb = (int)((rows + 7) / 8 < REDUCE_BLOCKS ? (rows + 7) / 8 : REDUCE_BLOCKS);
    layernorm_bwd_kernel<<<lb, 256, 0, st>>>(w.d_c, s.c, s.stats, ln->gamma, w.partial, rows);
    NRMS_LAUNCH_CHECK("layernorm_bwd");
    launch_partial_reduce_accum(w.partial, lb, 2 * D, D, ln->d_gamma, st);
    NRMS_LAUNCH_CHECK("dgamma_reduce");
    launch_partial_reduce_accum(w.partial + D, lb, 2 * D, D, ln->d_beta, st);
    NRMS_LAUNCH_CHECK("dbeta_reduce");
  }
  // attention backward (applies the dropout-2 mask to d_c on load)
#ifndef NRMS_ATTN_BWD_HC20
#define NRMS_ATTN_BWD_HC20 5        // heads per CTA of the title-length attention backward (measured: 5 -> 807 us, 15 -> 1,086 us per 7,040 titles)
#endif
  bool dqkv_t_written = false;
  if (S == 20 && tc && g_train_attn_mma) {
    // the kernel also leaves dQKV^T in t1 (the K-major operand of the dWqkv contraction below)
    if (int rc2 = attn_mma_bwd(s.qkv, w.d_c, w.d_qkv, w.t1, w.ldr, n_seq, p2, seed, offset, st)) return rc2;
    dqkv_t_written = true;
    e = cudaSuccess;
  } else if (S == 50 && text_train && tc && g_train_attn_mma) {
    if (int rc2 = attn_mma50_bwd(s.qkv, w.d_c, w.d_qkv, w.t1, w.ldr, n_seq, p2, seed, offset, st)) return rc2;
    dqkv_t_written = true;
    e = cudaSuccess;
  } else if (S == 20) e = launch_attention_bwd<20, NRMS_ATTN_BWD_HC20>(s.qkv, w.d_c, w.d_qkv, n_seq, p2, seed, offset, st);
  else if (S == 50) e = launch_attention_bwd<50, 5>(s.qkv, w.d_c, w.d_qkv, n_seq, p2, seed, offset, st);
  else {
    // every other length: dq | dk | dv into dQKV with the pitch of the stash
    const MhaOperands op{s.qkv, s.qkv + D, s.qkv + 2 * D, D3, D3, D3};
    if (int rc2 = mha_attn_bwd(op, w.d_c, w.d_qkv, w.d_qkv + D, w.d_qkv + 2 * D, n_seq, S, S, nullptr, mode, st, p2, seed,
                               offset))
      return rc2;
    e = cudaSuccess;
  }
  if (e != cudaSuccess) return cuda_fail(e, "attention_bwd");
  const QkvBwdWs qw{w.d_qkv, w.partial, w.t1, w.t2, w.wt, w.ldr};
  return qkv_proj_bwd(qw, s.x, wqkv, rows, d_x, d_wqkv, d_bqkv, tc, dqkv_t_written, st);
}

// nrms_news_encoder_* and nrms_mhsa_*: the compiled title / abstract lengths
static int check_common(int S, int mode) {
  NRMS_CHECK_ARG(S == 20 || S == 50, NRMS_E_UNSUPPORTED, "sequence length %d unsupported (compiled: 20, 50)", S);
  NRMS_CHECK_ARG(mode == NRMS_MODE_FP32 || mode == NRMS_MODE_TF32, NRMS_E_INVALID, "bad mode %d", mode);
  return NRMS_OK;
}

// nrms_text_encoder_*: any title / abstract length up to 64 (20 and 50 keep their compiled kernels)
constexpr int TEXT_MAXS = 64;
static int check_text(int L, int mode) {
  NRMS_CHECK_ARG(L >= 1 && L <= TEXT_MAXS, NRMS_E_UNSUPPORTED, "text length %d unsupported (1..%d)", L, TEXT_MAXS);
  NRMS_CHECK_ARG(mode == NRMS_MODE_FP32 || mode == NRMS_MODE_TF32, NRMS_E_INVALID, "bad mode %d", mode);
  return NRMS_OK;
}

// user encoder: any history length up to 64 (20 and 50 keep their compiled kernels)
constexpr int USER_MAXS = 64;
static int check_user(int S, int mode) {
  NRMS_CHECK_ARG(S >= 1 && S <= USER_MAXS, NRMS_E_UNSUPPORTED, "history length %d unsupported (1..%d)", S, USER_MAXS);
  NRMS_CHECK_ARG(mode == NRMS_MODE_FP32 || mode == NRMS_MODE_TF32, NRMS_E_INVALID, "bad mode %d", mode);
  return NRMS_OK;
}

}  // namespace nrms

using namespace nrms;

extern "C" {

size_t nrms_encoder_stash_bytes(int64_t n_seq, int S) {
  if (n_seq <= 0 || S <= 0) return 0;
  return carve_stash(nullptr, n_seq * S).bytes;
}

size_t nrms_encoder_ln_stash_bytes(int64_t n_seq, int S) {
  if (n_seq <= 0 || S <= 0) return 0;
  return carve_stash(nullptr, n_seq * S, true).bytes;
}

size_t nrms_encoder_fwd_workspace_bytes(int64_t n_seq, int S, int mode, int training, int64_t n_src_rows) {
  if (n_seq <= 0 || S <= 0) return 0;
  if (training) return 256;
  if (mode == NRMS_MODE_TF32) {
    size_t fused = tc_fused_workspace_bytes(n_seq, S, n_src_rows);
    if (fused != (size_t)-1) return fused + 256;
  }
  int64_t chunk_seq = INFER_CHUNK_ROWS / S;
  if (n_seq < chunk_seq) chunk_seq = n_seq;
  return carve_stash(nullptr, chunk_seq * S, true).bytes + 256;     // room for the LayerNorm variant's fields too
}

size_t nrms_encoder_bwd_workspace_bytes(int64_t n_seq, int S, int mode) {
  if (n_seq <= 0 || S <= 0) return 0;
  return carve_bwd(nullptr, n_seq * S, true, mode).bytes + 256;
}

static int check_ln(const LnArgs* ln, bool bwd) {
  if (!ln) return NRMS_OK;
  NRMS_CHECK_ARG(ln->gamma && aligned16(ln->gamma), NRMS_E_INVALID, "LayerNorm weight missing or misaligned");
  if (bwd) NRMS_CHECK_ARG(ln->d_gamma && ln->d_beta, NRMS_E_INVALID, "LayerNorm gradient pointers missing");
  else NRMS_CHECK_ARG(ln->beta && aligned16(ln->beta), NRMS_E_INVALID, "LayerNorm bias missing or misaligned");
  return NRMS_OK;
}

// The length rule is the caller's: check_common (nrms_news_encoder_*) or check_text (nrms_text_encoder_*)
typedef int (*LengthRule)(int L, int mode);

static int news_encoder_fwd_impl(const int64_t* tokens, int64_t n_titles, int L, const float* emb, int64_t num_words,
                                 const float* wqkv, const float* bqkv, const float* wa, const float* ba, const float* qa,
                                 float* out, void* stash, void* workspace, size_t workspace_bytes, float dropout_p,
                                 uint64_t seed, uint64_t offset, int mode, void* stream, const LnArgs* ln,
                                 LengthRule length_rule, const int64_t* news_rows = nullptr) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (int rc = check_ln(ln, false)) return rc;
  if (int rc = length_rule(L, mode)) return rc;
  NRMS_CHECK_ARG(news_rows == nullptr || stash != nullptr, NRMS_E_UNSUPPORTED,
                 "the index-only form (token table + news rows) is the training form: pass a stash");
  NRMS_CHECK_ARG(n_titles >= 0 && num_words > 0, NRMS_E_INVALID, "bad sizes");
  if (n_titles == 0) return NRMS_OK;
  NRMS_CHECK_ARG(tokens && emb && wqkv && bqkv && wa && ba && qa && out, NRMS_E_INVALID, "null pointer");
  NRMS_CHECK_ARG(aligned16(emb) && aligned16(wqkv) && aligned16(bqkv) && aligned16(wa) && aligned16(ba) && aligned16(out),
                 NRMS_E_INVALID, "pointers must be 16-byte aligned");
  NRMS_CHECK_ARG(dropout_p >= 0.f && dropout_p < 1.f, NRMS_E_INVALID, "dropout_p out of range");
  const float scale = dropout_p > 0.f ? 1.f / (1.f - dropout_p) : 1.f;

  if (stash) {  // training: everything kept for backward
    NRMS_CHECK_ARG(aligned16(stash), NRMS_E_INVALID, "stash misaligned");
    Stash s = carve_stash(stash, n_titles * L, ln != nullptr);
    const int64_t rows = n_titles * L;
    int64_t gb = (rows + 7) / 8;
    if (gb > (int64_t)num_sms() * 16) gb = (int64_t)num_sms() * 16;
    gather_embedding_kernel<<<(unsigned)gb, 256, 0, st>>>(tokens, rows, emb, s.x, dropout_p, scale, seed, offset,
                                                          news_rows, L);
    NRMS_LAUNCH_CHECK("gather_embedding");
    return encoder_core_fwd(s, n_titles, L, wqkv, bqkv, wa, ba, qa, out, dropout_p, seed, offset, 0, mode, st, ln, true);
  }
  // inference
  if (mode == NRMS_MODE_TF32 && dropout_p == 0.f && tc_fused_workspace_bytes(n_titles, L, num_words) != (size_t)-1) {
    return tc_encoder_fused(emb, nullptr, num_words, tokens, 1, n_titles, L, wqkv, bqkv, wa, ba, qa, out, workspace,
                            workspace_bytes, st, ln ? ln->gamma : nullptr, ln ? ln->beta : nullptr, /*hot_row = padding_idx*/ 0);
  }
  const int64_t chunk_seq = INFER_CHUNK_ROWS / L;
  const int64_t first = n_titles < chunk_seq ? n_titles : chunk_seq;
  NRMS_CHECK_ARG(workspace && aligned16(workspace) && workspace_bytes >= carve_stash(nullptr, first * L, true).bytes,
                 NRMS_E_WORKSPACE, "workspace too small: need %zu bytes", carve_stash(nullptr, first * L, true).bytes);
  for (int64_t s0 = 0; s0 < n_titles; s0 += chunk_seq) {
    const int64_t n = (n_titles - s0 < chunk_seq) ? (n_titles - s0) : chunk_seq;
    Stash s = carve_stash(workspace, n * L, ln != nullptr);
    const int64_t rows = n * L;
    int64_t gb = (rows + 7) / 8;
    if (gb > (int64_t)num_sms() * 16) gb = (int64_t)num_sms() * 16;
    // global row index keys the dropout stream, so a chunked pass equals a single pass
    gather_embedding_kernel<<<(unsigned)gb, 256, 0, st>>>(tokens + s0 * L, rows, emb, s.x, dropout_p, scale, seed,
                                                          offset + (uint64_t)s0 * L * D / 4);
    NRMS_LAUNCH_CHECK("gather_embedding");
    int rc = encoder_core_fwd(s, n, L, wqkv, bqkv, wa, ba, qa, out + s0 * D, dropout_p, seed, offset, s0 * L, mode, st,
                              ln);
    if (rc) return rc;
  }
  return NRMS_OK;
}

int nrms_news_encoder_fwd(const int64_t* tokens, int64_t n_titles, int L, const float* emb, int64_t num_words,
                          const float* wqkv, const float* bqkv, const float* wa, const float* ba, const float* qa,
                          float* out, void* stash, void* workspace, size_t workspace_bytes, float dropout_p,
                          uint64_t seed, uint64_t offset, int mode, void* stream) {
  return news_encoder_fwd_impl(tokens, n_titles, L, emb, num_words, wqkv, bqkv, wa, ba, qa, out, stash, workspace,
                               workspace_bytes, dropout_p, seed, offset, mode, stream, nullptr, check_common);
}

int nrms_news_encoder_i32_fwd(const int32_t* tokens, int64_t n_titles, int L, const float* emb, int64_t num_words,
                              const float* wqkv, const float* bqkv, const float* wa, const float* ba, const float* qa,
                              float* out, void* workspace, size_t workspace_bytes, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (int rc = check_common(L, NRMS_MODE_TF32)) return rc;
  NRMS_CHECK_ARG(n_titles >= 0 && num_words > 0, NRMS_E_INVALID, "bad sizes");
  if (n_titles == 0) return NRMS_OK;
  NRMS_CHECK_ARG(tokens && emb && wqkv && bqkv && wa && ba && qa && out, NRMS_E_INVALID, "null pointer");
  NRMS_CHECK_ARG(aligned16(emb) && aligned16(wqkv) && aligned16(bqkv) && aligned16(wa) && aligned16(ba) && aligned16(out),
                 NRMS_E_INVALID, "pointers must be 16-byte aligned");
  NRMS_CHECK_ARG(tc_fused_workspace_bytes(n_titles, L, num_words) != (size_t)-1, NRMS_E_UNSUPPORTED, "title length not compiled");
  return tc_encoder_fused(emb, nullptr, num_words, tokens, 2, n_titles, L, wqkv, bqkv, wa, ba, qa, out, workspace,
                          workspace_bytes, st, nullptr, nullptr, /*hot_row = padding_idx*/ 0);
}

int nrms_news_encoder_ln_fwd(const int64_t* tokens, int64_t n_titles, int L, const float* emb, int64_t num_words,
                             const float* wqkv, const float* bqkv, const float* ln_gamma, const float* ln_beta,
                             const float* wa, const float* ba, const float* qa, float* out, void* stash, void* workspace,
                             size_t workspace_bytes, float dropout_p, uint64_t seed, uint64_t offset, int mode,
                             void* stream) {
  const LnArgs ln{ln_gamma, ln_beta, nullptr, nullptr};
  return news_encoder_fwd_impl(tokens, n_titles, L, emb, num_words, wqkv, bqkv, wa, ba, qa, out, stash, workspace,
                               workspace_bytes, dropout_p, seed, offset, mode, stream, &ln, check_common);
}

static int news_encoder_bwd_impl(const float* d_out, const int64_t* tokens, int64_t n_titles, int L, int64_t num_words,
                                 const float* wqkv, const float* wa, const float* qa, const void* stash, float* d_emb,
                                 float* d_wqkv, float* d_bqkv, float* d_wa, float* d_ba, float* d_qa, void* workspace,
                                 size_t workspace_bytes, float dropout_p, uint64_t seed, uint64_t offset, int mode,
                                 void* stream, const LnArgs* ln, LengthRule length_rule,
                                 const int64_t* news_rows = nullptr) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (int rc = check_ln(ln, true)) return rc;
  if (int rc = length_rule(L, mode)) return rc;
  if (n_titles == 0) return NRMS_OK;
  NRMS_CHECK_ARG(n_titles > 0 && num_words > 0, NRMS_E_INVALID, "bad sizes");
  NRMS_CHECK_ARG(d_out && tokens && wqkv && wa && qa && stash && d_emb && d_wqkv && d_bqkv && d_wa && d_ba && d_qa,
                 NRMS_E_INVALID, "null pointer");
  NRMS_CHECK_ARG(aligned16(d_out) && aligned16(stash) && aligned16(d_emb) && aligned16(d_wqkv) && aligned16(d_wa),
                 NRMS_E_INVALID, "pointers must be 16-byte aligned");
  const int64_t rows = n_titles * L;
  NRMS_CHECK_ARG(workspace && aligned16(workspace) && workspace_bytes >= carve_bwd(nullptr, rows, true, mode).bytes,
                 NRMS_E_WORKSPACE, "workspace too small: need %zu bytes", carve_bwd(nullptr, rows, true, mode).bytes);
  Stash s = carve_stash(const_cast<void*>(stash), rows, ln != nullptr);
  BwdWs w = carve_bwd(workspace, rows, true, mode);
  int rc = encoder_core_bwd(s, w, d_out, n_titles, L, wqkv, wa, qa, w.d_x, d_wqkv, d_bqkv, d_wa, d_ba, d_qa,
                            dropout_p, seed, offset, mode, st, ln, true);
  if (rc) return rc;
  const float scale = dropout_p > 0.f ? 1.f / (1.f - dropout_p) : 1.f;
  int64_t gb = (rows + 7) / 8;
  if (gb > (int64_t)num_sms() * 16) gb = (int64_t)num_sms() * 16;
  scatter_embedding_grad_kernel<<<(unsigned)gb, 256, 0, st>>>(tokens, rows, w.d_x, d_emb, dropout_p, scale, seed, offset,
                                                              news_rows, L);
  NRMS_LAUNCH_CHECK("scatter_embedding_grad");
  return NRMS_OK;
}

int nrms_news_encoder_bwd(const float* d_out, const int64_t* tokens, int64_t n_titles, int L, int64_t num_words,
                          const float* wqkv, const float* wa, const float* qa, const void* stash, float* d_emb,
                          float* d_wqkv, float* d_bqkv, float* d_wa, float* d_ba, float* d_qa, void* workspace,
                          size_t workspace_bytes, float dropout_p, uint64_t seed, uint64_t offset, int mode,
                          void* stream) {
  return news_encoder_bwd_impl(d_out, tokens, n_titles, L, num_words, wqkv, wa, qa, stash, d_emb, d_wqkv, d_bqkv, d_wa,
                               d_ba, d_qa, workspace, workspace_bytes, dropout_p, seed, offset, mode, stream, nullptr,
                               check_common);
}

int nrms_news_encoder_ln_bwd(const float* d_out, const int64_t* tokens, int64_t n_titles, int L, int64_t num_words,
                             const float* wqkv, const float* ln_gamma, const float* wa, const float* qa,
                             const void* stash, float* d_emb, float* d_wqkv, float* d_bqkv, float* d_ln_gamma,
                             float* d_ln_beta, float* d_wa, float* d_ba, float* d_qa, void* workspace,
                             size_t workspace_bytes, float dropout_p, uint64_t seed, uint64_t offset, int mode,
                             void* stream) {
  const LnArgs ln{ln_gamma, nullptr, d_ln_gamma, d_ln_beta};
  return news_encoder_bwd_impl(d_out, tokens, n_titles, L, num_words, wqkv, wa, qa, stash, d_emb, d_wqkv, d_bqkv, d_wa,
                               d_ba, d_qa, workspace, workspace_bytes, dropout_p, seed, offset, mode, stream, &ln,
                               check_common);
}

int nrms_news_encoder_rows_fwd(const int64_t* token_table, int64_t n_news, const int64_t* news_rows, int64_t n_titles,
                               int L, const float* emb, int64_t num_words, const float* wqkv, const float* bqkv,
                               const float* ln_gamma, const float* ln_beta, const float* wa, const float* ba,
                               const float* qa, float* out, void* stash, float dropout_p, uint64_t seed, uint64_t offset,
                               int mode, void* stream) {
  NRMS_CHECK_ARG(n_news > 0 && (n_titles == 0 || news_rows), NRMS_E_INVALID, "bad token table / news rows");
  NRMS_CHECK_ARG((ln_gamma == nullptr) == (ln_beta == nullptr), NRMS_E_INVALID, "LayerNorm needs both weight and bias");
  const LnArgs ln{ln_gamma, ln_beta, nullptr, nullptr};
  return news_encoder_fwd_impl(token_table, n_titles, L, emb, num_words, wqkv, bqkv, wa, ba, qa, out, stash, nullptr, 0,
                               dropout_p, seed, offset, mode, stream, ln_gamma ? &ln : nullptr, check_common, news_rows);
}

int nrms_news_encoder_rows_bwd(const float* d_out, const int64_t* token_table, int64_t n_news, const int64_t* news_rows,
                               int64_t n_titles, int L, int64_t num_words, const float* wqkv, const float* ln_gamma,
                               const float* wa, const float* qa, const void* stash, float* d_emb, float* d_wqkv,
                               float* d_bqkv, float* d_ln_gamma, float* d_ln_beta, float* d_wa, float* d_ba, float* d_qa,
                               void* workspace, size_t workspace_bytes, float dropout_p, uint64_t seed, uint64_t offset,
                               int mode, void* stream) {
  NRMS_CHECK_ARG(n_news > 0 && (n_titles == 0 || news_rows), NRMS_E_INVALID, "bad token table / news rows");
  const LnArgs ln{ln_gamma, nullptr, d_ln_gamma, d_ln_beta};
  return news_encoder_bwd_impl(d_out, token_table, n_titles, L, num_words, wqkv, wa, qa, stash, d_emb, d_wqkv, d_bqkv,
                               d_wa, d_ba, d_qa, workspace, workspace_bytes, dropout_p, seed, offset, mode, stream,
                               ln_gamma ? &ln : nullptr, check_common, news_rows);
}

// Any text length 1..64, one pair for every form: dense tokens [n_texts, L] (news_rows NULL, n_token_rows >= n_texts)
// or the index-only form (text t is row news_rows[t] of the [n_token_rows, L] table, training only), with or without the
// LayerNorm, training (a stash) or inference.  The length is checked before anything else; then each form is checked as
// in nrms_news_encoder_{,ln_,rows_}fwd / bwd, and 20 / 50 run what those run.
int nrms_text_encoder_fwd(const int64_t* tokens, int64_t n_token_rows, const int64_t* news_rows, int64_t n_texts, int L,
                          const float* emb, int64_t num_words, const float* wqkv, const float* bqkv,
                          const float* ln_gamma, const float* ln_beta, const float* wa, const float* ba, const float* qa,
                          float* out, void* stash, void* workspace, size_t workspace_bytes, float dropout_p,
                          uint64_t seed, uint64_t offset, int mode, void* stream) {
  if (int rc = check_text(L, mode)) return rc;
  NRMS_CHECK_ARG(news_rows ? (n_token_rows > 0) : (n_token_rows >= n_texts), NRMS_E_INVALID,
                 "bad token rows: %lld for %lld texts", (long long)n_token_rows, (long long)n_texts);
  NRMS_CHECK_ARG((ln_gamma == nullptr) == (ln_beta == nullptr), NRMS_E_INVALID, "LayerNorm needs both weight and bias");
  const LnArgs ln{ln_gamma, ln_beta, nullptr, nullptr};
  return news_encoder_fwd_impl(tokens, n_texts, L, emb, num_words, wqkv, bqkv, wa, ba, qa, out, stash, workspace,
                               workspace_bytes, dropout_p, seed, offset, mode, stream, ln_gamma ? &ln : nullptr,
                               check_text, news_rows);
}

int nrms_text_encoder_bwd(const float* d_out, const int64_t* tokens, int64_t n_token_rows, const int64_t* news_rows,
                          int64_t n_texts, int L, int64_t num_words, const float* wqkv, const float* ln_gamma,
                          const float* wa, const float* qa, const void* stash, float* d_emb, float* d_wqkv,
                          float* d_bqkv, float* d_ln_gamma, float* d_ln_beta, float* d_wa, float* d_ba, float* d_qa,
                          void* workspace, size_t workspace_bytes, float dropout_p, uint64_t seed, uint64_t offset,
                          int mode, void* stream) {
  if (int rc = check_text(L, mode)) return rc;
  NRMS_CHECK_ARG(news_rows ? (n_token_rows > 0) : (n_token_rows >= n_texts), NRMS_E_INVALID,
                 "bad token rows: %lld for %lld texts", (long long)n_token_rows, (long long)n_texts);
  const LnArgs ln{ln_gamma, nullptr, d_ln_gamma, d_ln_beta};
  return news_encoder_bwd_impl(d_out, tokens, n_texts, L, num_words, wqkv, wa, qa, stash, d_emb, d_wqkv, d_bqkv, d_wa,
                               d_ba, d_qa, workspace, workspace_bytes, dropout_p, seed, offset, mode, stream,
                               ln_gamma ? &ln : nullptr, check_text, news_rows);
}

static int user_encoder_fwd_impl(const float* x, int64_t n_rows, const int32_t* rows_idx, int64_t n_users, int S,
                                 const float* wqkv, const float* bqkv, const float* wa, const float* ba, const float* qa,
                                 float* out, void* stash, void* workspace, size_t workspace_bytes, int mode,
                                 void* stream, const LnArgs* ln) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (int rc = check_user(S, mode)) return rc;     // the length first: outside 1..64 is NRMS_E_UNSUPPORTED
  if (int rc = check_ln(ln, false)) return rc;
  NRMS_CHECK_ARG(n_users >= 0, NRMS_E_INVALID, "bad sizes");
  if (n_users == 0) return NRMS_OK;
  NRMS_CHECK_ARG(x && wqkv && bqkv && wa && ba && qa && out, NRMS_E_INVALID, "null pointer");
  NRMS_CHECK_ARG(aligned16(x) && aligned16(wqkv) && aligned16(bqkv) && aligned16(wa) && aligned16(ba) && aligned16(out),
                 NRMS_E_INVALID, "pointers must be 16-byte aligned");
  if (stash) {
    NRMS_CHECK_ARG(rows_idx == nullptr, NRMS_E_UNSUPPORTED, "indexed input is inference-only");
    NRMS_CHECK_ARG(aligned16(stash), NRMS_E_INVALID, "stash misaligned");
    Stash s = carve_stash(stash, n_users * S, ln != nullptr);
    NRMS_CUDA(cudaMemcpyAsync(s.x, x, (size_t)n_users * S * D * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return encoder_core_fwd(s, n_users, S, wqkv, bqkv, wa, ba, qa, out, 0.f, 0, 0, 0, mode, st, ln);
  }
  NRMS_CHECK_ARG(rows_idx == nullptr || n_rows > 0, NRMS_E_INVALID, "indexed input needs n_rows (rows of the table)");
  if (mode == NRMS_MODE_TF32 && tc_fused_workspace_bytes(n_users, S, rows_idx ? n_rows : 0) != (size_t)-1) {
    return tc_encoder_fused(x, nullptr, rows_idx ? n_rows : 0, rows_idx, rows_idx ? 2 : 0, n_users, S, wqkv, bqkv, wa, ba, qa, out,
                            workspace, workspace_bytes, st, ln ? ln->gamma : nullptr, ln ? ln->beta : nullptr);
  }
  const int64_t chunk_seq = INFER_CHUNK_ROWS / S;
  const int64_t first = n_users < chunk_seq ? n_users : chunk_seq;
  NRMS_CHECK_ARG(workspace && aligned16(workspace) && workspace_bytes >= carve_stash(nullptr, first * S, true).bytes,
                 NRMS_E_WORKSPACE, "workspace too small: need %zu bytes", carve_stash(nullptr, first * S, true).bytes);
  for (int64_t s0 = 0; s0 < n_users; s0 += chunk_seq) {
    const int64_t n = (n_users - s0 < chunk_seq) ? (n_users - s0) : chunk_seq;
    Stash s = carve_stash(workspace, n * S, ln != nullptr);
    const int64_t rows = n * S;
    if (rows_idx) {
      int64_t gb = (rows + 7) / 8;
      if (gb > (int64_t)num_sms() * 16) gb = (int64_t)num_sms() * 16;
      gather_rows_kernel<int32_t><<<(unsigned)gb, 256, 0, st>>>(x, rows_idx + s0 * S, rows, DV4, s.x);
      NRMS_LAUNCH_CHECK("gather_rows");
    } else {
      s.x = const_cast<float*>(x) + s0 * S * D;  // dense input is read in place
    }
    int rc = encoder_core_fwd(s, n, S, wqkv, bqkv, wa, ba, qa, out + s0 * D, 0.f, 0, 0, 0, mode, st, ln);
    if (rc) return rc;
  }
  return NRMS_OK;
}

int nrms_user_encoder_fwd(const float* x, int64_t n_rows, const int32_t* rows_idx, int64_t n_users, int S, const float* wqkv,
                          const float* bqkv, const float* wa, const float* ba, const float* qa, float* out,
                          void* stash, void* workspace, size_t workspace_bytes, int mode, void* stream) {
  return user_encoder_fwd_impl(x, n_rows, rows_idx, n_users, S, wqkv, bqkv, wa, ba, qa, out, stash, workspace,
                               workspace_bytes, mode, stream, nullptr);
}

int nrms_user_encoder_ln_fwd(const float* x, int64_t n_rows, const int32_t* rows_idx, int64_t n_users, int S,
                             const float* wqkv, const float* bqkv, const float* ln_gamma, const float* ln_beta,
                             const float* wa, const float* ba, const float* qa, float* out, void* stash, void* workspace,
                             size_t workspace_bytes, int mode, void* stream) {
  const LnArgs ln{ln_gamma, ln_beta, nullptr, nullptr};
  return user_encoder_fwd_impl(x, n_rows, rows_idx, n_users, S, wqkv, bqkv, wa, ba, qa, out, stash, workspace,
                               workspace_bytes, mode, stream, &ln);
}

// S = 20 / 50: the fused kernels over the fp16 table; other lengths: chunks of fp32 stash rows widened from it
static int64_t table16_chunk_seq(int64_t n_users, int S) {
  const int64_t chunk_seq = INFER_CHUNK_ROWS / S;
  return n_users < chunk_seq ? n_users : chunk_seq;
}

size_t nrms_user_encoder_table16_workspace_bytes(int64_t n_users, int S, int64_t n_rows) {
  if (n_users <= 0 || S <= 0 || S > USER_MAXS || n_rows <= 0) return 0;
  size_t fused = tc_fused_workspace_bytes(n_users, S, n_rows, true);
  if (fused != (size_t)-1) return fused + 256;
  return carve_stash(nullptr, table16_chunk_seq(n_users, S) * S).bytes + 256;
}

int nrms_user_encoder_table16_fwd(const void* table16, int64_t n_rows, const int32_t* rows_idx, int64_t n_users, int S,
                                  const float* wqkv, const float* bqkv, const float* wa, const float* ba, const float* qa,
                                  float* out, void* workspace, size_t workspace_bytes, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (int rc = check_user(S, NRMS_MODE_TF32)) return rc;
  NRMS_CHECK_ARG(n_users >= 0 && n_rows > 0, NRMS_E_INVALID, "bad sizes");
  if (n_users == 0) return NRMS_OK;
  NRMS_CHECK_ARG(table16 && rows_idx && wqkv && bqkv && wa && ba && qa && out, NRMS_E_INVALID, "null pointer");
  NRMS_CHECK_ARG(aligned16(table16) && aligned16(wqkv) && aligned16(bqkv) && aligned16(wa) && aligned16(ba) && aligned16(out),
                 NRMS_E_INVALID, "pointers must be 16-byte aligned");
  if (tc_fused_workspace_bytes(n_users, S, n_rows, true) != (size_t)-1)
    return tc_encoder_fused(nullptr, table16, n_rows, rows_idx, 2, n_users, S, wqkv, bqkv, wa, ba, qa, out, workspace,
                            workspace_bytes, st);
  // other lengths: the tensor-mode core over fp32 rows widened from the fp16 table, chunk by chunk
  const int64_t chunk_seq = INFER_CHUNK_ROWS / S;
  const size_t need = carve_stash(nullptr, table16_chunk_seq(n_users, S) * S).bytes;
  NRMS_CHECK_ARG(workspace && aligned16(workspace) && workspace_bytes >= need, NRMS_E_WORKSPACE,
                 "workspace too small: need %zu bytes", need);
  for (int64_t s0 = 0; s0 < n_users; s0 += chunk_seq) {
    const int64_t n = (n_users - s0 < chunk_seq) ? (n_users - s0) : chunk_seq;
    Stash s = carve_stash(workspace, n * S);
    const int64_t rows = n * S;
    int64_t gb = (rows + 7) / 8;
    if (gb > (int64_t)num_sms() * 16) gb = (int64_t)num_sms() * 16;
    gather_rows_f16_kernel<<<(unsigned)gb, 256, 0, st>>>(reinterpret_cast<const __half*>(table16), rows_idx + s0 * S, rows,
                                                         s.x);
    NRMS_LAUNCH_CHECK("gather_rows_f16");
    if (int rc = encoder_core_fwd(s, n, S, wqkv, bqkv, wa, ba, qa, out + s0 * D, 0.f, 0, 0, 0, NRMS_MODE_TF32, st))
      return rc;
  }
  return NRMS_OK;
}

static int user_encoder_bwd_impl(const float* d_out, int64_t n_users, int S, const float* wqkv, const float* wa,
                                 const float* qa, const void* stash, float* d_x, float* d_wqkv, float* d_bqkv,
                                 float* d_wa, float* d_ba, float* d_qa, void* workspace, size_t workspace_bytes,
                                 int mode, void* stream, const LnArgs* ln) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (int rc = check_user(S, mode)) return rc;     // the length first: outside 1..64 is NRMS_E_UNSUPPORTED
  if (int rc = check_ln(ln, true)) return rc;
  if (n_users == 0) return NRMS_OK;
  NRMS_CHECK_ARG(n_users > 0, NRMS_E_INVALID, "bad sizes");
  NRMS_CHECK_ARG(d_out && wqkv && wa && qa && stash && d_x && d_wqkv && d_bqkv && d_wa && d_ba && d_qa, NRMS_E_INVALID,
                 "null pointer");
  NRMS_CHECK_ARG(aligned16(d_out) && aligned16(stash) && aligned16(d_x) && aligned16(d_wqkv) && aligned16(d_wa),
                 NRMS_E_INVALID, "pointers must be 16-byte aligned");
  const int64_t rows = n_users * S;
  NRMS_CHECK_ARG(workspace && aligned16(workspace) && workspace_bytes >= carve_bwd(nullptr, rows, false, mode).bytes,
                 NRMS_E_WORKSPACE, "workspace too small: need %zu bytes", carve_bwd(nullptr, rows, false, mode).bytes);
  Stash s = carve_stash(const_cast<void*>(stash), rows, ln != nullptr);
  BwdWs w = carve_bwd(workspace, rows, false, mode);
  return encoder_core_bwd(s, w, d_out, n_users, S, wqkv, wa, qa, d_x, d_wqkv, d_bqkv, d_wa, d_ba, d_qa, 0.f, 0, 0, mode,
                          st, ln);
}

int nrms_user_encoder_bwd(const float* d_out, int64_t n_users, int S, const float* wqkv, const float* wa,
                          const float* qa, const void* stash, float* d_x, float* d_wqkv, float* d_bqkv, float* d_wa,
                          float* d_ba, float* d_qa, void* workspace, size_t workspace_bytes, int mode, void* stream) {
  return user_encoder_bwd_impl(d_out, n_users, S, wqkv, wa, qa, stash, d_x, d_wqkv, d_bqkv, d_wa, d_ba, d_qa, workspace,
                               workspace_bytes, mode, stream, nullptr);
}

int nrms_user_encoder_ln_bwd(const float* d_out, int64_t n_users, int S, const float* wqkv, const float* ln_gamma,
                             const float* wa, const float* qa, const void* stash, float* d_x, float* d_wqkv,
                             float* d_bqkv, float* d_ln_gamma, float* d_ln_beta, float* d_wa, float* d_ba, float* d_qa,
                             void* workspace, size_t workspace_bytes, int mode, void* stream) {
  const LnArgs ln{ln_gamma, nullptr, d_ln_gamma, d_ln_beta};
  return user_encoder_bwd_impl(d_out, n_users, S, wqkv, wa, qa, stash, d_x, d_wqkv, d_bqkv, d_wa, d_ba, d_qa, workspace,
                               workspace_bytes, mode, stream, &ln);
}

// ---- standalone L0 blocks: MultiHeadSelfAttention.forward / AdditiveAttention.forward and their backwards ----
static int mhsa_fwd_impl(const float* x, const int32_t* lengths, int64_t n_seq, int S, const float* wqkv,
                         const float* bqkv, float* ctx, void* workspace, size_t workspace_bytes, int mode, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (int rc = check_common(S, mode)) return rc;
  NRMS_CHECK_ARG(n_seq >= 0, NRMS_E_INVALID, "bad sizes");
  if (n_seq == 0) return NRMS_OK;
  NRMS_CHECK_ARG(x && wqkv && bqkv && ctx, NRMS_E_INVALID, "null pointer");
  NRMS_CHECK_ARG(aligned16(x) && aligned16(wqkv) && aligned16(bqkv) && aligned16(ctx), NRMS_E_INVALID,
                 "pointers must be 16-byte aligned");
  const int64_t rows = n_seq * S;
  const size_t need = (size_t)rows * D3 * sizeof(float);
  NRMS_CHECK_ARG(workspace && aligned16(workspace) && workspace_bytes >= need, NRMS_E_WORKSPACE,
                 "workspace too small: need %zu bytes", need);
  float* qkv = reinterpret_cast<float*>(workspace);
  if (int rc = gemm_nt_bias(x, D, wqkv, D, bqkv, qkv, D3, rows, D3, D, mode, st)) return rc;
  cudaError_t e = (S == 20) ? launch_attention_fwd<20, 15>(qkv, ctx, n_seq, 0.f, 0, 0, st, lengths)
                            : launch_attention_fwd<50, 5>(qkv, ctx, n_seq, 0.f, 0, 0, st, lengths);
  if (e != cudaSuccess) return cuda_fail(e, "attention_fwd");
  return NRMS_OK;
}

int nrms_mhsa_fwd(const float* x, int64_t n_seq, int S, const float* wqkv, const float* bqkv, float* ctx,
                  void* workspace, size_t workspace_bytes, int mode, void* stream) {
  return mhsa_fwd_impl(x, nullptr, n_seq, S, wqkv, bqkv, ctx, workspace, workspace_bytes, mode, stream);
}

int nrms_mhsa_masked_fwd(const float* x, const int32_t* lengths, int64_t n_seq, int S, const float* wqkv,
                         const float* bqkv, float* ctx, void* workspace, size_t workspace_bytes, int mode, void* stream) {
  NRMS_CHECK_ARG(lengths != nullptr || n_seq == 0, NRMS_E_INVALID, "null lengths");
  return mhsa_fwd_impl(x, lengths, n_seq, S, wqkv, bqkv, ctx, workspace, workspace_bytes, mode, stream);
}

// workspace of nrms_mhsa_bwd: dQKV [rows,900] | partial sums [296,900]; tensor mode adds t1 [900,ldr] (dQKV^T) |
// t2 [300,ldr] (X^T) | wt [300,900] (Wqkv^T), ldr = rows rounded up to 4
static QkvBwdWs carve_mhsa_bwd(void* base, int64_t rows, int mode, size_t* bytes) {
  QkvBwdWs w{};
  char* p = reinterpret_cast<char*>(base);
  size_t off = 0;
  auto take = [&](size_t nfloat) {
    float* r = reinterpret_cast<float*>(p + off);
    off += align_up(nfloat * sizeof(float), 256);
    return r;
  };
  w.d_qkv = take((size_t)rows * D3);
  w.partial = take((size_t)REDUCE_BLOCKS * D3);
  w.ldr = (rows + 3) / 4 * 4;
  if (mode == NRMS_MODE_TF32) {
    w.t1 = take((size_t)w.ldr * D3);
    w.t2 = take((size_t)w.ldr * D);
    w.wt = take((size_t)D3 * D);
  }
  *bytes = off;
  return w;
}

size_t nrms_mhsa_bwd_workspace_bytes(int64_t n_seq, int S, int mode) {
  if (n_seq <= 0 || S <= 0) return 0;
  size_t bytes = 0;
  carve_mhsa_bwd(nullptr, n_seq * S, mode, &bytes);
  return bytes;
}

int nrms_mhsa_bwd(const float* d_ctx, const float* x, const int32_t* lengths, int64_t n_seq, int S, const float* wqkv,
                  const void* fwd_workspace, float* d_x, float* d_wqkv, float* d_bqkv, void* workspace,
                  size_t workspace_bytes, int mode, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (int rc = check_common(S, mode)) return rc;
  NRMS_CHECK_ARG(n_seq >= 0, NRMS_E_INVALID, "bad sizes");
  if (n_seq == 0) return NRMS_OK;
  NRMS_CHECK_ARG(d_ctx && x && wqkv && fwd_workspace && d_wqkv && d_bqkv, NRMS_E_INVALID, "null pointer");
  NRMS_CHECK_ARG(aligned16(d_ctx) && aligned16(x) && aligned16(wqkv) && aligned16(fwd_workspace) && aligned16(d_wqkv) &&
                     (!d_x || aligned16(d_x)) && (reinterpret_cast<uintptr_t>(lengths) & 3) == 0,
                 NRMS_E_INVALID, "pointers must be 16-byte aligned (lengths: 4-byte)");
  const int64_t rows = n_seq * S;
  size_t need = 0;
  QkvBwdWs w = carve_mhsa_bwd(workspace, rows, mode, &need);
  NRMS_CHECK_ARG(workspace && aligned16(workspace) && workspace_bytes >= need, NRMS_E_WORKSPACE,
                 "workspace too small: need %zu bytes", need);
  const bool tc = (mode == NRMS_MODE_TF32);
  const float* qkv = reinterpret_cast<const float*>(fwd_workspace);     // what nrms_mhsa_(masked_)fwd left there
  bool dqkv_t_written = false;
  if (tc && g_train_attn_mma) {
    // mma.sync tiles, as the encoders' training attention; the kernel also leaves dQKV^T in t1
    const int rc = S == 20 ? attn_mma_bwd(qkv, d_ctx, w.d_qkv, w.t1, w.ldr, n_seq, 0.f, 0, 0, st, lengths)
                           : attn_mma50_bwd(qkv, d_ctx, w.d_qkv, w.t1, w.ldr, n_seq, 0.f, 0, 0, st, lengths);
    if (rc) return rc;
    dqkv_t_written = true;
  } else {
    cudaError_t e;
    if (S == 20)
      e = lengths ? launch_attention_bwd<20, NRMS_ATTN_BWD_HC20, true>(qkv, d_ctx, w.d_qkv, n_seq, 0.f, 0, 0, st, lengths)
                  : launch_attention_bwd<20, NRMS_ATTN_BWD_HC20>(qkv, d_ctx, w.d_qkv, n_seq, 0.f, 0, 0, st);
    else
      e = lengths ? launch_attention_bwd<50, 5, true>(qkv, d_ctx, w.d_qkv, n_seq, 0.f, 0, 0, st, lengths)
                  : launch_attention_bwd<50, 5>(qkv, d_ctx, w.d_qkv, n_seq, 0.f, 0, 0, st);
    if (e != cudaSuccess) return cuda_fail(e, "attention_bwd");
  }
  return qkv_proj_bwd(w, x, wqkv, rows, d_x, d_wqkv, d_bqkv, tc, dqkv_t_written, st);
}

// ---- MultiHeadSelfAttention.forward(Q, K, V, length) at 1 <= Sq, Sk <= 64 (nrms_mha_*) ----
// Each input is projected onto the contiguous rows of Wqkv it needs, into its own buffer; an input passed in two roles
// whose weight rows are adjacent is projected once:
//   Q's input -> A [n*Sq, 300 c]: c = 3 when it is also K's and V's (self-attention, one 900-column GEMM), 2 when it is
//                also K's (q|k), else 1
//   K's input, when not Q's -> Bk [n*Sk, 600] (k|v) when it is also V's, else [n*Sk, 300]
//   V's input, when not K's -> Bv [n*Sk, 300] (when it is Q's but K's is another input, W_Q and W_V are not adjacent in
//                Wqkv: Q's input gets a second 300-column projection here, and its gradient is the sum of both)
// The forward workspace holds A | Bk | Bv at their largest (900, 300 and 300 columns; a [n*Sk, 600] Bk runs on into Bv's
// slot), and the backward's dA | dBk | dBv have the same layout, so the attention backward writes dq / dk / dv with the
// pitches of q / k / v and every projection backward reads one contiguous [rows, 300 c] matrix.
struct MhaPlan {
  int n_proj;                // projections (one per input, two for Q's input when it is V's but not K's)
  const float* x[3];
  int64_t rows[3];
  int c0[3], nc[3];          // rows [300 c0, 300 (c0 + nc)) of Wqkv
  float* buf[3];             // projection (or its gradient), [rows, 300 nc]
  MhaOperands op;
  size_t bytes;
};
static MhaPlan mha_plan(const float* xq, const float* xk, const float* xv, int64_t n_seq, int sq, int sk, void* base) {
  MhaPlan p{};
  char* b = reinterpret_cast<char*>(base);
  const size_t a_bytes = align_up((size_t)n_seq * sq * D3 * sizeof(float), 256);
  const size_t k_bytes = align_up((size_t)n_seq * sk * D * sizeof(float), 256);
  float* A = reinterpret_cast<float*>(b);
  float* Bk = reinterpret_cast<float*>(b + a_bytes);
  float* Bv = reinterpret_cast<float*>(b + a_bytes + k_bytes);
  p.bytes = a_bytes + 2 * k_bytes;
  const bool qk = xq == xk, qv = xq == xv, kv = xk == xv;
  auto add = [&](const float* x, int64_t rows, int c0, int nc, float* buf) {
    const int i = p.n_proj++;
    p.x[i] = x; p.rows[i] = rows; p.c0[i] = c0; p.nc[i] = nc; p.buf[i] = buf;
  };
  const int na = (qk && qv) ? 3 : (qk ? 2 : 1);
  add(xq, n_seq * sq, 0, na, A);
  p.op.q = A; p.op.ldq = (int64_t)D * na;
  if (qk) {
    p.op.k = A + D; p.op.ldk = p.op.ldq;
  } else {
    add(xk, n_seq * sk, 1, kv ? 2 : 1, Bk);
    p.op.k = Bk; p.op.ldk = kv ? 2 * D : D;
  }
  if (qk && qv) {
    p.op.v = A + 2 * D; p.op.ldv = p.op.ldq;
  } else if (kv) {
    p.op.v = Bk + D; p.op.ldv = 2 * D;
  } else {
    add(xv, n_seq * sk, 2, 1, Bv);
    p.op.v = Bv; p.op.ldv = D;
  }
  return p;
}

// the checks both directions share, in order: mode, shapes, sizes (n_seq == 0 -> done), null / misaligned pointers,
// inputs passed twice with different row counts
static int mha_check(const float* xq, const float* xk, const float* xv, int64_t n_seq, int sq, int sk,
                     const int32_t* lengths, const float* wqkv, int mode, bool* done) {
  *done = false;
  NRMS_CHECK_ARG(mode == NRMS_MODE_FP32 || mode == NRMS_MODE_TF32, NRMS_E_INVALID, "bad mode %d", mode);
  NRMS_CHECK_ARG(sq >= 1 && sq <= 64 && sk >= 1 && sk <= 64, NRMS_E_UNSUPPORTED,
                 "query / key counts %d / %d unsupported (compiled: 1..64)", sq, sk);
  NRMS_CHECK_ARG(lengths == nullptr || sq == sk || sq == 1, NRMS_E_UNSUPPORTED,
                 "a length mask needs as many queries as keys, or one query (%d queries, %d keys)", sq, sk);
  NRMS_CHECK_ARG(n_seq >= 0, NRMS_E_INVALID, "bad sizes");
  if (n_seq == 0) {
    *done = true;
    return NRMS_OK;
  }
  NRMS_CHECK_ARG(xq && xk && xv && wqkv, NRMS_E_INVALID, "null pointer");
  NRMS_CHECK_ARG(aligned16(xq) && aligned16(xk) && aligned16(xv) && aligned16(wqkv) &&
                     (reinterpret_cast<uintptr_t>(lengths) & 3) == 0,
                 NRMS_E_INVALID, "pointers must be 16-byte aligned (lengths: 4-byte)");
  NRMS_CHECK_ARG((xq != xk && xq != xv) || sq == sk, NRMS_E_INVALID,
                 "the query input is also the key or value input: Sq (%d) must equal Sk (%d)", sq, sk);
  return NRMS_OK;
}

size_t nrms_mha_fwd_workspace_bytes(int64_t n_seq, int Sq, int Sk) {
  if (n_seq <= 0 || Sq <= 0 || Sk <= 0) return 0;
  return mha_plan(nullptr, nullptr, nullptr, n_seq, Sq, Sk, nullptr).bytes;
}

int nrms_mha_fwd(const float* xq, const float* xk, const float* xv, int64_t n_seq, int Sq, int Sk, const int32_t* lengths,
                 const float* wqkv, const float* bqkv, float* ctx, void* workspace, size_t workspace_bytes, int mode,
                 void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  bool done;
  if (int rc = mha_check(xq, xk, xv, n_seq, Sq, Sk, lengths, wqkv, mode, &done)) return rc;
  if (done) return NRMS_OK;
  NRMS_CHECK_ARG(bqkv && ctx, NRMS_E_INVALID, "null pointer");
  NRMS_CHECK_ARG(aligned16(bqkv) && aligned16(ctx), NRMS_E_INVALID, "pointers must be 16-byte aligned");
  NRMS_CHECK_ARG(ctx != xq && ctx != xk && ctx != xv, NRMS_E_INVALID, "ctx must not alias an input");
  NRMS_CHECK_ARG(aligned16(workspace), NRMS_E_INVALID, "workspace must be 16-byte aligned");
  const MhaPlan p = mha_plan(xq, xk, xv, n_seq, Sq, Sk, workspace);
  NRMS_CHECK_ARG(workspace && workspace_bytes >= p.bytes, NRMS_E_WORKSPACE,
                 "workspace too small: need %zu bytes", p.bytes);
  for (int i = 0; i < p.n_proj; ++i) {
    const int64_t w0 = (int64_t)p.c0[i] * D;
    if (int rc = gemm_nt_bias(p.x[i], D, wqkv + w0 * D, D, bqkv + w0, p.buf[i], (int64_t)D * p.nc[i], p.rows[i], D * p.nc[i],
                              D, mode, st)) return rc;
  }
  return mha_attn_fwd(p.op, ctx, n_seq, Sq, Sk, lengths, mode, st);
}

// workspace of nrms_mha_bwd: dA | dBk | dBv (mha_plan) | partial sums [296,900]; tensor mode adds t1 [900,ldr] |
// t2 [300,ldr] | wt [300,900], ldr = n_seq * max(Sq, Sk) rounded up to 4 (shared by the inputs, one after the other)
static size_t carve_mha_bwd(void* base, int64_t n_seq, int sq, int sk, int mode, QkvBwdWs* w) {
  const MhaPlan dp = mha_plan(nullptr, nullptr, nullptr, n_seq, sq, sk, nullptr);
  char* p = reinterpret_cast<char*>(base);
  size_t off = dp.bytes;
  auto take = [&](size_t nfloat) {
    float* r = reinterpret_cast<float*>(p + off);
    off += align_up(nfloat * sizeof(float), 256);
    return r;
  };
  QkvBwdWs ws{};
  ws.partial = take((size_t)REDUCE_BLOCKS * D3);
  ws.ldr = (n_seq * (sq > sk ? sq : sk) + 3) / 4 * 4;
  if (mode == NRMS_MODE_TF32) {
    ws.t1 = take((size_t)ws.ldr * D3);
    ws.t2 = take((size_t)ws.ldr * D);
    ws.wt = take((size_t)D3 * D);
  }
  if (w) *w = ws;
  return off;
}

size_t nrms_mha_bwd_workspace_bytes(int64_t n_seq, int Sq, int Sk, int mode) {
  if (n_seq <= 0 || Sq <= 0 || Sk <= 0) return 0;
  return carve_mha_bwd(nullptr, n_seq, Sq, Sk, mode, nullptr);
}

int nrms_mha_bwd(const float* d_ctx, const float* xq, const float* xk, const float* xv, int64_t n_seq, int Sq, int Sk,
                 const int32_t* lengths, const float* wqkv, const void* fwd_workspace, float* d_xq, float* d_xk,
                 float* d_xv, float* d_wqkv, float* d_bqkv, void* workspace, size_t workspace_bytes, int mode,
                 void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  bool done;
  if (int rc = mha_check(xq, xk, xv, n_seq, Sq, Sk, lengths, wqkv, mode, &done)) return rc;
  if (done) return NRMS_OK;
  NRMS_CHECK_ARG(d_ctx && fwd_workspace && d_wqkv && d_bqkv, NRMS_E_INVALID, "null pointer");
  NRMS_CHECK_ARG(aligned16(d_ctx) && aligned16(fwd_workspace) && aligned16(d_wqkv) && aligned16(d_bqkv) &&
                     (!d_xq || aligned16(d_xq)) && (!d_xk || aligned16(d_xk)) && (!d_xv || aligned16(d_xv)) &&
                     aligned16(workspace),
                 NRMS_E_INVALID, "pointers must be 16-byte aligned");
  // aliasing: an input passed twice has one gradient buffer (or NULL for the alias), which receives the sum; gradients
  // of distinct inputs are distinct buffers, and no gradient buffer is an input
  const float* xs[3] = {xq, xk, xv};
  float* ds[3] = {d_xq, d_xk, d_xv};
  for (int a = 0; a < 3; ++a) {
    for (int b = a + 1; b < 3; ++b) {
      if (xs[a] == xs[b])
        NRMS_CHECK_ARG(!ds[a] || !ds[b] || ds[a] == ds[b], NRMS_E_INVALID,
                       "an input passed twice takes one gradient buffer (the other NULL or the same)");
      else
        NRMS_CHECK_ARG(!ds[a] || !ds[b] || ds[a] != ds[b], NRMS_E_INVALID, "distinct inputs need distinct gradient buffers");
    }
    NRMS_CHECK_ARG(!ds[a] || (ds[a] != xq && ds[a] != xk && ds[a] != xv && ds[a] != d_ctx), NRMS_E_INVALID,
                   "a gradient buffer must not alias an input");
  }
  QkvBwdWs w;
  const size_t need = carve_mha_bwd(workspace, n_seq, Sq, Sk, mode, &w);
  NRMS_CHECK_ARG(workspace && workspace_bytes >= need, NRMS_E_WORKSPACE, "workspace too small: need %zu bytes", need);
  const MhaPlan p = mha_plan(xq, xk, xv, n_seq, Sq, Sk, const_cast<void*>(fwd_workspace));   // the forward's projections
  const MhaPlan dp = mha_plan(xq, xk, xv, n_seq, Sq, Sk, workspace);                          // their gradients
  if (int rc = mha_attn_bwd(p.op, d_ctx, const_cast<float*>(dp.op.q), const_cast<float*>(dp.op.k), const_cast<float*>(dp.op.v),
                            n_seq, Sq, Sk, lengths, mode, st)) return rc;
  const bool tc = (mode == NRMS_MODE_TF32);
  for (int i = 0; i < p.n_proj; ++i) {
    float* dx = nullptr;          // the one gradient buffer of this input, if any of its roles has one
    for (int r = 2; r >= 0; --r)
      if (xs[r] == p.x[i] && ds[r]) dx = ds[r];
    bool accum = false;           // a second projection of the same input adds to the first one's dX
    for (int j = 0; j < i; ++j) accum = accum || p.x[j] == p.x[i];
    const int64_t w0 = (int64_t)p.c0[i] * D;
    QkvBwdWs wi = w;
    wi.d_qkv = dp.buf[i];
    if (int rc = qkv_proj_bwd(wi, p.x[i], wqkv + w0 * D, p.rows[i], dx, d_wqkv + w0 * D, d_bqkv + w0, tc, false, st,
                              D * p.nc[i], accum)) return rc;
  }
  return NRMS_OK;
}

int nrms_additive_fwd(const float* c, int64_t n_seq, int S, const float* wa, const float* ba, const float* qa,
                      float* out, void* workspace, size_t workspace_bytes, int mode, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  NRMS_CHECK_ARG(additive_len_ok(S), NRMS_E_UNSUPPORTED, "candidate size %d unsupported (1..64)", S);
  NRMS_CHECK_ARG(mode == NRMS_MODE_FP32 || mode == NRMS_MODE_TF32, NRMS_E_INVALID, "bad mode %d", mode);
  NRMS_CHECK_ARG(n_seq >= 0, NRMS_E_INVALID, "bad sizes");
  if (n_seq == 0) return NRMS_OK;
  NRMS_CHECK_ARG(c && wa && ba && qa && out, NRMS_E_INVALID, "null pointer");
  NRMS_CHECK_ARG(aligned16(c) && aligned16(wa) && aligned16(ba) && aligned16(out), NRMS_E_INVALID,
                 "pointers must be 16-byte aligned");
  const int64_t rows = n_seq * S;
  const size_t t_bytes = align_up((size_t)rows * QD * sizeof(float), 256);
  const size_t need = t_bytes + (size_t)rows * sizeof(float);
  NRMS_CHECK_ARG(workspace && aligned16(workspace) && workspace_bytes >= need, NRMS_E_WORKSPACE,
                 "workspace too small: need %zu bytes", need);
  float* t = reinterpret_cast<float*>(workspace);
  float* w = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + t_bytes);
  // the 2..4-row form (Exp1's final attention) is 3 % of a text encoder's work: always on the CUDA cores
  if (int rc = gemm_nt_bias(c, D, wa, D, ba, t, QD, rows, QD, D, S < 20 ? NRMS_MODE_FP32 : mode, st)) return rc;
  if (cudaError_t e = launch_additive_fwd(c, t, qa, w, out, n_seq, S, st)) return cuda_fail(e, "additive_fwd");
  return NRMS_OK;
}

size_t nrms_additive_bwd_workspace_bytes(int64_t n_seq, int S, int mode) {
  const int64_t rows = n_seq * S;
  const int64_t ldr = (rows + 3) / 4 * 4;
  size_t b = align_up((size_t)rows * QD * sizeof(float), 256) + align_up((size_t)REDUCE_BLOCKS * D3 * sizeof(float), 256);
  if (mode == NRMS_MODE_TF32 && S >= 20)
    b += align_up((size_t)ldr * QD * sizeof(float), 256) + align_up((size_t)ldr * D * sizeof(float), 256) +
         align_up((size_t)D * QD * sizeof(float), 256);
  return b;
}

int nrms_additive_bwd(const float* d_out, const float* c, int64_t n_seq, int S, const float* wa, const float* qa,
                      const void* fwd_workspace, float* d_c, float* d_wa, float* d_ba, float* d_qa, void* workspace,
                      size_t workspace_bytes, int mode, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  NRMS_CHECK_ARG(additive_len_ok(S), NRMS_E_UNSUPPORTED, "candidate size %d unsupported (1..64)", S);
  NRMS_CHECK_ARG(mode == NRMS_MODE_FP32 || mode == NRMS_MODE_TF32, NRMS_E_INVALID, "bad mode %d", mode);
  NRMS_CHECK_ARG(n_seq >= 0, NRMS_E_INVALID, "bad sizes");
  if (n_seq == 0) return NRMS_OK;
  NRMS_CHECK_ARG(d_out && c && wa && qa && fwd_workspace && d_c && d_wa && d_ba && d_qa, NRMS_E_INVALID, "null pointer");
  NRMS_CHECK_ARG(aligned16(d_out) && aligned16(c) && aligned16(wa) && aligned16(d_c) && aligned16(d_wa) &&
                     aligned16(fwd_workspace), NRMS_E_INVALID, "pointers must be 16-byte aligned");
  const size_t need = nrms_additive_bwd_workspace_bytes(n_seq, S, mode);
  NRMS_CHECK_ARG(workspace && aligned16(workspace) && workspace_bytes >= need, NRMS_E_WORKSPACE,
                 "workspace too small: need %zu bytes", need);
  const int64_t rows = n_seq * S;
  const bool tc = (mode == NRMS_MODE_TF32 && S >= 20);
  const float* t = reinterpret_cast<const float*>(fwd_workspace);
  const float* wv = reinterpret_cast<const float*>(reinterpret_cast<const char*>(fwd_workspace) +
                                                   align_up((size_t)rows * QD * sizeof(float), 256));
  AddBwdWs aw{};
  char* p = reinterpret_cast<char*>(workspace);
  size_t off = 0;
  auto take = [&](size_t nfloat) {
    float* r = reinterpret_cast<float*>(p + off);
    off += align_up(nfloat * sizeof(float), 256);
    return r;
  };
  aw.d_u = take((size_t)rows * QD);
  aw.partial = take((size_t)REDUCE_BLOCKS * D3);
  aw.ldr = (rows + 3) / 4 * 4;
  if (tc) {
    aw.t1 = take((size_t)aw.ldr * QD);
    aw.t2 = take((size_t)aw.ldr * D);
    aw.wt = take((size_t)D * QD);
  }
  return additive_block_bwd(d_out, c, t, wv, wa, qa, d_c, aw, n_seq, S, d_wa, d_ba, d_qa, tc, st);
}

int nrms_set_option(const char* key, int value) {
  NRMS_CHECK_ARG(key != nullptr, NRMS_E_INVALID, "null option key");
  if (strcmp(key, "table_ratio") == 0) {
    NRMS_CHECK_ARG(set_table_ratio(value) == NRMS_OK, NRMS_E_INVALID, "table_ratio must be 1..1024");
    return NRMS_OK;
  }
  if (strcmp(key, "news_table_attn") == 0) {
    set_news_table_attn(value != 0);
    return NRMS_OK;
  }
  if (strcmp(key, "user_table_attn") == 0) {
    set_table_attn(value != 0);
    return NRMS_OK;
  }
  if (strcmp(key, "fused_pool") == 0) {
    set_fused_pool(value != 0);
    return NRMS_OK;
  }
  if (strcmp(key, "gemm_tma_epilogue") == 0) {
    set_gemm_tma_epilogue(value != 0);
    return NRMS_OK;
  }
  if (strcmp(key, "k1f_debug") == 0) {
    set_k1f_debug(value);
    return NRMS_OK;
  }
  if (strcmp(key, "attn_safe_softmax") == 0) {
    set_attn_safe_softmax(value);
    return NRMS_OK;
  }
  if (strcmp(key, "train_attn_mma") == 0) {
    g_train_attn_mma = value != 0;
    return NRMS_OK;
  }
  if (strcmp(key, "time_k1") == 0) {
    set_time_k1(value != 0);
    return NRMS_OK;
  }
  set_error("unknown option '%s'", key);
  return NRMS_E_INVALID;
}

double nrms_get_stat(const char* key) {
  if (!key) return -1.0;
  // "<kind>_ms" / "<kind>_launches" / "<kind>_sequences"; kind: k1 = user-encoder K1 (per-user projection),
  // k1n = news-encoder K1, k1g = user-encoder table attention
  static const char* kinds[4] = {"k1_", "k1n_", "k1g_", "k1gn_"};
  static const char* whats[3] = {"ms", "launches", "sequences"};
  for (int k = 3; k >= 0; --k) {          // longest prefix first (k1gn_ before k1g_, k1n_ before k1_)
    const size_t n = strlen(kinds[k]);
    if (strncmp(key, kinds[k], n) == 0)
      for (int w = 0; w < 3; ++w)
        if (strcmp(key + n, whats[w]) == 0) return get_k1_stat(3 * k + w);
  }
  return -1.0;
}

int nrms_gemm_nt(const float* A, int64_t lda, const float* B, int64_t ldb, const float* bias, float* C, int64_t ldc,
                 int64_t M, int N, int K, int mode, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  NRMS_CHECK_ARG(A && B && C, NRMS_E_INVALID, "null pointer");
  NRMS_CHECK_ARG(M >= 0 && N > 0 && K > 0 && (N % 4) == 0 && (K % 4) == 0 && (lda % 4) == 0 && (ldb % 4) == 0 && (ldc % 4) == 0,
                 NRMS_E_UNSUPPORTED, "N, K and leading dimensions must be multiples of 4");
  NRMS_CHECK_ARG(aligned16(A) && aligned16(B) && aligned16(C) && (!bias || aligned16(bias)), NRMS_E_INVALID,
                 "pointers must be 16-byte aligned");
  return gemm_nt_bias(A, lda, B, ldb, bias, C, ldc, M, N, K, mode, st);
}

}  // extern "C"
