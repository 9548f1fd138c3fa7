// Host-side entry points of the tensor-core (tcgen05) kernels, called from encoder.cu.
#pragma once
#include "common.cuh"

namespace nrms {

// C[M,N] = A[M,K] * B[N,K]^T (+ bias[N]); operands rounded to TF32 (rna) on the way into shared
// memory, fp32 accumulation in TMEM.  Same layout contract as sgemm (multiples of 4, 16B aligned).
int tc_gemm_nt(const float* A, int64_t lda, const float* B, int64_t ldb, const float* bias, float* C, int64_t ldc,
               int64_t M, int N, int K, cudaStream_t st);
// Same contraction with an epilogue mode (store / C += / atomic C +=) and an optional split along K (atomic only).
enum { TC_EPI_STORE = 0, TC_EPI_ACCUM = 1, TC_EPI_ATOMIC = 2, TC_EPI_STORE_F16 = 3, TC_EPI_STORE_F16_QKV = 4, TC_EPI_STORE_F16_TMA = 5 };
int tc_gemm_nt_ex(const float* A, int64_t lda, const float* B, int64_t ldb, const float* bias, float* C, int64_t ldc,
                  int64_t M, int N, int K, int k_splits, int epi, cudaStream_t st);
int tc_gemm_auto_splits(int64_t M, int N, int K);
// Same contraction, result rounded to fp16: C16[m*ldc + n] = half((acc + bias[n]) * (n < scale_cols ? scale : 1)), ldc in halfs.
// qkv_layout = 1 (N = 900): columns are scattered into K1g's padded head-group row layout (k1g_table_attn.cu).
int tc_gemm_nt_f16out(const float* A, int64_t lda, const float* B, int64_t ldb, const float* bias, void* C16, int64_t ldc,
                      int64_t M, int N, int K, float scale, int scale_cols, int qkv_layout, cudaStream_t st);
// dst[c][r] = src[r][c]: the K-major (NT) tensor-core GEMM sees A^T B and A B contractions through transposed copies
int transpose_f32(const float* src, int64_t ld_src, float* dst, int64_t ld_dst, int64_t R, int C, cudaStream_t st);

// Tensor-mode encoder forward (inference), fused_host.cu: table path (K1g / K1f) or per-sequence projection (K1 v6),
// then additive pooling (K2).  Input rows come from `src` [*,300] fp32 -- or from `src16`, the caller's fp16 copy of the
// gather source in pack_rows16's layout ([n_src_rows + 1][320] halfs, 1.0 in column 300, zero last row), when src is null:
//   idx_kind 0: dense rows (sequence s, position i -> row s*S+i), 1: int64 ids, 2: int32 ids.
// tc_fused_workspace_bytes returns (size_t)-1 when the fused path does not apply (S not 20/50).
// n_src_rows = rows of the gather source (idx_kind 1/2), 0 for dense input.
size_t tc_fused_workspace_bytes(int64_t n_seq, int S, int64_t n_src_rows, bool rows16_given = false);
// ln_gamma / ln_beta (nullable): LayerNorm(300) on the context rows between K1 and K2 (config-5 variant).
int tc_encoder_fused(const float* src, const void* src16, int64_t n_src_rows, const void* idx, int idx_kind, int64_t n_seq,
                     int S, const float* wqkv, const float* bqkv, const float* wa, const float* ba, const float* qa,
                     float* out, void* workspace, size_t workspace_bytes, cudaStream_t st, const float* ln_gamma = nullptr,
                     const float* ln_beta = nullptr, int64_t hot_row = -1);
// hot_row: a source row that a large share of the indices name (the padding token 0 of the titles); the table path keeps
// replicas of its projected row and spreads the references over them (an L2 hot spot otherwise).  -1 = none.
int pack_rows16(const float* src, int64_t n_rows, void* src16, cudaStream_t st);    // pack.cu

// fp16 operands (A16 [M, lda halfs], B16 [N, ldb halfs], 16-byte aligned rows), kind::f16, same fp16 epilogue (no bias)
int tc_gemm_nt_f16(const void* A16, int64_t lda, const void* B16, int64_t ldb, void* C16, int64_t ldc, int64_t M, int N,
                   int K, float scale, int scale_cols, int qkv_layout, cudaStream_t st);
// attn_mma.cu: tensor-mode TRAINING attention over 20-token titles on mma.sync TF32 tiles (forward, and the backward that
// recomputes the probabilities from the stashed q|k|v rows); qkv [n_seq*20, 900], ctx / d_ctx [n_seq*20, 300]
int attn_mma_fwd(const float* qkv, float* ctx, int64_t n_seq, float p, uint64_t seed, uint64_t offset, cudaStream_t st);
// d_qkv_t (nullable): the same gradients also written transposed, [900, ldt] (the dWqkv contraction's K-major operand)
// lengths (nullable, int32 [n_seq]): the key mask of the standalone block -- keys at positions >= lengths[seq] are left out
int attn_mma_bwd(const float* qkv, const float* d_ctx, float* d_qkv, float* d_qkv_t, int64_t ldt, int64_t n_seq, float p,
                 uint64_t seed, uint64_t offset, cudaStream_t st, const int32_t* lengths = nullptr);
// the same two passes over 50-token texts (abstracts): qkv [n_seq*50, 900], ctx / d_ctx [n_seq*50, 300]
int attn_mma50_fwd(const float* qkv, float* ctx, int64_t n_seq, float p, uint64_t seed, uint64_t offset, cudaStream_t st);
int attn_mma50_bwd(const float* qkv, const float* d_ctx, float* d_qkv, float* d_qkv_t, int64_t ldt, int64_t n_seq, float p,
                   uint64_t seed, uint64_t offset, cudaStream_t st, const int32_t* lengths = nullptr);
// attn_cross.cu: attention of the standalone block at 1 <= sq, sk <= 64 (self- or cross-attention), both modes.  q rows
// [n_seq*sq] and k / v rows [n_seq*sk] of 300 used columns each, at their own pitches; ctx / d_ctx [n_seq*sq, 300].
// lengths (nullable, int32 [n_seq]): the reference's `length` (sq == sk: keys j < length; sq == 1 < sk: all keys iff
// length >= 1).  The backward writes dq / dk / dv with the pitches of q / k / v.  p > 0: the news encoder's dropout #2
// on the context (self-attention, sq == sk, the row index of the call keys the mask; p == 0 launches the kernels without
// dropout).
struct MhaOperands {
  const float *q, *k, *v;
  int64_t ldq, ldk, ldv;
};
int mha_attn_fwd(const MhaOperands& in, float* ctx, int64_t n_seq, int sq, int sk, const int32_t* lengths, int mode,
                 cudaStream_t st, float p = 0.f, uint64_t seed = 0, uint64_t offset = 0);
int mha_attn_bwd(const MhaOperands& in, const float* d_ctx, float* dq, float* dk, float* dv, int64_t n_seq, int sq, int sk,
                 const int32_t* lengths, int mode, cudaStream_t st, float p = 0.f, uint64_t seed = 0, uint64_t offset = 0);
// K1f (k1f_attn_pool.cu): table attention + additive pooling in one kernel (the context rows stay on the SM)
int k1f_qk_bound(const void* table16, int64_t n_rows, float* bound, cudaStream_t st);
int k1f_run(int S, int idx_kind, const void* table16, int64_t n_table_rows, const void* rows, int64_t n_seq,
            const void* wa16, const float* ba, const float* qa, const float* bound, float* out, cudaStream_t st);
void set_attn_safe_softmax(int v);
int get_attn_safe_softmax();   // -1 auto (bound over the projected table), 0 plain 2^s, 1 row-shifted form
void set_gemm_tma_epilogue(bool on); // fp32 GEMM results through bulk tensor stores / reductions (default 1)
void set_k1f_debug(int v);           // component-removal timing switches of K1f (garbage results)
void set_fused_pool(bool on);        // table path: 1 (default) = K1f, 0 = K1g + K2 (context rows through HBM)
int tc_gemm_nt_f16_tma(const void* A16, int64_t lda, const void* B16, int64_t ldb, void* C16, int64_t ldc, int64_t M, int N,
                       int K, cudaStream_t st);   // fp16 in / fp16 out, dense row-major result through bulk tensor stores
void set_news_table_attn(bool on);   // news encoder over the projected embedding table (default on)
void set_table_attn(bool on);   // indexed user encoder: project the table once + K1g (default on)
int set_table_ratio(int v);  // gathered rows per source row from which the table path is taken (default 4)
void set_time_k1(bool on);   // CUDA-event timing of the K1 launches (bench.py roofline)
double get_k1_stat(int key); // 3 * kind (0 users K1 v6, 1 news K1 v6, 2 users table attention, 3 news table attention) + (0 total ms, 1 launches, 2 sequences)

}  // namespace nrms
