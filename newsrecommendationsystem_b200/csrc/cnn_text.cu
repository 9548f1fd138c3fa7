// NAML's CNN text encoder (reference src/model/NAML/news_encoder.py:9-40): embedding gather + dropout, Conv2d(1, 300,
// (3, 300), padding=(1, 0)), ReLU, dropout, additive pooling -- forward and backward, both arithmetic modes.
//
// Mapping.  With x the [L, 300] embedded rows of one text and W the conv weight viewed as [300, 900] (w*300 + d order),
//   conv[i, f] = b[f] + sum_w sum_d W[f, w*300 + d] * x[i + w - 1, d],   x[-1] = x[L] = 0.
// The three taps are one projection P = X Wcat^T, Wcat [900, 300] with Wcat[w*300 + f, d] = W[f, w*300 + d]: the
// [rows, 300] x [300, 900] contraction of the q|k|v projection (tcgen05 in tensor mode, the CUDA-core SGEMM in FP32
// mode).  The conv is then the shift-add conv[i] = b + P_0[i - 1] + P_1[i] + P_2[i + 1], with the neighbours outside
// the text left out; that is the zero padding, so no halo rows are stored and no row straddles two texts.
// Backward: dconv = d_a * mask2 * (h > 0); dP_w[j] = dconv[j + 1 - w] (inside the text, else 0); then
//   d_W[:, w*300 : w*300 + 300] += dP_w^T X,   d_b += colsum(dconv),   dX = dP Wcat,
// and dX * mask1 is scattered into d_emb through the token ids (row 0, the padding_idx, untouched).
#include <string.h>
#include "common.cuh"
#include "sgemm.cuh"
#include "tc_api.cuh"

namespace nrms {
namespace cnn {

constexpr uint32_t DROPOUT_STREAM_EMB = 1, DROPOUT_STREAM_CTX = 2;   // encoder_kernels.cuh
constexpr int MAXL = 64;
constexpr int64_t INFER_CHUNK_ROWS = 2048 * 20;                        // encoder.cu

__device__ __forceinline__ int64_t token_of(const int64_t* __restrict__ tokens, const int64_t* __restrict__ news_rows,
                                            int L, int64_t r) {
  return news_rows ? tokens[news_rows[r / L] * L + r % L] : tokens[r];
}

// X[r] = emb[token(r)] * mask1(r): one warp per row.  `row0` = the call's index of row 0 (chunks of an inference call).
__global__ void __launch_bounds__(256)
cnn_gather_kernel(const int64_t* __restrict__ tokens, const int64_t* __restrict__ news_rows, int L, int64_t row0,
                  int64_t n_rows, const float* __restrict__ emb, float* __restrict__ x, float p, float scale,
                  uint64_t seed, uint64_t offset) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t r = warp; r < n_rows; r += nwarps) {
    const int64_t g = row0 + r;
    const float4* src = reinterpret_cast<const float4*>(emb + token_of(tokens, news_rows, L, g) * D);
    float4* dst = reinterpret_cast<float4*>(x + r * D);
    for (int l = lane; l < DV4; l += 32) {
      float4 v = __ldg(src + l);
      if (p > 0.f) {
        const float4 m = dropout_mask4((uint64_t)g * D + 4 * l, DROPOUT_STREAM_EMB, p, scale, seed, offset);
        v.x *= m.x; v.y *= m.y; v.z *= m.z; v.w *= m.w;
      }
      dst[l] = v;
    }
  }
}

// conv epilogue: h = relu(b + P_0[i-1] + P_1[i] + P_2[i+1]) (h stored when non-null), a = h * mask2.  Thread = one
// float4 of one row.
__global__ void __launch_bounds__(256)
cnn_conv_epilogue_kernel(const float* __restrict__ P, const float* __restrict__ bias, int L, int64_t row0,
                         int64_t n_rows, float* __restrict__ h_out, float* __restrict__ a_out, float p, float scale,
                         uint64_t seed, uint64_t offset) {
  const int64_t total = n_rows * DV4;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = e / DV4;
    const int q = (int)(e - r * DV4);
    const int i = (int)((row0 + r) % L);
    const float4* pr = reinterpret_cast<const float4*>(P + r * D3);
    float4 c = __ldg(reinterpret_cast<const float4*>(bias) + q);
    const float4 p1 = __ldg(pr + DV4 + q);
    c.x += p1.x; c.y += p1.y; c.z += p1.z; c.w += p1.w;
    if (i > 0) {
      const float4 p0 = __ldg(pr - 3 * DV4 + q);          // P_0 of row r - 1
      c.x += p0.x; c.y += p0.y; c.z += p0.z; c.w += p0.w;
    }
    if (i < L - 1) {
      const float4 p2 = __ldg(pr + 3 * DV4 + 2 * DV4 + q);  // P_2 of row r + 1
      c.x += p2.x; c.y += p2.y; c.z += p2.z; c.w += p2.w;
    }
    c = make_float4(fmaxf(c.x, 0.f), fmaxf(c.y, 0.f), fmaxf(c.z, 0.f), fmaxf(c.w, 0.f));
    if (h_out) reinterpret_cast<float4*>(h_out + r * D)[q] = c;
    if (p > 0.f) {
      const float4 m = dropout_mask4((uint64_t)(row0 + r) * D + 4 * q, DROPOUT_STREAM_CTX, p, scale, seed, offset);
      c.x *= m.x; c.y *= m.y; c.z *= m.z; c.w *= m.w;
    }
    reinterpret_cast<float4*>(a_out + r * D)[q] = c;
  }
}

// dconv = d_a * mask2 * (h > 0), in place, and d_b += colsum(dconv).  Block = 4 row groups x 75 column quads over a
// contiguous range of rows; one float4 atomic per thread at the end.
constexpr int DCONV_THREADS = 4 * DV4;
__global__ void __launch_bounds__(DCONV_THREADS)
cnn_dconv_kernel(float* __restrict__ d, const float* __restrict__ h, int64_t n_rows, int64_t rows_per_block,
                 float* __restrict__ d_bias, float p, float scale, uint64_t seed, uint64_t offset) {
  const int q = threadIdx.x % DV4, rg = threadIdx.x / DV4;
  const int64_t r0 = (int64_t)blockIdx.x * rows_per_block;
  const int64_t r1 = r0 + rows_per_block < n_rows ? r0 + rows_per_block : n_rows;
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int64_t r = r0 + rg; r < r1; r += 4) {
    float4 g = reinterpret_cast<float4*>(d + r * D)[q];
    const float4 hv = __ldg(reinterpret_cast<const float4*>(h + r * D) + q);
    if (p > 0.f) {
      const float4 m = dropout_mask4((uint64_t)r * D + 4 * q, DROPOUT_STREAM_CTX, p, scale, seed, offset);
      g.x *= m.x; g.y *= m.y; g.z *= m.z; g.w *= m.w;
    }
    g.x = hv.x > 0.f ? g.x : 0.f;
    g.y = hv.y > 0.f ? g.y : 0.f;
    g.z = hv.z > 0.f ? g.z : 0.f;
    g.w = hv.w > 0.f ? g.w : 0.f;
    reinterpret_cast<float4*>(d + r * D)[q] = g;
    s.x += g.x; s.y += g.y; s.z += g.z; s.w += g.w;
  }
  if (r1 > r0) atomicAdd(reinterpret_cast<float4*>(d_bias) + q, s);
}

// dP[r, w*300 + f] = dconv[r + 1 - w, f] when that row is in the same text, else 0
__global__ void __launch_bounds__(256)
cnn_shift_kernel(const float* __restrict__ dconv, int L, int64_t n_rows, float* __restrict__ dP) {
  const int64_t total = n_rows * 3 * DV4;
  const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = e / (3 * DV4);
    const int c = (int)(e - r * 3 * DV4);
    const int w = c / DV4, q = c - w * DV4;
    const int i = (int)(r % L) + 1 - w;                   // position of the source row in its text
    reinterpret_cast<float4*>(dP + r * D3)[c] =
        (i >= 0 && i < L) ? __ldg(reinterpret_cast<const float4*>(dconv + (r + 1 - w) * D) + q) : z;
  }
}

// Wcat[w*300 + f, d] = W[f, w*300 + d] (transposed = 0, [900, 300]) or its transpose WcatT[d, w*300 + f]
// (transposed = 1, [300, 900]: the K-major operand of dX = dP Wcat on the tensor cores)
__global__ void __launch_bounds__(256)
cnn_permute_taps_kernel(const float* __restrict__ W, float* __restrict__ out, int transposed) {
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < D * D3; e += gridDim.x * blockDim.x) {
    const int f = e / D3, c = e - f * D3;                // W[f, c], c = w*300 + d
    const int w = c / D, d = c - w * D;
    if (transposed) out[(int64_t)d * D3 + w * D + f] = W[e];
    else out[(int64_t)(w * D + f) * D + d] = W[e];
  }
}

// d_emb[token(r)] += dX[r] * mask1(r); token 0 (padding_idx) skipped
__global__ void __launch_bounds__(256)
cnn_scatter_kernel(const int64_t* __restrict__ tokens, const int64_t* __restrict__ news_rows, int L, int64_t n_rows,
                   const float* __restrict__ dx, float* __restrict__ d_emb, float p, float scale, uint64_t seed,
                   uint64_t offset) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t r = warp; r < n_rows; r += nwarps) {
    const int64_t tok = token_of(tokens, news_rows, L, r);
    if (tok == 0) continue;
    const float4* src = reinterpret_cast<const float4*>(dx + r * D);
    float4* dst = reinterpret_cast<float4*>(d_emb + tok * D);
    for (int l = lane; l < DV4; l += 32) {
      float4 v = src[l];
      if (p > 0.f) {
        const float4 m = dropout_mask4((uint64_t)r * D + 4 * l, DROPOUT_STREAM_EMB, p, scale, seed, offset);
        v.x *= m.x; v.y *= m.y; v.z *= m.z; v.w *= m.w;
      }
      atomicAdd(dst + l, v);
    }
  }
}

// ---- buffer layouts ---------------------------------------------------------------------------------------------
struct Carver {
  char* p;
  size_t off = 0;
  explicit Carver(void* base) : p(reinterpret_cast<char*>(base)) {}
  float* take(size_t nfloat) {
    float* r = reinterpret_cast<float*>(p + off);
    off += align_up(nfloat * sizeof(float), 256);
    return r;
  }
};
// Stash of a training forward (also the per-chunk layout of inference): X [rows,300] (dropped embedding rows) |
// H [rows,300] (relu(conv), before dropout #2) | A [rows,300] (H * mask2, the additive block's input) | T [rows,200] |
// w [rows] (T | w: the workspace layout of nrms_additive_fwd).
struct CnnStash {
  float *x, *h, *a, *t, *w;
  size_t bytes;
};
static CnnStash carve_stash(void* base, int64_t rows) {
  Carver c(base);
  CnnStash s;
  s.x = c.take((size_t)rows * D);
  s.h = c.take((size_t)rows * D);
  s.a = c.take((size_t)rows * D);
  s.t = c.take((size_t)rows * QD);
  s.w = c.take((size_t)rows);
  s.bytes = c.off;
  return s;
}
// forward workspace: Wcat [900,300] | P [rows,900] | (inference) the chunk's stash
struct FwdWs {
  float *wcat, *P;
  CnnStash chunk;
  size_t bytes;
};
static FwdWs carve_fwd(void* base, int64_t rows, bool training) {
  Carver c(base);
  FwdWs f;
  f.wcat = c.take((size_t)D3 * D);
  f.P = c.take((size_t)rows * D3);
  f.chunk = carve_stash(training ? nullptr : c.p + c.off, rows);
  if (!training) c.off += f.chunk.bytes;
  f.bytes = c.off;
  return f;
}
// backward workspace: Wcat or WcatT [900*300] | dA = dconv, then dX [rows,300] | dP [rows,900] |
// tensor mode: t1 = dP^T [900, ldr] | t2 = X^T [300, ldr] | the additive backward's own workspace
struct BwdWs {
  float *wcat, *d, *dP, *t1, *t2;
  void* add_ws;
  size_t add_bytes;
  int64_t ldr;
  size_t bytes;
};
static BwdWs carve_bwd(void* base, int64_t n_texts, int L, int mode) {
  const int64_t rows = n_texts * L;
  Carver c(base);
  BwdWs b;
  b.wcat = c.take((size_t)D3 * D);
  b.d = c.take((size_t)rows * D);
  b.dP = c.take((size_t)rows * D3);
  b.ldr = (rows + 3) / 4 * 4;
  b.t1 = b.t2 = nullptr;
  if (mode == NRMS_MODE_TF32) {
    b.t1 = c.take((size_t)b.ldr * D3);
    b.t2 = c.take((size_t)b.ldr * D);
  }
  b.add_ws = c.p + c.off;
  b.add_bytes = align_up(nrms_additive_bwd_workspace_bytes(n_texts, L, mode), 256);
  c.off += b.add_bytes;
  b.bytes = c.off;
  return b;
}

static int64_t chunk_texts(int64_t n_texts, int L) {
  const int64_t c = INFER_CHUNK_ROWS / L;
  return n_texts < c ? n_texts : c;
}

static int check_len(int L, int mode) {
  NRMS_CHECK_ARG(L >= 1 && L <= MAXL, NRMS_E_UNSUPPORTED, "text length %d unsupported (1..%d)", L, MAXL);
  NRMS_CHECK_ARG(mode == NRMS_MODE_FP32 || mode == NRMS_MODE_TF32, NRMS_E_INVALID, "bad mode %d", mode);
  return NRMS_OK;
}

static unsigned grid_for(int64_t work, int64_t per_block, int cap_per_sm) {
  int64_t g = (work + per_block - 1) / per_block;
  const int64_t cap = (int64_t)num_sms() * cap_per_sm;
  if (g > cap) g = cap;
  return (unsigned)(g > 0 ? g : 1);
}

// the forward of n texts whose rows are call rows [row0, row0 + n*L): X, P, H (nullable), A, T, w in `s`
static int fwd_texts(const int64_t* tokens, const int64_t* news_rows, int64_t row0, int64_t n, int L, const float* emb,
                     const float* wcat, const float* conv_b, const float* wa, const float* ba, const float* qa,
                     float* out, const CnnStash& s, float* P, float p, uint64_t seed, uint64_t offset, int mode,
                     cudaStream_t st) {
  const int64_t rows = n * L;
  const float scale = p > 0.f ? 1.f / (1.f - p) : 1.f;
  cnn_gather_kernel<<<grid_for(rows, 8, 16), 256, 0, st>>>(tokens, news_rows, L, row0, rows, emb, s.x, p, scale, seed,
                                                           offset);
  NRMS_LAUNCH_CHECK("cnn_gather");
  if (mode == NRMS_MODE_TF32) {
    if (int rc = tc_gemm_nt(s.x, D, wcat, D, nullptr, P, D3, rows, D3, D, st)) return rc;
  } else {
    cudaError_t e = sgemm_launch<0, 0, EPI_STORE>(s.x, D, wcat, D, nullptr, P, D3, rows, D3, D, 1, st);
    if (e != cudaSuccess) return cuda_fail(e, "sgemm conv");
  }
  cnn_conv_epilogue_kernel<<<grid_for(rows * DV4, 256, 8), 256, 0, st>>>(P, conv_b, L, row0, rows, s.h, s.a, p, scale,
                                                                       seed, offset);
  NRMS_LAUNCH_CHECK("cnn_conv_epilogue");
  const size_t add_bytes = (size_t)(reinterpret_cast<char*>(s.w) - reinterpret_cast<char*>(s.t)) + rows * sizeof(float);
  return nrms_additive_fwd(s.a, n, L, wa, ba, qa, out, s.t, add_bytes, mode, st);
}

}  // namespace cnn
}  // namespace nrms

using namespace nrms;
using namespace nrms::cnn;

extern "C" {

size_t nrms_cnn_text_stash_bytes(int64_t n_texts, int L) {
  if (n_texts <= 0 || L <= 0) return 0;
  return cnn::carve_stash(nullptr, n_texts * L).bytes;
}

size_t nrms_cnn_text_fwd_workspace_bytes(int64_t n_texts, int L, int mode, int training) {
  (void)mode;
  if (n_texts <= 0 || L <= 0) return 0;
  if (training) return carve_fwd(nullptr, n_texts * L, true).bytes;
  return carve_fwd(nullptr, chunk_texts(n_texts, L) * L, false).bytes;
}

size_t nrms_cnn_text_bwd_workspace_bytes(int64_t n_texts, int L, int mode) {
  if (n_texts <= 0 || L <= 0) return 0;
  return cnn::carve_bwd(nullptr, n_texts, L, mode).bytes;
}

int nrms_cnn_text_fwd(const int64_t* tokens, int64_t n_token_rows, const int64_t* news_rows, int64_t n_texts, int L,
                      const float* emb, int64_t num_words, const float* conv_w, const float* conv_b, const float* wa,
                      const float* ba, const float* qa, float* out, void* stash, void* workspace,
                      size_t workspace_bytes, float dropout_p, uint64_t seed, uint64_t offset, int mode, void* stream) {
  if (int rc = check_len(L, mode)) return rc;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  NRMS_CHECK_ARG(n_texts >= 0 && num_words > 0, NRMS_E_INVALID, "bad sizes");
  NRMS_CHECK_ARG(news_rows ? (n_token_rows > 0) : (n_token_rows >= n_texts), NRMS_E_INVALID,
                 "bad token rows: %lld for %lld texts", (long long)n_token_rows, (long long)n_texts);
  if (n_texts == 0) return NRMS_OK;
  NRMS_CHECK_ARG(tokens && emb && conv_w && conv_b && wa && ba && qa && out, NRMS_E_INVALID, "null pointer");
  NRMS_CHECK_ARG(aligned16(emb) && aligned16(conv_w) && aligned16(conv_b) && aligned16(wa) && aligned16(ba) &&
                     aligned16(out) && aligned16(stash) && aligned16(workspace),
                 NRMS_E_INVALID, "pointers must be 16-byte aligned");
  NRMS_CHECK_ARG(dropout_p >= 0.f && dropout_p < 1.f, NRMS_E_INVALID, "dropout_p out of range");
  const bool training = stash != nullptr;
  const int64_t chunk = training ? n_texts : chunk_texts(n_texts, L);
  const FwdWs f = carve_fwd(workspace, chunk * L, training);
  NRMS_CHECK_ARG(workspace && workspace_bytes >= f.bytes, NRMS_E_WORKSPACE, "workspace too small: need %zu bytes",
                 f.bytes);
  cnn_permute_taps_kernel<<<grid_for(D * D3, 256, 4), 256, 0, st>>>(conv_w, f.wcat, 0);
  NRMS_LAUNCH_CHECK("cnn_permute_taps");
  if (training) {
    const CnnStash s = cnn::carve_stash(stash, n_texts * L);
    return fwd_texts(tokens, news_rows, 0, n_texts, L, emb, f.wcat, conv_b, wa, ba, qa, out, s, f.P, dropout_p, seed,
                     offset, mode, st);
  }
  for (int64_t s0 = 0; s0 < n_texts; s0 += chunk) {
    const int64_t n = n_texts - s0 < chunk ? n_texts - s0 : chunk;
    CnnStash s = f.chunk;
    s.h = nullptr;                    // inference keeps no pre-dropout activation
    if (int rc = fwd_texts(tokens, news_rows, s0 * L, n, L, emb, f.wcat, conv_b, wa, ba, qa, out + s0 * D, s, f.P,
                           dropout_p, seed, offset, mode, st))
      return rc;
  }
  return NRMS_OK;
}

int nrms_cnn_text_bwd(const float* d_out, const int64_t* tokens, int64_t n_token_rows, const int64_t* news_rows,
                      int64_t n_texts, int L, int64_t num_words, const float* conv_w, const float* wa, const float* qa,
                      const void* stash, float* d_emb, float* d_conv_w, float* d_conv_b, float* d_wa, float* d_ba,
                      float* d_qa, void* workspace, size_t workspace_bytes, float dropout_p, uint64_t seed,
                      uint64_t offset, int mode, void* stream) {
  if (int rc = check_len(L, mode)) return rc;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  NRMS_CHECK_ARG(n_texts >= 0 && num_words > 0, NRMS_E_INVALID, "bad sizes");
  NRMS_CHECK_ARG(news_rows ? (n_token_rows > 0) : (n_token_rows >= n_texts), NRMS_E_INVALID,
                 "bad token rows: %lld for %lld texts", (long long)n_token_rows, (long long)n_texts);
  if (n_texts == 0) return NRMS_OK;
  NRMS_CHECK_ARG(d_out && tokens && conv_w && wa && qa && stash && d_emb && d_conv_w && d_conv_b && d_wa && d_ba && d_qa,
                 NRMS_E_INVALID, "null pointer");
  NRMS_CHECK_ARG(aligned16(d_out) && aligned16(conv_w) && aligned16(wa) && aligned16(stash) && aligned16(d_emb) &&
                     aligned16(d_conv_w) && aligned16(d_conv_b) && aligned16(d_wa) && aligned16(workspace),
                 NRMS_E_INVALID, "pointers must be 16-byte aligned");
  NRMS_CHECK_ARG(dropout_p >= 0.f && dropout_p < 1.f, NRMS_E_INVALID, "dropout_p out of range");
  const int64_t rows = n_texts * L;
  const BwdWs b = cnn::carve_bwd(workspace, n_texts, L, mode);
  NRMS_CHECK_ARG(workspace && workspace_bytes >= b.bytes, NRMS_E_WORKSPACE, "workspace too small: need %zu bytes",
                 b.bytes);
  const CnnStash s = cnn::carve_stash(const_cast<void*>(stash), rows);
  const bool tc = mode == NRMS_MODE_TF32;
  const float scale = dropout_p > 0.f ? 1.f / (1.f - dropout_p) : 1.f;
  // additive block: d = dL/dA (overwritten), d_wa / d_ba / d_qa accumulated
  if (int rc = nrms_additive_bwd(d_out, s.a, n_texts, L, wa, qa, s.t, b.d, d_wa, d_ba, d_qa, b.add_ws, b.add_bytes, mode,
                                 st))
    return rc;
  // through dropout #2 and the ReLU; d_b += colsum(dconv)
  {
    const int64_t rpb = 64;
    cnn_dconv_kernel<<<(unsigned)((rows + rpb - 1) / rpb), DCONV_THREADS, 0, st>>>(b.d, s.h, rows, rpb, d_conv_b,
                                                                                  dropout_p, scale, seed, offset);
    NRMS_LAUNCH_CHECK("cnn_dconv");
  }
  cnn_shift_kernel<<<grid_for(rows * 3 * DV4, 256, 8), 256, 0, st>>>(b.d, L, rows, b.dP);
  NRMS_LAUNCH_CHECK("cnn_shift");
  cnn_permute_taps_kernel<<<grid_for(D * D3, 256, 4), 256, 0, st>>>(conv_w, b.wcat, tc ? 1 : 0);
  NRMS_LAUNCH_CHECK("cnn_permute_taps");
  if (tc) {
    // d_W[:, w*300 .. +300] += dP_w^T X = NT(dP^T [w*300 .. +300, rows], X^T [300, rows]), split along rows
    if (int rc = transpose_f32(b.dP, D3, b.t1, b.ldr, rows, D3, st)) return rc;
    if (int rc = transpose_f32(s.x, D, b.t2, b.ldr, rows, D, st)) return rc;
    for (int w = 0; w < 3; ++w)
      if (int rc = tc_gemm_nt_ex(b.t1 + (int64_t)w * D * b.ldr, b.ldr, b.t2, b.ldr, nullptr, d_conv_w + w * D, D3, D, D,
                                 (int)rows, tc_gemm_auto_splits(D, D, (int)rows), TC_EPI_ATOMIC, st))
        return rc;
    // dX = dP Wcat = NT(dP [rows, 900], WcatT [300, 900]) (dconv is no longer needed: dX takes its buffer)
    if (int rc = tc_gemm_nt_ex(b.dP, D3, b.wcat, D3, nullptr, b.d, D, rows, D, D3, 1, TC_EPI_STORE, st)) return rc;
  } else {
    int splits = (int)((rows + 4095) / 4096);
    if (splits > 64) splits = 64;
    for (int w = 0; w < 3; ++w) {
      cudaError_t e = sgemm_launch<1, 1, EPI_ATOMIC>(b.dP + w * D, D3, s.x, D, nullptr, d_conv_w + w * D, D3, D, D, rows,
                                                     splits, st);
      if (e != cudaSuccess) return cuda_fail(e, "sgemm dW conv");
    }
    cudaError_t e = sgemm_launch<0, 1, EPI_STORE>(b.dP, D3, b.wcat, D, nullptr, b.d, D, rows, D, D3, 1, st);
    if (e != cudaSuccess) return cuda_fail(e, "sgemm dX conv");
  }
  cnn_scatter_kernel<<<grid_for(rows, 8, 16), 256, 0, st>>>(tokens, news_rows, L, rows, b.d, d_emb, dropout_p, scale,
                                                            seed, offset);
  NRMS_LAUNCH_CHECK("cnn_scatter");
  return NRMS_OK;
}

}  // extern "C"
