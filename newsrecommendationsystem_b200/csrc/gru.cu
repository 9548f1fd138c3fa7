// LSTUR's user encoder (reference src/model/LSTUR/user_encoder.py): one-layer nn.GRU over the first `length` rows of
// each sequence (pack_padded_sequence), started from h0 -- forward and backward (BPTT), both arithmetic modes.  Also the
// row gather of LSTUR's embeddings (category and user rows, the user rows under the model's whole-row dropout2d mask).
//
// Equations (torch's gate order r, z, n):
//   gi = W_ih x_t + b_ih,  gh = W_hh h + b_hh,  r = sig(gi_r + gh_r),  z = sig(gi_z + gh_z),
//   n = tanh(gi_n + r * gh_n),  h' = (1 - z) * n + z * h.
// Mapping.
//   - The input projection GI = X W_ih^T + b_ih runs once over every input row (tcgen05 tc_gemm_nt in tensor mode, the
//     CUDA-core SGEMM in FP32 mode).  In the indexed form the rows are a news-vector table and step t of sequence s reads
//     the projected row x_rows[s*T + t]: the history rows are never projected one by one.
//   - The sequences are sorted by length, descending, on the host (the lengths are host memory), so the sequences still
//     running at step t are a prefix of the sorted order.  A step is one GEMM GH = h W_hh^T over that prefix and one gate
//     kernel, which adds b_hh and the step's GI row, applies the gates and writes h in place.  The work is
//     sum(length) * 2 * H * 3H, not n_seq * T.
//   - H = 450 rows are 1,800 bytes, off the GEMMs' 16-byte pitch; every hidden-state operand is kept at a padded pitch
//     HP = roundup(H, 4) whose pad columns are zero (W_hh and W_ih are copied into padded, zero-filled layouts), so the
//     pads contribute nothing to any contraction.  The public tensors keep their [*, H] / [3H, *] shapes.
// Training stash, rows packed step-major (step t's active sequences at rows off_t .. off_t + count_t): h_{t-1} | r | z |
// n | gh_n = W_hn h_{t-1} + b_hn.
// Backward.  Only dh_{t-1} = dh_t * z + dG_h W_hh is sequential: per step, a gate-backward kernel writes dG_h (packed)
// and dG_i (at the input row's dense position) and sets dh <- dh * z, then one GEMM accumulates dG_h W_hh into dh.  After
// the loop: dW_hh += dG_h^T h_prev, db_hh += colsum(dG_h), dW_ih += dG_i^T X, db_ih += colsum(dG_i), dX = dG_i W_ih.
#include <string.h>
#include <vector>
#include "common.cuh"
#include "sgemm.cuh"
#include "tc_api.cuh"

namespace nrms {
namespace gru {

constexpr uint32_t DROPOUT_STREAM_ROW = 3;   // whole-row mask of the embedding rows (streams 1, 2: the text encoders)

struct Dims {
  int64_t n_seq;
  int T, I, H, HP, G;   // G = 3 * HP: the padded gate width
};

static Dims make_dims(int64_t n_seq, int T, int I, int H) {
  Dims d;
  d.n_seq = n_seq;
  d.T = T;
  d.I = I;
  d.H = H;
  d.HP = (H + 3) / 4 * 4;
  d.G = 3 * d.HP;
  return d;
}

static int check_shape(int I, int H, int mode) {
  NRMS_CHECK_ARG(I == 900 && (H == 900 || H == 450), NRMS_E_UNSUPPORTED,
                 "GRU (input %d, hidden %d) unsupported: (900, 900) and (900, 450) are compiled", I, H);
  NRMS_CHECK_ARG(mode == NRMS_MODE_FP32 || mode == NRMS_MODE_TF32, NRMS_E_INVALID, "bad mode %d", mode);
  return NRMS_OK;
}

__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }

// dst[g*HP + j, c] = src[g*H + j, c] for j < H, c < cols; zero in the pad rows j >= H and pad columns c >= cols
// (dst pitch ld_dst >= cols).  transposed = 1 writes dst^T instead: dstT[c, g*HP + j] (pitch ld_dst >= 3*HP).
__global__ void __launch_bounds__(256)
gru_pad_weight_kernel(const float* __restrict__ src, int H, int HP, int cols, float* __restrict__ dst, int64_t ld_dst,
                      int dst_cols, int transposed) {
  const int64_t total = (int64_t)3 * HP * dst_cols;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int row = (int)(e / dst_cols), c = (int)(e - (int64_t)row * dst_cols);   // padded row, column
    const int g = row / HP, j = row - g * HP;
    const float v = (j < H && c < cols) ? src[(int64_t)(g * H + j) * cols + c] : 0.f;
    if (transposed) dst[(int64_t)c * ld_dst + row] = v;
    else dst[(int64_t)row * ld_dst + c] = v;
  }
}

// dst[g*H + j, c] += src[g*HP + j, c] (c < cols): a padded weight gradient added into the public [3H, cols] one
__global__ void __launch_bounds__(256)
gru_unpad_add_kernel(const float* __restrict__ src, int64_t ld_src, int H, int HP, int cols, float* __restrict__ dst) {
  const int64_t total = (int64_t)3 * H * cols;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int row = (int)(e / cols), c = (int)(e - (int64_t)row * cols);
    const int g = row / H, j = row - g * H;
    dst[e] += src[(int64_t)(g * HP + j) * ld_src + c];
  }
}

// sorted-order state in/out: dst[s, j] = src[order[s], j] (gather = 1) or dst[order[s], j] = src[s, j] (gather = 0),
// j < H; src null -> zeros.  Sorted rows have pitch HP, caller rows pitch H.
__global__ void __launch_bounds__(256)
gru_permute_kernel(const float* __restrict__ src, const int32_t* __restrict__ order, int64_t n, int H, int HP,
                   float* __restrict__ dst, int gather) {
  const int64_t total = n * H;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t s = e / H;
    const int j = (int)(e - s * H);
    const int64_t o = order[s];
    if (gather) dst[s * HP + j] = src ? src[o * H + j] : 0.f;
    else dst[o * H + j] = src[s * HP + j];
  }
}

// one step of the forward over the `count` active sorted sequences: gh [count, G] (no bias) -> h [count, HP] in place.
// stash_h / stash_g (nullable, training): h_{t-1} [.., HP] and r | z | n | gh_n [.., 4*HP] at the step's packed rows.
__global__ void __launch_bounds__(256)
gru_step_fwd_kernel(const float* __restrict__ gh, const float* __restrict__ gi, const int64_t* __restrict__ x_rows,
                    const int32_t* __restrict__ order, int t, int T, int64_t count, int H, int HP,
                    const float* __restrict__ b_hh, float* __restrict__ h, float* __restrict__ stash_h,
                    float* __restrict__ stash_g) {
  const int G = 3 * HP;
  const int64_t total = count * H;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t s = e / H;
    const int j = (int)(e - s * H);
    const int64_t pos = (int64_t)order[s] * T + t;
    const float* gir = gi + (x_rows ? x_rows[pos] : pos) * G;
    const float* ghr = gh + s * G;
    const float r = sigmoidf_(gir[j] + ghr[j] + __ldg(b_hh + j));
    const float z = sigmoidf_(gir[HP + j] + ghr[HP + j] + __ldg(b_hh + H + j));
    const float ghn = ghr[2 * HP + j] + __ldg(b_hh + 2 * H + j);
    const float n = tanhf(gir[2 * HP + j] + r * ghn);
    const float hp = h[s * HP + j];
    h[s * HP + j] = (1.f - z) * n + z * hp;
    if (stash_h) {
      stash_h[s * HP + j] = hp;
      float* g = stash_g + s * 4 * HP;
      g[j] = r;
      g[HP + j] = z;
      g[2 * HP + j] = n;
      g[3 * HP + j] = ghn;
    }
  }
}

// one step of the backward: dh [count, HP] (dL/dh_t) -> dh * z in place; dgh [count, G] packed, dgi at the input row's
// dense position [n_seq*T, G].
__global__ void __launch_bounds__(256)
gru_step_bwd_kernel(const float* __restrict__ stash_h, const float* __restrict__ stash_g,
                    const int32_t* __restrict__ order, int t, int T, int64_t count, int H, int HP, float* __restrict__ dh,
                    float* __restrict__ dgh, float* __restrict__ dgi) {
  const int G = 3 * HP;
  const int64_t total = count * H;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t s = e / H;
    const int j = (int)(e - s * H);
    const float* g = stash_g + s * 4 * HP;
    const float r = g[j], z = g[HP + j], n = g[2 * HP + j], ghn = g[3 * HP + j];
    const float hp = stash_h[s * HP + j];
    const float d = dh[s * HP + j];
    const float dnp = d * (1.f - z) * (1.f - n * n);
    const float dzp = d * (hp - n) * z * (1.f - z);
    const float drp = dnp * ghn * r * (1.f - r);
    float* a = dgh + s * G;
    a[j] = drp;
    a[HP + j] = dzp;
    a[2 * HP + j] = dnp * r;
    float* b = dgi + ((int64_t)order[s] * T + t) * G;
    b[j] = drp;
    b[HP + j] = dzp;
    b[2 * HP + j] = dnp;
    dh[s * HP + j] = d * z;
  }
}

// out[g*H + j] += sum_r src[r, g*HP + j] over rows [0, n_rows): 256 columns x a slice of rows per block
__global__ void __launch_bounds__(256)
gru_colsum_kernel(const float* __restrict__ src, int64_t n_rows, int64_t rows_per_block, int H, int HP,
                  float* __restrict__ out) {
  const int col = blockIdx.y * blockDim.x + threadIdx.x;
  if (col >= 3 * HP) return;
  const int g = col / HP, j = col - g * HP;
  if (j >= H) return;
  const int64_t r0 = (int64_t)blockIdx.x * rows_per_block;
  const int64_t r1 = r0 + rows_per_block < n_rows ? r0 + rows_per_block : n_rows;
  float s = 0.f;
  for (int64_t r = r0; r < r1; ++r) s += src[r * 3 * HP + col];
  if (r1 > r0) atomicAdd(out + g * H + j, s);
}

// out[i, c] = src[row(i), c] * m(i), c < width; row(i) = idx ? idx[i] : i; m(i) = whole-row dropout mask (p > 0)
__device__ __forceinline__ float row_mask(int64_t i, float p, float scale, uint64_t seed, uint64_t offset) {
  if (p <= 0.f) return 1.f;
  return dropout_mask4(4 * (uint64_t)i, DROPOUT_STREAM_ROW, p, scale, seed, offset).x;
}

__global__ void __launch_bounds__(256)
rows_fwd_kernel(const float* __restrict__ src, int64_t ld_src, const int64_t* __restrict__ idx, int64_t n, int width,
                float* __restrict__ out, int64_t ld_out, float p, float scale, uint64_t seed, uint64_t offset) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t i = warp; i < n; i += nwarps) {
    const float m = row_mask(i, p, scale, seed, offset);
    const float* s = src + (idx ? idx[i] : i) * ld_src;
    float* o = out + i * ld_out;
    for (int c = lane; c < width; c += 32) o[c] = s[c] * m;
  }
}

// d_src[idx[i], c] += d_out[i, c] * m(i); rows with idx == padding_idx are skipped
__global__ void __launch_bounds__(256)
rows_bwd_kernel(const float* __restrict__ d_out, int64_t ld_dout, const int64_t* __restrict__ idx, int64_t n, int width,
                float* __restrict__ d_src, int64_t ld_dsrc, int64_t padding_idx, float p, float scale, uint64_t seed,
                uint64_t offset) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t i = warp; i < n; i += nwarps) {
    const int64_t r = idx[i];
    if (r == padding_idx) continue;
    const float m = row_mask(i, p, scale, seed, offset);
    if (m == 0.f) continue;
    const float* g = d_out + i * ld_dout;
    float* d = d_src + r * ld_dsrc;
    for (int c = lane; c < width; c += 32) atomicAdd(d + c, g[c] * m);
  }
}

// ---- host side ---------------------------------------------------------------------------------------------------
struct Carver {
  char* p;
  size_t off = 0;
  explicit Carver(void* base) : p(reinterpret_cast<char*>(base)) {}
  void* take_bytes(size_t n) {
    void* r = p + off;
    off += align_up(n, 256);
    return r;
  }
  float* take(size_t nfloat) { return reinterpret_cast<float*>(take_bytes(nfloat * sizeof(float))); }
};

// stash: order [n_seq] int32 | h_prev [n_seq*T, HP] | gates [n_seq*T, 4*HP] (sized for every sequence at length T)
struct Stash {
  int32_t* order;
  float *h, *g;
  size_t bytes;
};
static Stash carve_stash(void* base, const Dims& d) {
  Carver c(base);
  Stash s;
  const size_t rows = (size_t)d.n_seq * d.T;
  s.order = reinterpret_cast<int32_t*>(c.take_bytes((size_t)d.n_seq * sizeof(int32_t)));
  s.h = c.take(rows * d.HP);
  s.g = c.take(rows * 4 * d.HP);
  s.bytes = c.off;
  return s;
}

// forward workspace: W_ih padded [G, I] | W_hh padded [G, HP] | b_ih padded [G] | order (inference) | h [n_seq, HP] |
// gh [n_seq, G] | gi [n_gi_rows, G]
struct FwdWs {
  float *wih, *whh, *bih, *h, *gh, *gi;
  int32_t* order;
  size_t bytes;
};
static FwdWs carve_fwd(void* base, const Dims& d, int64_t n_gi_rows) {
  Carver c(base);
  FwdWs f;
  f.wih = c.take((size_t)d.G * d.I);
  f.whh = c.take((size_t)d.G * d.HP);
  f.bih = c.take((size_t)d.G);
  f.order = reinterpret_cast<int32_t*>(c.take_bytes((size_t)d.n_seq * sizeof(int32_t)));
  f.h = c.take((size_t)d.n_seq * d.HP);
  f.gh = c.take((size_t)d.n_seq * d.G);
  f.gi = c.take((size_t)n_gi_rows * d.G);
  f.bytes = c.off;
  return f;
}

// backward workspace: W_ih padded [G, I] (FP32) or its transpose [I, G] (tensor) | W_hh padded [G, HP] or transpose
// [HP, G] | dh [n_seq, HP] | dgh [n_seq*T, G] (packed) | dgi [n_seq*T, G] (dense) | dW_ih padded [G, I] |
// dW_hh padded [G, HP] | tensor mode: t1 [G, ldr] | t2 [max(I, HP), ldr] (K-major copies of the weight-gradient operands)
struct BwdWs {
  float *wih, *whh, *dh, *dgh, *dgi, *dwih, *dwhh, *t1, *t2;
  int64_t ldr;
  size_t bytes;
};
static BwdWs carve_bwd(void* base, const Dims& d, int mode) {
  Carver c(base);
  BwdWs b;
  const size_t rows = (size_t)d.n_seq * d.T;
  b.wih = c.take((size_t)d.G * d.I);
  b.whh = c.take((size_t)d.G * d.HP);
  b.dh = c.take((size_t)d.n_seq * d.HP);
  b.dgh = c.take(rows * d.G);
  b.dgi = c.take(rows * d.G);
  b.dwih = c.take((size_t)d.G * d.I);
  b.dwhh = c.take((size_t)d.G * d.HP);
  b.ldr = ((int64_t)rows + 3) / 4 * 4;
  b.t1 = b.t2 = nullptr;
  if (mode == NRMS_MODE_TF32) {
    b.t1 = c.take((size_t)b.ldr * d.G);
    b.t2 = c.take((size_t)b.ldr * (d.I > d.HP ? d.I : d.HP));
  }
  b.bytes = c.off;
  return b;
}

static unsigned grid_for(int64_t work, int64_t per_block, int cap_per_sm) {
  int64_t g = (work + per_block - 1) / per_block;
  const int64_t cap = (int64_t)num_sms() * cap_per_sm;
  if (g > cap) g = cap;
  return (unsigned)(g > 0 ? g : 1);
}

// Sequences sorted by length, descending (stable); count[t] = sequences with length > t; off[t] = sum of count[< t].
struct Schedule {
  std::vector<int32_t> order;
  std::vector<int64_t> count, off;
  int64_t rows = 0;
};
static int make_schedule(const int32_t* lengths, int64_t n_seq, int T, Schedule& s) {
  NRMS_CHECK_ARG(lengths != nullptr, NRMS_E_INVALID, "null lengths");
  std::vector<int64_t> hist(T + 2, 0);
  for (int64_t i = 0; i < n_seq; ++i) {
    NRMS_CHECK_ARG(lengths[i] >= 0 && lengths[i] <= T, NRMS_E_INVALID, "length %d of sequence %lld outside 0..%d",
                   lengths[i], (long long)i, T);
    ++hist[lengths[i]];
  }
  std::vector<int64_t> start(T + 2, 0);     // first sorted slot of each length, longest first
  for (int l = T - 1; l >= 0; --l) start[l] = start[l + 1] + hist[l + 1];
  s.order.assign(n_seq, 0);
  for (int64_t i = 0; i < n_seq; ++i) s.order[start[lengths[i]]++] = (int32_t)i;
  s.count.assign(T, 0);
  s.off.assign(T, 0);
  int64_t run = n_seq - hist[0];
  for (int t = 0; t < T; ++t) {
    s.count[t] = run;
    run -= hist[t + 1];
  }
  for (int t = 1; t < T; ++t) s.off[t] = s.off[t - 1] + s.count[t - 1];
  s.rows = T > 0 ? s.off[T - 1] + s.count[T - 1] : 0;
  return NRMS_OK;
}

// C[M, N] = A[M, K] B[N, K]^T (+ bias), both modes
static int gemm_nt(const float* A, int64_t lda, const float* B, int64_t ldb, const float* bias, float* C, int64_t ldc,
                   int64_t M, int N, int K, int mode, cudaStream_t st) {
  if (M <= 0) return NRMS_OK;
  if (mode == NRMS_MODE_TF32) return tc_gemm_nt(A, lda, B, ldb, bias, C, ldc, M, N, K, st);
  cudaError_t e = sgemm_launch<0, 0, EPI_STORE>(A, lda, B, ldb, bias, C, ldc, M, N, K, 1, st);
  return e == cudaSuccess ? NRMS_OK : cuda_fail(e, "sgemm gru");
}

// C[M, N] = A^T B with A [K, M] (lda), B [K, N] (ldb), C zeroed first; tensor mode through K-major copies t1 / t2
static int gemm_tn_store(const float* A, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc, int M, int N,
                         int64_t K, int mode, float* t1, float* t2, int64_t ldr, cudaStream_t st) {
  NRMS_CUDA(cudaMemsetAsync(C, 0, (size_t)M * ldc * sizeof(float), st));
  if (K <= 0) return NRMS_OK;
  if (mode == NRMS_MODE_TF32) {
    if (int rc = transpose_f32(A, lda, t1, ldr, K, M, st)) return rc;
    if (int rc = transpose_f32(B, ldb, t2, ldr, K, N, st)) return rc;
    return tc_gemm_nt_ex(t1, ldr, t2, ldr, nullptr, C, ldc, M, N, (int)K, tc_gemm_auto_splits(M, N, (int)K),
                         TC_EPI_ATOMIC, st);
  }
  int splits = (int)((K + 4095) / 4096);
  if (splits > 64) splits = 64;
  cudaError_t e = sgemm_launch<1, 1, EPI_ATOMIC>(A, lda, B, ldb, nullptr, C, ldc, M, N, K, splits, st);
  return e == cudaSuccess ? NRMS_OK : cuda_fail(e, "sgemm gru dW");
}

static int colsum(const float* src, int64_t n_rows, const Dims& d, float* out, cudaStream_t st) {
  if (n_rows <= 0) return NRMS_OK;
  const int64_t rpb = 128;
  dim3 grid((unsigned)((n_rows + rpb - 1) / rpb), (unsigned)((d.G + 255) / 256));
  gru_colsum_kernel<<<grid, 256, 0, st>>>(src, n_rows, rpb, d.H, d.HP, out);
  NRMS_LAUNCH_CHECK("gru_colsum");
  return NRMS_OK;
}

// The sorted order goes to the device from a pinned staging buffer (one per device and host thread), so the copy is
// queued like a kernel and the host keeps running ahead of the GPU; a pageable source may make the host wait for the
// stream.  Before the buffer is rewritten, the host waits for the previous copy out of it (long done in the common case:
// it was queued one training step or one call earlier).
struct PinnedOrder {
  int32_t* p = nullptr;
  size_t cap = 0;
  cudaEvent_t done = nullptr;
};
static int upload_order(const Schedule& s, int32_t* order, cudaStream_t st) {
  static thread_local PinnedOrder bufs[64];
  int dev = 0;
  NRMS_CUDA(cudaGetDevice(&dev));
  NRMS_CHECK_ARG(dev >= 0 && dev < 64, NRMS_E_INVALID, "device ordinal %d", dev);
  PinnedOrder& b = bufs[dev];
  const size_t n = s.order.size();
  if (b.done) NRMS_CUDA(cudaEventSynchronize(b.done));
  else NRMS_CUDA(cudaEventCreateWithFlags(&b.done, cudaEventDisableTiming));
  if (n > b.cap) {
    if (b.p) NRMS_CUDA(cudaFreeHost(b.p));
    b.p = nullptr;
    b.cap = 0;
    NRMS_CUDA(cudaMallocHost(reinterpret_cast<void**>(&b.p), n * sizeof(int32_t)));
    b.cap = n;
  }
  memcpy(b.p, s.order.data(), n * sizeof(int32_t));
  NRMS_CUDA(cudaMemcpyAsync(order, b.p, n * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  NRMS_CUDA(cudaEventRecord(b.done, st));
  return NRMS_OK;
}

}  // namespace gru
}  // namespace nrms

using namespace nrms;
using namespace nrms::gru;

extern "C" {

size_t nrms_gru_stash_bytes(int64_t n_seq, int T, int I, int H) {
  if (n_seq <= 0 || T <= 0 || I <= 0 || H <= 0) return 0;
  return gru::carve_stash(nullptr, make_dims(n_seq, T, I, H)).bytes;
}

size_t nrms_gru_fwd_workspace_bytes(int64_t n_seq, int T, int64_t n_x_rows, int I, int H) {
  if (n_seq <= 0 || T <= 0 || I <= 0 || H <= 0 || n_x_rows < 0) return 0;
  return carve_fwd(nullptr, make_dims(n_seq, T, I, H), n_x_rows).bytes;
}

size_t nrms_gru_bwd_workspace_bytes(int64_t n_seq, int T, int I, int H, int mode) {
  if (n_seq <= 0 || T <= 0 || I <= 0 || H <= 0) return 0;
  return carve_bwd(nullptr, make_dims(n_seq, T, I, H), mode).bytes;
}

int nrms_gru_fwd(const float* x, int64_t n_x_rows, const int64_t* x_rows, int64_t n_seq, int T, int I, int H,
                 const int32_t* lengths, const float* h0, const float* w_ih, const float* w_hh, const float* b_ih,
                 const float* b_hh, float* h_out, void* stash, void* workspace, size_t workspace_bytes, int mode,
                 void* stream) {
  if (int rc = check_shape(I, H, mode)) return rc;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  NRMS_CHECK_ARG(n_seq >= 0 && T >= 1, NRMS_E_INVALID, "bad sizes");
  NRMS_CHECK_ARG(x_rows ? n_x_rows > 0 : n_x_rows == n_seq * T, NRMS_E_INVALID,
                 "bad input rows: %lld for %lld sequences of %d steps", (long long)n_x_rows, (long long)n_seq, T);
  NRMS_CHECK_ARG(!(x_rows && stash), NRMS_E_INVALID, "training takes dense input rows");
  if (n_seq == 0) return NRMS_OK;
  NRMS_CHECK_ARG(x && w_ih && w_hh && b_ih && b_hh && h_out, NRMS_E_INVALID, "null pointer");
  NRMS_CHECK_ARG(aligned16(x) && aligned16(stash) && aligned16(workspace), NRMS_E_INVALID,
                 "pointers must be 16-byte aligned");
  const Dims d = make_dims(n_seq, T, I, H);
  Schedule sc;
  if (int rc = make_schedule(lengths, n_seq, T, sc)) return rc;
  const FwdWs f = carve_fwd(workspace, d, n_x_rows);
  NRMS_CHECK_ARG(workspace && workspace_bytes >= f.bytes, NRMS_E_WORKSPACE, "workspace too small: need %zu bytes",
                 f.bytes);
  const Stash s = gru::carve_stash(stash, d);
  int32_t* order = stash ? s.order : f.order;
  if (int rc = upload_order(sc, order, st)) return rc;
  gru_pad_weight_kernel<<<grid_for((int64_t)d.G * I, 256, 4), 256, 0, st>>>(w_ih, H, d.HP, I, f.wih, I, I, 0);
  NRMS_LAUNCH_CHECK("gru_pad_weight");
  gru_pad_weight_kernel<<<grid_for((int64_t)d.G * d.HP, 256, 4), 256, 0, st>>>(w_hh, H, d.HP, H, f.whh, d.HP, d.HP, 0);
  NRMS_LAUNCH_CHECK("gru_pad_weight");
  gru_pad_weight_kernel<<<grid_for(d.G, 256, 4), 256, 0, st>>>(b_ih, H, d.HP, 1, f.bih, 1, 1, 0);
  NRMS_LAUNCH_CHECK("gru_pad_weight");
  // GI over every input row (table rows in the indexed form)
  if (int rc = gemm_nt(x, I, f.wih, I, f.bih, f.gi, d.G, n_x_rows, d.G, I, mode, st)) return rc;
  NRMS_CUDA(cudaMemsetAsync(f.h, 0, (size_t)n_seq * d.HP * sizeof(float), st));
  gru_permute_kernel<<<grid_for(n_seq * H, 256, 8), 256, 0, st>>>(h0, order, n_seq, H, d.HP, f.h, 1);
  NRMS_LAUNCH_CHECK("gru_permute");
  for (int t = 0; t < T; ++t) {
    const int64_t cnt = sc.count[t];
    if (cnt == 0) break;
    if (int rc = gemm_nt(f.h, d.HP, f.whh, d.HP, nullptr, f.gh, d.G, cnt, d.G, d.HP, mode, st)) return rc;
    float* sh = stash ? s.h + sc.off[t] * d.HP : nullptr;
    float* sg = stash ? s.g + sc.off[t] * 4 * d.HP : nullptr;
    gru_step_fwd_kernel<<<grid_for(cnt * H, 256, 8), 256, 0, st>>>(f.gh, f.gi, x_rows, order, t, T, cnt, H, d.HP, b_hh,
                                                                  f.h, sh, sg);
    NRMS_LAUNCH_CHECK("gru_step_fwd");
  }
  gru_permute_kernel<<<grid_for(n_seq * H, 256, 8), 256, 0, st>>>(f.h, order, n_seq, H, d.HP, h_out, 0);
  NRMS_LAUNCH_CHECK("gru_permute");
  return NRMS_OK;
}

int nrms_gru_bwd(const float* d_out, const float* x, int64_t n_seq, int T, int I, int H, const int32_t* lengths,
                 const float* w_ih, const float* w_hh, const void* stash, float* d_x, float* d_h0, float* d_w_ih,
                 float* d_w_hh, float* d_b_ih, float* d_b_hh, void* workspace, size_t workspace_bytes, int mode,
                 void* stream) {
  if (int rc = check_shape(I, H, mode)) return rc;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  NRMS_CHECK_ARG(n_seq >= 0 && T >= 1, NRMS_E_INVALID, "bad sizes");
  if (n_seq == 0) return NRMS_OK;
  NRMS_CHECK_ARG(d_out && x && w_ih && w_hh && stash && d_w_ih && d_w_hh && d_b_ih && d_b_hh, NRMS_E_INVALID,
                 "null pointer");
  NRMS_CHECK_ARG(aligned16(x) && aligned16(stash) && aligned16(workspace) && aligned16(d_x), NRMS_E_INVALID,
                 "pointers must be 16-byte aligned");
  const Dims d = make_dims(n_seq, T, I, H);
  Schedule sc;
  if (int rc = make_schedule(lengths, n_seq, T, sc)) return rc;
  const BwdWs b = carve_bwd(workspace, d, mode);
  NRMS_CHECK_ARG(workspace && workspace_bytes >= b.bytes, NRMS_E_WORKSPACE, "workspace too small: need %zu bytes",
                 b.bytes);
  const Stash s = gru::carve_stash(const_cast<void*>(stash), d);
  const bool tc = mode == NRMS_MODE_TF32;
  const int64_t rows = n_seq * T;
  // the per-step dh GEMM and dX read W_hh / W_ih as their B operand: K-major ([HP, G] / [I, G]) on the tensor cores
  gru_pad_weight_kernel<<<grid_for((int64_t)d.G * d.HP, 256, 4), 256, 0, st>>>(w_hh, H, d.HP, H, b.whh,
                                                                              tc ? d.G : d.HP, d.HP, tc ? 1 : 0);
  NRMS_LAUNCH_CHECK("gru_pad_weight");
  gru_pad_weight_kernel<<<grid_for((int64_t)d.G * I, 256, 4), 256, 0, st>>>(w_ih, H, d.HP, I, b.wih, tc ? d.G : I, I,
                                                                           tc ? 1 : 0);
  NRMS_LAUNCH_CHECK("gru_pad_weight");
  NRMS_CUDA(cudaMemsetAsync(b.dh, 0, (size_t)n_seq * d.HP * sizeof(float), st));
  NRMS_CUDA(cudaMemsetAsync(b.dgh, 0, (size_t)rows * d.G * sizeof(float), st));
  NRMS_CUDA(cudaMemsetAsync(b.dgi, 0, (size_t)rows * d.G * sizeof(float), st));
  gru_permute_kernel<<<grid_for(n_seq * H, 256, 8), 256, 0, st>>>(d_out, s.order, n_seq, H, d.HP, b.dh, 1);
  NRMS_LAUNCH_CHECK("gru_permute");
  for (int t = T - 1; t >= 0; --t) {
    const int64_t cnt = sc.count[t];
    if (cnt == 0) continue;
    float* dgh_t = b.dgh + sc.off[t] * d.G;
    gru_step_bwd_kernel<<<grid_for(cnt * H, 256, 8), 256, 0, st>>>(s.h + sc.off[t] * d.HP, s.g + sc.off[t] * 4 * d.HP,
                                                                  s.order, t, T, cnt, H, d.HP, b.dh, dgh_t, b.dgi);
    NRMS_LAUNCH_CHECK("gru_step_bwd");
    // dh[0:cnt] += dG_h W_hh
    if (tc) {
      if (int rc = tc_gemm_nt_ex(dgh_t, d.G, b.whh, d.G, nullptr, b.dh, d.HP, cnt, d.HP, d.G, 1, TC_EPI_ACCUM, st))
        return rc;
    } else {
      cudaError_t e = sgemm_launch<0, 1, EPI_ACCUM>(dgh_t, d.G, b.whh, d.HP, nullptr, b.dh, d.HP, cnt, d.HP, d.G, 1, st);
      if (e != cudaSuccess) return cuda_fail(e, "sgemm gru dh");
    }
  }
  if (d_h0) {
    gru_permute_kernel<<<grid_for(n_seq * H, 256, 8), 256, 0, st>>>(b.dh, s.order, n_seq, H, d.HP, d_h0, 0);
    NRMS_LAUNCH_CHECK("gru_permute");
  }
  // dW_hh += dG_h^T h_prev (packed rows), dW_ih += dG_i^T X (dense rows; the rows past a length are zero)
  if (int rc = gemm_tn_store(b.dgh, d.G, s.h, d.HP, b.dwhh, d.HP, d.G, d.HP, sc.rows, mode, b.t1, b.t2, b.ldr, st))
    return rc;
  gru_unpad_add_kernel<<<grid_for((int64_t)3 * H * H, 256, 4), 256, 0, st>>>(b.dwhh, d.HP, H, d.HP, H, d_w_hh);
  NRMS_LAUNCH_CHECK("gru_unpad_add");
  if (int rc = gemm_tn_store(b.dgi, d.G, x, I, b.dwih, I, d.G, I, rows, mode, b.t1, b.t2, b.ldr, st)) return rc;
  gru_unpad_add_kernel<<<grid_for((int64_t)3 * H * I, 256, 4), 256, 0, st>>>(b.dwih, I, H, d.HP, I, d_w_ih);
  NRMS_LAUNCH_CHECK("gru_unpad_add");
  if (int rc = colsum(b.dgh, sc.rows, d, d_b_hh, st)) return rc;
  if (int rc = colsum(b.dgi, rows, d, d_b_ih, st)) return rc;
  // dX = dG_i W_ih
  if (d_x) {
    if (tc) {
      if (int rc = tc_gemm_nt_ex(b.dgi, d.G, b.wih, d.G, nullptr, d_x, I, rows, I, d.G, 1, TC_EPI_STORE, st)) return rc;
    } else {
      cudaError_t e = sgemm_launch<0, 1, EPI_STORE>(b.dgi, d.G, b.wih, I, nullptr, d_x, I, rows, I, d.G, 1, st);
      if (e != cudaSuccess) return cuda_fail(e, "sgemm gru dX");
    }
  }
  return NRMS_OK;
}

int nrms_rows_fwd(const float* src, int64_t n_src_rows, int64_t ld_src, const int64_t* idx, int64_t n, int width,
                  float* out, int64_t ld_out, float dropout_p, uint64_t seed, uint64_t offset, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  NRMS_CHECK_ARG(n >= 0 && width > 0 && ld_src >= width && ld_out >= width && n_src_rows >= 0, NRMS_E_INVALID,
                 "bad sizes / strides");
  NRMS_CHECK_ARG(idx || n_src_rows >= n, NRMS_E_INVALID, "%lld rows read from %lld", (long long)n,
                 (long long)n_src_rows);
  NRMS_CHECK_ARG(dropout_p >= 0.f && dropout_p < 1.f, NRMS_E_INVALID, "dropout_p out of range");
  if (n == 0) return NRMS_OK;
  NRMS_CHECK_ARG(src && out, NRMS_E_INVALID, "null pointer");
  const float scale = dropout_p > 0.f ? 1.f / (1.f - dropout_p) : 1.f;
  rows_fwd_kernel<<<grid_for(n, 8, 16), 256, 0, st>>>(src, ld_src, idx, n, width, out, ld_out, dropout_p, scale, seed,
                                                      offset);
  NRMS_LAUNCH_CHECK("rows_fwd");
  return NRMS_OK;
}

int nrms_rows_bwd(const float* d_out, int64_t ld_dout, const int64_t* idx, int64_t n, int width, float* d_src,
                  int64_t ld_dsrc, int64_t padding_idx, float dropout_p, uint64_t seed, uint64_t offset, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  NRMS_CHECK_ARG(n >= 0 && width > 0 && ld_dout >= width && ld_dsrc >= width, NRMS_E_INVALID, "bad sizes / strides");
  NRMS_CHECK_ARG(dropout_p >= 0.f && dropout_p < 1.f, NRMS_E_INVALID, "dropout_p out of range");
  if (n == 0) return NRMS_OK;
  NRMS_CHECK_ARG(d_out && idx && d_src, NRMS_E_INVALID, "null pointer");
  const float scale = dropout_p > 0.f ? 1.f / (1.f - dropout_p) : 1.f;
  rows_bwd_kernel<<<grid_for(n, 8, 16), 256, 0, st>>>(d_out, ld_dout, idx, n, width, d_src, ld_dsrc, padding_idx,
                                                      dropout_p, scale, seed, offset);
  NRMS_LAUNCH_CHECK("rows_bwd");
  return NRMS_OK;
}

}  // extern "C"
