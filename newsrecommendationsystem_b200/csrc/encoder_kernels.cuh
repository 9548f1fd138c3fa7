// Device kernels of the decomposed encoder pipeline (everything except the dense contractions):
// embedding gather / scatter, multi-head exp-softmax attention fwd/bwd, additive pooling fwd/bwd,
// deterministic column sums.  Math follows the reference exactly (see include/nrms_b200.h for the
// file:line map): scores = QK^T / sqrt(20); e = exp(scores) (no max subtraction);
// attn = e / (sum e + 1e-8); ctx = attn V; pooling = stable softmax over tanh(linear(c)) . q.
#pragma once
#include <cuda_fp16.h>
#include "common.cuh"

namespace nrms {

constexpr float SQRT_DH = 4.47213595499957939f;  // np.sqrt(20) rounded to fp32 by the cast
constexpr float ATTN_EPS = 1e-8f;
constexpr uint32_t DROPOUT_STREAM_EMB = 1, DROPOUT_STREAM_CTX = 2;

// ----------------------------------------------------------------------------------------
// a1: embedding gather (+ dropout #1).  One warp per token row: 75 coalesced float4.
// ----------------------------------------------------------------------------------------
// news_rows (nullable, with L = tokens per title): the index-only minibatch form (SURVEY 8 f2) -- row r of the batch is
// token r % L of title news_rows[r / L] of the device-resident pre-tokenised table (reference dataset.py:17-85 ships the
// token tensors themselves); null = tokens already holds the batch's own rows.
__device__ __forceinline__ int64_t token_of_row(const int64_t* __restrict__ tokens, const int64_t* __restrict__ news_rows,
                                                int L, int64_t r) {
  return news_rows ? tokens[news_rows[r / L] * L + r % L] : tokens[r];
}

static __global__ void __launch_bounds__(256)
gather_embedding_kernel(const int64_t* __restrict__ tokens, int64_t n_rows, const float* __restrict__ emb,
                        float* __restrict__ x, float p, float scale, uint64_t seed, uint64_t offset,
                        const int64_t* __restrict__ news_rows = nullptr, int L = 1) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t r = warp; r < n_rows; r += nwarps) {
    const int64_t tok = token_of_row(tokens, news_rows, L, r);
    const float4* src = reinterpret_cast<const float4*>(emb + tok * D);
    float4* dst = reinterpret_cast<float4*>(x + r * D);
#pragma unroll
    for (int l = lane; l < DV4; l += 32) {
      float4 v = __ldg(src + l);
      if (p > 0.f) {
        float4 m = dropout_mask4((uint64_t)r * D + 4 * l, DROPOUT_STREAM_EMB, p, scale, seed, offset);
        v.x *= m.x; v.y *= m.y; v.z *= m.z; v.w *= m.w;
      }
      dst[l] = v;
    }
  }
}

// generic row gather with int32/int64 indices (user-encoder indexed input, evaluate tables)
template <typename IdxT>
__global__ void __launch_bounds__(256)
gather_rows_kernel(const float* __restrict__ src, const IdxT* __restrict__ rows, int64_t n, int width4,
                   float* __restrict__ dst) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t r = warp; r < n; r += nwarps) {
    const float4* s = reinterpret_cast<const float4*>(src) + (int64_t)rows[r] * width4;
    float4* d = reinterpret_cast<float4*>(dst) + r * width4;
    for (int l = lane; l < width4; l += 32) d[l] = __ldg(s + l);
  }
}

// the same gather from an fp16 table in pack_rows_f16's layout ([*, 320] halfs, values in columns 0..299): each row's 300
// values widened to an fp32 row of dst [n, 300].  One warp per row, four halfs (8 bytes) per lane and step.
static __global__ void __launch_bounds__(256)
gather_rows_f16_kernel(const __half* __restrict__ src, const int32_t* __restrict__ rows, int64_t n,
                       float* __restrict__ dst) {
  constexpr int SRC_LD = 320;
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t r = warp; r < n; r += nwarps) {
    const uint2* s = reinterpret_cast<const uint2*>(src + (int64_t)rows[r] * SRC_LD);
    float4* d = reinterpret_cast<float4*>(dst) + r * DV4;
    for (int l = lane; l < DV4; l += 32) {
      const uint2 u = __ldg(s + l);
      const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&u.x));
      const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&u.y));
      d[l] = make_float4(a.x, a.y, b.x, b.y);
    }
  }
}

// embedding backward: dE[tok] += dX[row] * mask1 ; token 0 (padding_idx) skipped.
static __global__ void __launch_bounds__(256)
scatter_embedding_grad_kernel(const int64_t* __restrict__ tokens, int64_t n_rows, const float* __restrict__ dx,
                              float* __restrict__ d_emb, float p, float scale, uint64_t seed, uint64_t offset,
                              const int64_t* __restrict__ news_rows = nullptr, int L = 1) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t r = warp; r < n_rows; r += nwarps) {
    const int64_t tok = token_of_row(tokens, news_rows, L, r);
    if (tok == 0) continue;
    const float4* src = reinterpret_cast<const float4*>(dx + r * D);
    float4* dst = reinterpret_cast<float4*>(d_emb + tok * D);
#pragma unroll
    for (int l = lane; l < DV4; l += 32) {
      float4 v = src[l];
      if (p > 0.f) {
        float4 m = dropout_mask4((uint64_t)r * D + 4 * l, DROPOUT_STREAM_EMB, p, scale, seed, offset);
        v.x *= m.x; v.y *= m.y; v.z *= m.z; v.w *= m.w;
      }
      atomicAdd(dst + l, v);
    }
  }
}

// ----------------------------------------------------------------------------------------
// a3/a4: attention forward.  CTA = (sequence, chunk of HC heads); thread = (head, query i).
// K,V slices staged in smem (every read is a warp broadcast), q_i and the context in registers.
// ----------------------------------------------------------------------------------------
template <int S, int HC>
__global__ void __launch_bounds__(((S * HC + 31) / 32) * 32)
attention_fwd_kernel(const float* __restrict__ qkv, float* __restrict__ ctx, int64_t n_seq,
                     float p, float scale, uint64_t seed, uint64_t offset, const int32_t* __restrict__ lengths = nullptr) {
  constexpr int W = HC * DH;  // columns of this head chunk
  extern __shared__ __align__(16) float smem[];
  float* Ks = smem;          // [S][W]
  float* Vs = smem + S * W;  // [S][W]
  const int hc = blockIdx.y;
  const int tid = threadIdx.x;
  const int hl = tid / S, i = tid % S;
  const bool active = tid < S * HC;
  constexpr int W4 = W / 4;

  for (int64_t seq = blockIdx.x; seq < n_seq; seq += gridDim.x) {
    const float* base = qkv + seq * S * D3;
    __syncthreads();
    for (int f = tid; f < S * W4 * 2; f += blockDim.x) {
      int which = f / (S * W4);  // 0 = K, 1 = V
      int g = f % (S * W4);
      int j = g / W4, c4 = g % W4;
      float4 v = *reinterpret_cast<const float4*>(base + (int64_t)j * D3 + (1 + which) * D + hc * W + c4 * 4);
      *reinterpret_cast<float4*>((which ? Vs : Ks) + j * W + c4 * 4) = v;
    }
    __syncthreads();
    if (!active) continue;
    float q[DH], acc[DH];
    {
      const float4* qp = reinterpret_cast<const float4*>(base + (int64_t)i * D3 + hc * W + hl * DH);
#pragma unroll
      for (int c = 0; c < DH / 4; ++c) {
        float4 v = qp[c];
        q[4 * c] = v.x; q[4 * c + 1] = v.y; q[4 * c + 2] = v.z; q[4 * c + 3] = v.w;
      }
    }
#pragma unroll
    for (int d = 0; d < DH; ++d) acc[d] = 0.f;
    float Z = 0.f;
    // `length` mask of multihead_self.py:60-68,18-19: exp(scores) * (j < length) -- keys past the length add nothing
    // to the sum or the context; length <= 0 leaves 0 / (0 + 1e-8) = 0, like the reference
    int jmax = S;
    if (lengths != nullptr) { const int l = lengths[seq]; jmax = l < 0 ? 0 : (l < S ? l : S); }
    // one key per step, but the 20-term dot product runs as five independent 4-term chains (the serial 20-FMA chain
    // left the FMA pipe at ~1/4 of its rate: 4 cycles per dependent FMA and few warps per scheduler)
#pragma unroll 4
    for (int j = 0; j < jmax; ++j) {
      const float4* kp = reinterpret_cast<const float4*>(Ks + j * W + hl * DH);
      float sp[DH / 4];
#pragma unroll
      for (int c = 0; c < DH / 4; ++c) {
        float4 k = kp[c];
        sp[c] = fmaf(q[4 * c + 3], k.w, fmaf(q[4 * c + 2], k.z, fmaf(q[4 * c + 1], k.y, q[4 * c] * k.x)));
      }
      const float s = ((sp[0] + sp[1]) + (sp[2] + sp[3])) + sp[4];
      const float e = expf(s / SQRT_DH);
      Z += e;
      const float4* vp = reinterpret_cast<const float4*>(Vs + j * W + hl * DH);
#pragma unroll
      for (int c = 0; c < DH / 4; ++c) {
        float4 v = vp[c];
        acc[4 * c] = fmaf(e, v.x, acc[4 * c]); acc[4 * c + 1] = fmaf(e, v.y, acc[4 * c + 1]);
        acc[4 * c + 2] = fmaf(e, v.z, acc[4 * c + 2]); acc[4 * c + 3] = fmaf(e, v.w, acc[4 * c + 3]);
      }
    }
    const float inv = 1.f / (Z + ATTN_EPS);
    const int64_t row = seq * S + i;
    const int col = hc * W + hl * DH;
    float4* op = reinterpret_cast<float4*>(ctx + row * D + col);
#pragma unroll
    for (int c = 0; c < DH / 4; ++c) {
      float4 o = make_float4(acc[4 * c] * inv, acc[4 * c + 1] * inv, acc[4 * c + 2] * inv, acc[4 * c + 3] * inv);
      if (p > 0.f) {
        float4 m = dropout_mask4((uint64_t)row * D + col + 4 * c, DROPOUT_STREAM_CTX, p, scale, seed, offset);
        o.x *= m.x; o.y *= m.y; o.z *= m.z; o.w *= m.w;
      }
      op[c] = o;
    }
  }
}

// ----------------------------------------------------------------------------------------
// attention backward.  Phase 1: thread (h,i) computes row i of the scores once (e_ij = exp(s_ij), da_ij = g_i . v_j),
// its Zinv_i and delta_i, then dQ_i, leaving attn_ij and ds_ij in shared memory.  Phase 2: thread (h,j) reads
// column j of both and accumulates dK_j, dV_j -- no score, exponential or dot product is computed twice.
//   attn = e/(Z+eps)  =>  ds_ij = attn_ij (dattn_ij - sum_k attn_ik dattn_ik) / sqrt(d)
// P/DS rows have a pitch of S+1 words: phase 1 (threads = consecutive i, same j) and phase 2 (threads = consecutive j)
// are both bank-conflict free.
// MASKED (the standalone block's `length`): phase 1 runs over the keys j < jmax of the forward kernel and writes attn = 0
// and ds = 0 for the others, so phase 2 gives exactly zero dK / dV rows for masked keys.  Unmasked, `lengths` is unread.
// ----------------------------------------------------------------------------------------
template <int S, int HC, bool MASKED = false>
__global__ void __launch_bounds__(((S * HC + 31) / 32) * 32)
attention_bwd_kernel(const float* __restrict__ qkv, const float* __restrict__ d_ctx, float* __restrict__ d_qkv,
                     int64_t n_seq, float p, float scale, uint64_t seed, uint64_t offset,
                     const int32_t* __restrict__ lengths = nullptr) {
  constexpr int W = HC * DH;
  constexpr int W4 = W / 4;
  constexpr int SP = S + 1;
  constexpr float INV_SQRT_DH = 1.f / SQRT_DH;
  extern __shared__ __align__(16) float smem[];
  float* Qs = smem;
  float* Ks = Qs + S * W;
  float* Vs = Ks + S * W;
  float* Gs = Vs + S * W;     // d_ctx (after dropout-2 mask)
  float* Ps = Gs + S * W;     // [HC*S][S+1] e, then attn
  float* Ds = Ps + HC * S * SP;   // [HC*S][S+1] da, then ds
  const int hc = blockIdx.y;
  const int tid = threadIdx.x;
  const int hl = tid / S, i = tid % S;
  const bool active = tid < S * HC;

  for (int64_t seq = blockIdx.x; seq < n_seq; seq += gridDim.x) {
    const float* base = qkv + seq * S * D3;
    __syncthreads();
    for (int f = tid; f < S * W4 * 4; f += blockDim.x) {
      int which = f / (S * W4);  // 0 Q, 1 K, 2 V, 3 dCtx
      int g = f % (S * W4);
      int j = g / W4, c4 = g % W4;
      float4 v;
      if (which < 3) {
        v = *reinterpret_cast<const float4*>(base + (int64_t)j * D3 + which * D + hc * W + c4 * 4);
      } else {
        const int64_t row = seq * S + j;
        const int col = hc * W + c4 * 4;
        v = *reinterpret_cast<const float4*>(d_ctx + row * D + col);
        if (p > 0.f) {
          float4 m = dropout_mask4((uint64_t)row * D + col, DROPOUT_STREAM_CTX, p, scale, seed, offset);
          v.x *= m.x; v.y *= m.y; v.z *= m.z; v.w *= m.w;
        }
      }
      *reinterpret_cast<float4*>(smem + which * S * W + j * W + c4 * 4) = v;
    }
    __syncthreads();

    float a[DH], b[DH], r[DH];
    // ---- phase 1 ---------------------------------------------------------------------
    if (active) {
      float* prow = Ps + (hl * S + i) * SP;
      float* drow = Ds + (hl * S + i) * SP;
#pragma unroll
      for (int d = 0; d < DH; ++d) { a[d] = Qs[i * W + hl * DH + d]; b[d] = Gs[i * W + hl * DH + d]; r[d] = 0.f; }
      float Z = 0.f, num = 0.f;
      int jmax = S;
      if (MASKED) { const int l = lengths[seq]; jmax = l < 0 ? 0 : (l < S ? l : S); }
#pragma unroll 4
      for (int j = 0; j < jmax; ++j) {
        const float4* kp = reinterpret_cast<const float4*>(Ks + j * W + hl * DH);
        const float4* vp = reinterpret_cast<const float4*>(Vs + j * W + hl * DH);
        float sp[DH / 4], dp[DH / 4];      // five independent 4-term chains per dot product, in the forward's order
#pragma unroll
        for (int c = 0; c < DH / 4; ++c) {
          float4 k = kp[c], v = vp[c];
          sp[c] = fmaf(a[4 * c + 3], k.w, fmaf(a[4 * c + 2], k.z, fmaf(a[4 * c + 1], k.y, a[4 * c] * k.x)));
          dp[c] = fmaf(b[4 * c + 3], v.w, fmaf(b[4 * c + 2], v.z, fmaf(b[4 * c + 1], v.y, b[4 * c] * v.x)));
        }
        const float s = ((sp[0] + sp[1]) + (sp[2] + sp[3])) + sp[4];
        const float da = ((dp[0] + dp[1]) + (dp[2] + dp[3])) + dp[4];
        const float e = expf(s / SQRT_DH);      // same expression as the forward kernel
        Z += e;
        num = fmaf(e, da, num);
        prow[j] = e;
        drow[j] = da;
      }
      const float zinv = 1.f / (Z + ATTN_EPS);
      const float delta = num * zinv;
#pragma unroll 4
      for (int j = 0; j < jmax; ++j) {
        const float4* kp = reinterpret_cast<const float4*>(Ks + j * W + hl * DH);
        const float at = prow[j] * zinv;
        const float ds = at * (drow[j] - delta) * INV_SQRT_DH;
        prow[j] = at;
        drow[j] = ds;
#pragma unroll
        for (int c = 0; c < DH / 4; ++c) {
          float4 k = kp[c];
          r[4 * c] = fmaf(ds, k.x, r[4 * c]); r[4 * c + 1] = fmaf(ds, k.y, r[4 * c + 1]);
          r[4 * c + 2] = fmaf(ds, k.z, r[4 * c + 2]); r[4 * c + 3] = fmaf(ds, k.w, r[4 * c + 3]);
        }
      }
      if (MASKED)
        for (int j = jmax; j < S; ++j) prow[j] = drow[j] = 0.f;
      float4* op = reinterpret_cast<float4*>(d_qkv + (seq * S + i) * D3 + hc * W + hl * DH);
#pragma unroll
      for (int c = 0; c < DH / 4; ++c) op[c] = make_float4(r[4 * c], r[4 * c + 1], r[4 * c + 2], r[4 * c + 3]);
    }
    __syncthreads();
    // ---- phase 2 (thread index i now plays the key/value row j) ---------------------------
    if (active) {
      const int j = i;
      const float* pcol = Ps + hl * S * SP + j;
      const float* dcol = Ds + hl * S * SP + j;
#pragma unroll
      for (int d = 0; d < DH; ++d) { a[d] = 0.f; b[d] = 0.f; }     // a = dK_j, b = dV_j
#pragma unroll 4
      for (int ii = 0; ii < S; ++ii) {
        const float4* qp = reinterpret_cast<const float4*>(Qs + ii * W + hl * DH);
        const float4* gp = reinterpret_cast<const float4*>(Gs + ii * W + hl * DH);
        const float at = pcol[ii * SP];
        const float ds = dcol[ii * SP];
#pragma unroll
        for (int c = 0; c < DH / 4; ++c) {
          float4 qv = qp[c], g = gp[c];
          a[4 * c] = fmaf(ds, qv.x, a[4 * c]); a[4 * c + 1] = fmaf(ds, qv.y, a[4 * c + 1]);
          a[4 * c + 2] = fmaf(ds, qv.z, a[4 * c + 2]); a[4 * c + 3] = fmaf(ds, qv.w, a[4 * c + 3]);
          b[4 * c] = fmaf(at, g.x, b[4 * c]); b[4 * c + 1] = fmaf(at, g.y, b[4 * c + 1]);
          b[4 * c + 2] = fmaf(at, g.z, b[4 * c + 2]); b[4 * c + 3] = fmaf(at, g.w, b[4 * c + 3]);
        }
      }
      float* orow = d_qkv + (seq * S + j) * D3 + hc * W + hl * DH;
      float4* ok = reinterpret_cast<float4*>(orow + D);
      float4* ov = reinterpret_cast<float4*>(orow + 2 * D);
#pragma unroll
      for (int c = 0; c < DH / 4; ++c) {
        ok[c] = make_float4(a[4 * c], a[4 * c + 1], a[4 * c + 2], a[4 * c + 3]);
        ov[c] = make_float4(b[4 * c], b[4 * c + 1], b[4 * c + 2], b[4 * c + 3]);
      }
    }
  }
}

// ----------------------------------------------------------------------------------------
// a5: additive pooling forward.  t holds linear(c)+bias on entry and tanh(.) on exit.
// ----------------------------------------------------------------------------------------
template <int S>
__global__ void __launch_bounds__(256)
additive_fwd_kernel(const float* __restrict__ c, float* __restrict__ t, const float* __restrict__ qa,
                    float* __restrict__ w, float* __restrict__ out, int64_t n_seq) {
  __shared__ float sc[S];
  __shared__ float wv[S];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int64_t seq = blockIdx.x; seq < n_seq; seq += gridDim.x) {
    for (int i = warp; i < S; i += 8) {
      float* trow = t + (seq * S + i) * QD;
      float part = 0.f;
      for (int q = lane; q < QD; q += 32) {
        float v = tanhf(trow[q]);
        trow[q] = v;
        part = fmaf(v, __ldg(qa + q), part);
      }
      part = warp_sum(part);
      if (lane == 0) sc[i] = part;
    }
    __syncthreads();
    if (warp == 0) {
      float m = -INFINITY;
      for (int i = lane; i < S; i += 32) m = fmaxf(m, sc[i]);
      m = warp_max(m);
      float sum = 0.f;
      for (int i = lane; i < S; i += 32) { float e = expf(sc[i] - m); wv[i] = e; sum += e; }
      sum = warp_sum(sum);
      for (int i = lane; i < S; i += 32) { float x = wv[i] / sum; wv[i] = x; w[seq * S + i] = x; }
    }
    __syncthreads();
    for (int d = tid; d < D; d += 256) {
      const float* cp = c + seq * S * D + d;
      float acc = 0.f;
#pragma unroll 5
      for (int i = 0; i < S; ++i) acc = fmaf(wv[i], cp[(int64_t)i * D], acc);
      out[seq * D + d] = acc;
    }
    __syncthreads();
  }
}

// additive pooling backward (everything except the two contractions dU*Wa and dU^T*C):
//   d_c[i,:]  = w_i * d_out           (first term; the GEMM adds dU * Wa afterwards)
//   d_u[i,q]  = ds_i * qa[q] * (1 - t^2)
//   partial_dqa[block, q] = sum over this block's sequences of ds_i * t[i,q]
//   partial_dqa[gridDim.x + block, q] = sum over this block's rows of d_u[i,q]   (the bias gradient: no colsum pass)
template <int S>
__global__ void __launch_bounds__(256)
additive_bwd_kernel(const float* __restrict__ d_out, const float* __restrict__ c, const float* __restrict__ t,
                    const float* __restrict__ w, const float* __restrict__ qa,
                    float* __restrict__ d_c, float* __restrict__ d_u, float* __restrict__ partial_dqa,
                    int64_t n_seq) {
  __shared__ float dwv[S];
  __shared__ float dsv[S];
  __shared__ float wv[S];
  __shared__ __align__(16) float go[D];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  float dqa_acc = 0.f, dba_acc = 0.f;
  const float qv = (tid < QD) ? qa[tid] : 0.f;
  for (int64_t seq = blockIdx.x; seq < n_seq; seq += gridDim.x) {
    for (int d = tid; d < D; d += 256) go[d] = d_out[seq * D + d];
    if (tid < S) wv[tid] = w[seq * S + tid];
    __syncthreads();
    for (int i = warp; i < S; i += 8) {
      const float* cp = c + (seq * S + i) * D;
      float part = 0.f;
      for (int d = lane; d < D; d += 32) part = fmaf(go[d], cp[d], part);
      part = warp_sum(part);
      if (lane == 0) dwv[i] = part;
    }
    __syncthreads();
    if (warp == 0) {
      float dot = 0.f;
      for (int i = lane; i < S; i += 32) dot = fmaf(wv[i], dwv[i], dot);
      dot = warp_sum(dot);
      for (int i = lane; i < S; i += 32) dsv[i] = wv[i] * (dwv[i] - dot);
    }
    __syncthreads();
    if (tid < QD) {
      for (int i = 0; i < S; ++i) {
        const int64_t row = seq * S + i;
        const float tv = t[row * QD + tid];
        const float ds = dsv[i];
        const float du = ds * qv * (1.f - tv * tv);
        d_u[row * QD + tid] = du;
        dba_acc += du;
        dqa_acc = fmaf(ds, tv, dqa_acc);
      }
    }
    for (int f = tid; f < S * DV4; f += 256) {
      const int i = f / DV4, l = f % DV4;
      const float wi = wv[i];
      float4 g = *reinterpret_cast<const float4*>(go + 4 * l);
      *reinterpret_cast<float4*>(d_c + (seq * S + i) * D + 4 * l) = make_float4(wi * g.x, wi * g.y, wi * g.z, wi * g.w);
    }
    __syncthreads();
  }
  if (tid < QD) {
    partial_dqa[(int64_t)blockIdx.x * QD + tid] = dqa_acc;
    partial_dqa[(int64_t)(gridDim.x + blockIdx.x) * QD + tid] = dba_acc;
  }
}

// The two additive kernels above with the sequence length passed at run time, 1 <= S <= ADD_MAXS: the user encoder at
// any history length and the standalone block at any candidate count.  The compiled lengths keep their templates.
constexpr int ADD_MAXS = 64;

static __global__ void __launch_bounds__(256)
additive_fwd_rt_kernel(const float* __restrict__ c, float* __restrict__ t, const float* __restrict__ qa,
                       float* __restrict__ w, float* __restrict__ out, int64_t n_seq, int S) {
  __shared__ float sc[ADD_MAXS];
  __shared__ float wv[ADD_MAXS];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int64_t seq = blockIdx.x; seq < n_seq; seq += gridDim.x) {
    for (int i = warp; i < S; i += 8) {
      float* trow = t + (seq * S + i) * QD;
      float part = 0.f;
      for (int q = lane; q < QD; q += 32) {
        float v = tanhf(trow[q]);
        trow[q] = v;
        part = fmaf(v, __ldg(qa + q), part);
      }
      part = warp_sum(part);
      if (lane == 0) sc[i] = part;
    }
    __syncthreads();
    if (warp == 0) {
      float m = -INFINITY;
      for (int i = lane; i < S; i += 32) m = fmaxf(m, sc[i]);
      m = warp_max(m);
      float sum = 0.f;
      for (int i = lane; i < S; i += 32) { float e = expf(sc[i] - m); wv[i] = e; sum += e; }
      sum = warp_sum(sum);
      for (int i = lane; i < S; i += 32) { float x = wv[i] / sum; wv[i] = x; w[seq * S + i] = x; }
    }
    __syncthreads();
    for (int d = tid; d < D; d += 256) {
      const float* cp = c + seq * S * D + d;
      float acc = 0.f;
#pragma unroll 5
      for (int i = 0; i < S; ++i) acc = fmaf(wv[i], cp[(int64_t)i * D], acc);
      out[seq * D + d] = acc;
    }
    __syncthreads();
  }
}

static __global__ void __launch_bounds__(256)
additive_bwd_rt_kernel(const float* __restrict__ d_out, const float* __restrict__ c, const float* __restrict__ t,
                       const float* __restrict__ w, const float* __restrict__ qa,
                       float* __restrict__ d_c, float* __restrict__ d_u, float* __restrict__ partial_dqa,
                       int64_t n_seq, int S) {
  __shared__ float dwv[ADD_MAXS];
  __shared__ float dsv[ADD_MAXS];
  __shared__ float wv[ADD_MAXS];
  __shared__ __align__(16) float go[D];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  float dqa_acc = 0.f, dba_acc = 0.f;
  const float qv = (tid < QD) ? qa[tid] : 0.f;
  for (int64_t seq = blockIdx.x; seq < n_seq; seq += gridDim.x) {
    for (int d = tid; d < D; d += 256) go[d] = d_out[seq * D + d];
    if (tid < S) wv[tid] = w[seq * S + tid];
    __syncthreads();
    for (int i = warp; i < S; i += 8) {
      const float* cp = c + (seq * S + i) * D;
      float part = 0.f;
      for (int d = lane; d < D; d += 32) part = fmaf(go[d], cp[d], part);
      part = warp_sum(part);
      if (lane == 0) dwv[i] = part;
    }
    __syncthreads();
    if (warp == 0) {
      float dot = 0.f;
      for (int i = lane; i < S; i += 32) dot = fmaf(wv[i], dwv[i], dot);
      dot = warp_sum(dot);
      for (int i = lane; i < S; i += 32) dsv[i] = wv[i] * (dwv[i] - dot);
    }
    __syncthreads();
    if (tid < QD) {
      for (int i = 0; i < S; ++i) {
        const int64_t row = seq * S + i;
        const float tv = t[row * QD + tid];
        const float ds = dsv[i];
        const float du = ds * qv * (1.f - tv * tv);
        d_u[row * QD + tid] = du;
        dba_acc += du;
        dqa_acc = fmaf(ds, tv, dqa_acc);
      }
    }
    for (int f = tid; f < S * DV4; f += 256) {
      const int i = f / DV4, l = f % DV4;
      const float wi = wv[i];
      float4 g = *reinterpret_cast<const float4*>(go + 4 * l);
      *reinterpret_cast<float4*>(d_c + (seq * S + i) * D + 4 * l) = make_float4(wi * g.x, wi * g.y, wi * g.z, wi * g.w);
    }
    __syncthreads();
  }
  if (tid < QD) {
    partial_dqa[(int64_t)blockIdx.x * QD + tid] = dqa_acc;
    partial_dqa[(int64_t)(gridDim.x + blockIdx.x) * QD + tid] = dba_acc;
  }
}

// ----------------------------------------------------------------------------------------
// deterministic column sums: partial[b, col] over a contiguous row range, then a fixed-order
// final accumulate  out[col] += sum_b partial[b, col].
// ----------------------------------------------------------------------------------------
static __global__ void __launch_bounds__(256)
colsum_partial_kernel(const float* __restrict__ x, int64_t n_rows, int N, float* __restrict__ partial) {
  const int64_t per = (n_rows + gridDim.x - 1) / gridDim.x;
  const int64_t r0 = (int64_t)blockIdx.x * per;
  const int64_t r1 = (r0 + per < n_rows) ? r0 + per : n_rows;
  // four columns per thread (N % 4 == 0: 900 / 200 / 300), eight rows in flight: the walk is a pure stream and was
  // latency-bound with one 4-byte load per thread and iteration (2 TB/s of the 507 MB dQKV matrix)
  for (int c4 = threadIdx.x; 4 * c4 < N; c4 += blockDim.x) {
    const float4* xp = reinterpret_cast<const float4*>(x) + c4;
    const int64_t ld4 = N / 4;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int64_t r = r0;
    for (; r + 8 <= r1; r += 8) {
      float4 v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = __ldg(xp + (r + j) * ld4);
#pragma unroll
      for (int j = 0; j < 8; ++j) { acc.x += v[j].x; acc.y += v[j].y; acc.z += v[j].z; acc.w += v[j].w; }
    }
    for (; r < r1; ++r) {
      const float4 v = __ldg(xp + r * ld4);
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    reinterpret_cast<float4*>(partial + (int64_t)blockIdx.x * N)[c4] = acc;
  }
}

// out[col] += sum_b partial[b * stride + col], col < n_cols.  One block = 32 columns x 8 row groups (the serial walk of
// one thread per column over ~300 partial rows took 20 us per launch, six launches per training step); launch with
// (n_cols + 31) / 32 blocks of 256 threads.  Summation order is fixed (deterministic).
static __global__ void __launch_bounds__(256)
partial_reduce_accum_strided_kernel(const float* __restrict__ partial, int n_blocks, int stride, int n_cols,
                                    float* __restrict__ out) {
  __shared__ float red[8][33];
  const int cx = threadIdx.x & 31, g = threadIdx.x >> 5;
  const int col = blockIdx.x * 32 + cx;
  float acc = 0.f;
  if (col < n_cols)
    for (int b = g; b < n_blocks; b += 8) acc += partial[(int64_t)b * stride + col];
  red[g][cx] = acc;
  __syncthreads();
  if (g == 0 && col < n_cols) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += red[k][cx];
    out[col] += t;
  }
}
static inline void launch_partial_reduce_accum(const float* partial, int n_blocks, int stride, int n_cols, float* out,
                                               cudaStream_t st) {
  partial_reduce_accum_strided_kernel<<<(n_cols + 31) / 32, 256, 0, st>>>(partial, n_blocks, stride, n_cols, out);
}

// ----------------------------------------------------------------------------------------
// LayerNorm(300) over the context rows (config-5 variant, builder-defined: DESIGN.md section 1; torch semantics:
// biased variance, eps inside the square root).  One warp per row, the row in registers (three float4 per lane).
// ----------------------------------------------------------------------------------------
__device__ __forceinline__ float ln_warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

static __global__ void __launch_bounds__(256)
layernorm_fwd_kernel(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
                     float* __restrict__ y, float* __restrict__ stats, int64_t n_rows, float eps) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = warp0; r < n_rows; r += n_warps) {
    const float4* xr = reinterpret_cast<const float4*>(x + r * D);
    float4 v[3];
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const int i = lane + 32 * j;
      v[j] = (i < DV4) ? xr[i] : make_float4(0.f, 0.f, 0.f, 0.f);
      s += v[j].x + v[j].y + v[j].z + v[j].w;
    }
    const float mean = ln_warp_sum(s) * (1.f / D);
    float q = 0.f;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      if (lane + 32 * j < DV4) {
        const float a = v[j].x - mean, b = v[j].y - mean, c = v[j].z - mean, d = v[j].w - mean;
        q += a * a + b * b + c * c + d * d;
      }
    }
    const float rstd = rsqrtf(ln_warp_sum(q) * (1.f / D) + eps);
    float4* yr = reinterpret_cast<float4*>(y + r * D);
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const int i = lane + 32 * j;
      if (i < DV4) {
        const float4 g = __ldg(reinterpret_cast<const float4*>(gamma) + i);
        const float4 b = __ldg(reinterpret_cast<const float4*>(beta) + i);
        yr[i] = make_float4((v[j].x - mean) * rstd * g.x + b.x, (v[j].y - mean) * rstd * g.y + b.y,
                            (v[j].z - mean) * rstd * g.z + b.z, (v[j].w - mean) * rstd * g.w + b.w);
      }
    }
    if (stats && lane == 0) {
      stats[2 * r] = mean;
      stats[2 * r + 1] = rstd;
    }
  }
}

// dy (in) -> dx (in place); per-block partial sums of d_gamma (columns [0,300)) and d_beta ([300,600)) go to
// partial[blockIdx.x][600], reduced by partial_reduce_accum_kernel.  Block = 8 warps, each warp owns rows.
static __global__ void __launch_bounds__(256)
layernorm_bwd_kernel(float* __restrict__ dy_dx, const float* __restrict__ x, const float* __restrict__ stats,
                     const float* __restrict__ gamma, float* __restrict__ partial, int64_t n_rows) {
  __shared__ float red[8][2 * D];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t warp0 = (int64_t)blockIdx.x * 8 + warp;
  const int64_t n_warps = (int64_t)gridDim.x * 8;
  float4 dg[3], db[3];
#pragma unroll
  for (int j = 0; j < 3; ++j) dg[j] = db[j] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int64_t r = warp0; r < n_rows; r += n_warps) {
    const float mean = stats[2 * r], rstd = stats[2 * r + 1];
    const float4* xr = reinterpret_cast<const float4*>(x + r * D);
    float4* dr = reinterpret_cast<float4*>(dy_dx + r * D);
    float4 xh[3], g[3];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const int i = lane + 32 * j;
      xh[j] = g[j] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (i < DV4) {
        const float4 xv = xr[i], dyv = dr[i];
        const float4 gm = __ldg(reinterpret_cast<const float4*>(gamma) + i);
        xh[j] = make_float4((xv.x - mean) * rstd, (xv.y - mean) * rstd, (xv.z - mean) * rstd, (xv.w - mean) * rstd);
        g[j] = make_float4(dyv.x * gm.x, dyv.y * gm.y, dyv.z * gm.z, dyv.w * gm.w);
        dg[j].x += dyv.x * xh[j].x; dg[j].y += dyv.y * xh[j].y; dg[j].z += dyv.z * xh[j].z; dg[j].w += dyv.w * xh[j].w;
        db[j].x += dyv.x; db[j].y += dyv.y; db[j].z += dyv.z; db[j].w += dyv.w;
        s1 += g[j].x + g[j].y + g[j].z + g[j].w;
        s2 += g[j].x * xh[j].x + g[j].y * xh[j].y + g[j].z * xh[j].z + g[j].w * xh[j].w;
      }
    }
    const float m1 = ln_warp_sum(s1) * (1.f / D), m2 = ln_warp_sum(s2) * (1.f / D);
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const int i = lane + 32 * j;
      if (i < DV4)
        dr[i] = make_float4(rstd * (g[j].x - m1 - xh[j].x * m2), rstd * (g[j].y - m1 - xh[j].y * m2),
                            rstd * (g[j].z - m1 - xh[j].z * m2), rstd * (g[j].w - m1 - xh[j].w * m2));
    }
  }
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    const int i = lane + 32 * j;
    if (i < DV4) {
      reinterpret_cast<float4*>(red[warp])[i] = dg[j];
      reinterpret_cast<float4*>(red[warp] + D)[i] = db[j];
    }
  }
  __syncthreads();
  for (int col = threadIdx.x; col < 2 * D; col += 256) {
    float a = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) a += red[w][col];
    partial[(int64_t)blockIdx.x * (2 * D) + col] = a;
  }
}

}  // namespace nrms
