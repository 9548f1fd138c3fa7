// Attention of the standalone MultiHeadSelfAttention at any query / key count 1 <= Sq, Sk <= 64, self- or
// cross-attention (reference src/model/general/attention/multihead_self.py:15-23,46-76 with K and V given): forward and
// backward, in both modes.  Per head h:
//   e[i, j] = exp(q_i^h . k_j^h / sqrt 20) * keep[b, j]  (no max shift),  ctx_i^h = sum_j e[i, j] v_j^h / (sum_j e[i, j] + 1e-8)
// The lengths are run-time arguments, and q, k and v are read through their own row pointers and pitches, so one kernel
// reads both the [rows, 900] q|k|v rows of self-attention and a q [n*Sq, 300] buffer beside k|v rows of another input.
// Key mask: `lengths` is the reference's `length` argument.  With Sq == Sk a sequence keeps the keys j < length[b]; with
// Sq == 1 < Sk the reference's [B, H, 1, 1] mask broadcasts, so every key is kept iff length[b] >= 1 (key_limit).
//
// Tensor mode (namespace amha): mma.sync.m16n8k8 TF32 with fp32 accumulation, one warp per (sequence, head), the two
// passes of the 50-token kernels (attn_mma.cu, amma50) with run-time extents.  Tiles Q, K, V (and G = dO in the
// backward) of [R][28] floats, R = the row count rounded up to 16 (at most 64): queries take up to 4 m16 tiles, keys up
// to 8 n8 tiles; the head dimension pads to 3 k8 steps (columns 20..27 stay zero) and the padding rows stay zero.
// The accumulators are arrays over all 8 n8 tiles, indexed only inside fully unrolled loops: the tiles past the extent
// are skipped by warp-uniform predicates, so the arrays stay in registers (a loop with a run-time bound over them makes
// ptxas put them in local memory).  Padded key columns get an exponential of exactly 0 (their zero rows would give
// exp(0) = 1), as do masked keys, so masked and padded keys get exactly zero dK and dV rows.
//   forward, per 16-query tile:  S = Q K^T, attn, O = attn V
//   backward, pass 1, per 16-query tile: S, attn, dP = G V^T, dS, dQ = dS K; 1 / (sum + eps) and delta = sum_j attn dP of
//             every query row are kept in shared memory
//   backward, pass 2, per 16-key tile:   S^T = K Q^T, attn^T, dP^T = V G^T, dS^T, dK = dS^T Q (dS split hi + lo: the
//             K-bias gradient is a sum that cancels), dV = attn^T G
// FP32 mode (attn_cross_fwd/bwd_kernel): CUDA-core kernels in the style of attention_fwd/bwd_kernel<S, HC>
// (encoder_kernels.cuh) with run-time lengths: thread = (head, query), K and V in shared memory, the same arithmetic
// (reference-exact up to summation order).
// DROPOUT (the news encoder's dropout #2 at text lengths other than 20 and 50, reference
// src/model/NRMS/news_encoder.py:43-45; self-attention only, ctx pitch 300): the forward multiplies the context by the
// mask where it stores it, the backward multiplies d_ctx by the same mask where it loads it.  The mask of element
// (seq * sq + i) * 300 + col is dropout_mask4(.., DROPOUT_STREAM_CTX, p, 1 / (1 - p), seed, offset), the stream the
// compiled 20- and 50-token kernels draw: one Philox evaluation covers four aligned columns, and heads start at multiples
// of 20 columns, so a group never straddles two heads.  Without it the kernels are those of the standalone block.
#include "common.cuh"
#include "tc_api.cuh"

namespace nrms {
namespace amha {

constexpr int ST = 28;           // tile row pitch in floats (pitch mod 32 = 28: conflict-free fragment loads)
constexpr int NT = 8;            // n8 tiles over 64 keys (pass 1) or 64 queries (pass 2)
constexpr int ZS = 64;           // floats per per-row vector (1 / (sum + eps), delta) of the backward
constexpr float SQRT_DH = 4.47213595499957939f;
constexpr float SCALE_LOG2E = 1.4426950408889634f / SQRT_DH;     // exp(s / sqrt 20) = 2^(s * log2(e) / sqrt 20)
constexpr float INV_SQRT_DH = 1.f / SQRT_DH;
constexpr float ATTN_EPS = 1e-8f;
constexpr uint32_t DROPOUT_STREAM_CTX = 2;     // encoder_kernels.cuh

// dropout #2 of the call (read only by the DROPOUT instantiations)
struct Drop {
  float p, scale;
  uint64_t seed, offset;
};

typedef float Row[NT][4];        // accumulators of 16 rows x 64 columns
typedef float Out[3][4];         // accumulators of 16 rows x 24 columns (the head dimension)

__host__ __device__ constexpr int round16(int x) { return (x + 15) / 16 * 16; }

__device__ __forceinline__ float tf32_round(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}
__device__ __forceinline__ void mma_tf32(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                         uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t ld(const float* p) { return __float_as_uint(*p); }
__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  const uint32_t s = (uint32_t)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }

template <typename F>
__device__ __forceinline__ void zero(F& c) {
  float* f = &c[0][0];
#pragma unroll
  for (int i = 0; i < (int)(sizeof(F) / sizeof(float)); ++i) f[i] = 0.f;
}

// c[i][j] += sum_d A[m0 + i][d] B[j][d]     (16 rows of tile A from row m0; rows of tile B in the first nb n8 tiles)
__device__ __forceinline__ void gemm_nt(Row& c, const float* A, int m0, const float* B, int nb, int g, int t) {
  const int r0 = m0 + g, r1 = r0 + 8;
#pragma unroll
  for (int ks = 0; ks < 3; ++ks) {
    const uint32_t a0 = ld(A + r0 * ST + ks * 8 + t), a2 = ld(A + r0 * ST + ks * 8 + t + 4);
    const uint32_t a1 = ld(A + r1 * ST + ks * 8 + t), a3 = ld(A + r1 * ST + ks * 8 + t + 4);
#pragma unroll
    for (int nt = 0; nt < NT; ++nt)
      if (nt < nb) {
        const uint32_t b0 = ld(B + (nt * 8 + g) * ST + ks * 8 + t), b1 = ld(B + (nt * 8 + g) * ST + ks * 8 + t + 4);
        mma_tf32(c[nt], a0, a1, a2, a3, b0, b1);
      }
  }
}

// c[i][d] += sum_j P[i][j] B[j][d] over the first nb 8-column blocks of P (the accumulators used in place as the A
// operand, see amma::gemm_frag_n).  SPLIT: P is taken as tf32(P) + tf32(P - tf32(P)), two products per step
template <bool SPLIT>
__device__ __forceinline__ void gemm_frag_n(Out& c, const Row& p, const float* B, int nb, int g, int t) {
#pragma unroll
  for (int ks = 0; ks < NT; ++ks)
    if (ks < nb) {
      float hi[4], lo[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        hi[e] = tf32_round(p[ks][e]);
        lo[e] = SPLIT ? tf32_round(p[ks][e] - hi[e]) : 0.f;
      }
#pragma unroll
      for (int nt = 0; nt < 3; ++nt) {
        const uint32_t b0 = ld(B + (ks * 8 + 2 * t) * ST + nt * 8 + g), b1 = ld(B + (ks * 8 + 2 * t + 1) * ST + nt * 8 + g);
        mma_tf32(c[nt], __float_as_uint(hi[0]), __float_as_uint(hi[2]), __float_as_uint(hi[1]), __float_as_uint(hi[3]), b0, b1);
        if (SPLIT)
          mma_tf32(c[nt], __float_as_uint(lo[0]), __float_as_uint(lo[2]), __float_as_uint(lo[1]), __float_as_uint(lo[3]), b0, b1);
      }
    }
}

// raw scores -> attention weights in place (key columns >= jmax -> exactly 0, padding included);
// inv[half] = 1 / (row sum + 1e-8) of row g + 8 half
__device__ __forceinline__ void softmax_rows(Row& c, int t, float (&inv)[2], int jmax) {
#pragma unroll
  for (int half = 0; half < 2; ++half) {
    float sum = 0.f;
#pragma unroll
    for (int nt = 0; nt < NT; ++nt)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int col = nt * 8 + 2 * t + e;
        const float v = col < jmax ? ex2(c[nt][half * 2 + e] * SCALE_LOG2E) : 0.f;
        c[nt][half * 2 + e] = v;
        sum += v;
      }
    sum += __shfl_xor_sync(0xffffffffu, sum, 1);
    sum += __shfl_xor_sync(0xffffffffu, sum, 2);
    inv[half] = 1.f / (sum + ATTN_EPS);
#pragma unroll
    for (int nt = 0; nt < NT; ++nt)
#pragma unroll
      for (int e = 0; e < 2; ++e) c[nt][half * 2 + e] *= inv[half];
  }
}

// rows m0 .. m0 + 15 (those < n) of an Out fragment to global rows of pitch ld_ (two floats per store)
__device__ __forceinline__ void store_rows(float* dst, int64_t ld_, const Out& c, int m0, int n, int g, int t) {
#pragma unroll
  for (int nt = 0; nt < 3; ++nt)
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      const int row = m0 + g + 8 * half, col = nt * 8 + 2 * t;
      if (row < n && col < DH)
        *reinterpret_cast<float2*>(dst + row * ld_ + col) = make_float2(c[nt][half * 2], c[nt][half * 2 + 1]);
    }
}

// warp-private staging of one head: tile <- the 20 columns at `src` of n rows of pitch ld_, 16-byte async copies; call
// fetch_round after cp_async_wait_all to round the same pieces to TF32 in place (every lane converts exactly the
// pieces it copied itself, so no barrier sits between the copy and the conversion)
__device__ __forceinline__ void fetch_issue(float* tile, const float* __restrict__ src, int64_t ld_, int n, int lane) {
  for (int f = lane; f < n * (DH / 4); f += 32) {
    const int j = f / (DH / 4), d4 = f % (DH / 4);
    cp_async16(tile + j * ST + d4 * 4, src + (int64_t)j * ld_ + d4 * 4);
  }
}
__device__ __forceinline__ void fetch_round(float* tile, int n, int lane) {
  for (int f = lane; f < n * (DH / 4); f += 32) {
    const int j = f / (DH / 4), d4 = f % (DH / 4);
    float4* q = reinterpret_cast<float4*>(tile + j * ST + d4 * 4);
    const float4 x = *q;
    *q = make_float4(tf32_round(x.x), tf32_round(x.y), tf32_round(x.z), tf32_round(x.w));
  }
}
// fetch_round of the d_ctx tile with the dropout-2 mask applied before the rounding: row j of the tile is row row0 + j
// of the call, its columns start at column `col` of the 300
__device__ __forceinline__ void fetch_round_masked(float* tile, int n, int lane, int64_t row0, int col, const Drop& dr) {
  for (int f = lane; f < n * (DH / 4); f += 32) {
    const int j = f / (DH / 4), d4 = f % (DH / 4);
    float4* q = reinterpret_cast<float4*>(tile + j * ST + d4 * 4);
    const float4 x = *q;
    const float4 m = dropout_mask4((uint64_t)(row0 + j) * D + col + d4 * 4, DROPOUT_STREAM_CTX, dr.p, dr.scale, dr.seed,
                                   dr.offset);
    *q = make_float4(tf32_round(x.x * m.x), tf32_round(x.y * m.y), tf32_round(x.z * m.z), tf32_round(x.w * m.w));
  }
}

// keys of sequence `seq` that the mask keeps (see the file header)
__device__ __forceinline__ int key_limit(const int32_t* __restrict__ lengths, int64_t seq, int sq, int sk) {
  if (lengths == nullptr) return sk;
  const int l = lengths[seq];
  if (sq < sk) return l >= 1 ? sk : 0;
  return l < 0 ? 0 : (l < sk ? l : sk);
}

template <bool DROPOUT>
__global__ void __launch_bounds__(32)
mha_fwd_kernel(const float* __restrict__ q, int64_t ldq, const float* __restrict__ k, int64_t ldk,
               const float* __restrict__ v, int64_t ldv, float* __restrict__ ctx, int64_t n_seq, int sq, int sk,
               const int32_t* __restrict__ lengths, Drop dr) {
  extern __shared__ __align__(16) float smem[];
  const int lane = threadIdx.x, g = lane >> 2, t = lane & 3;
  const int rq = round16(sq), rk = round16(sk);
  for (int f = lane; f < (rq + 2 * rk) * ST; f += 32) smem[f] = 0.f;
  __syncwarp();
  float* Q = smem;
  float* K = Q + rq * ST;
  float* V = K + rk * ST;
  const int col = blockIdx.y * DH;            // the head's columns
  const int nkb = (sk + 7) / 8;               // n8 tiles over the keys
  for (int64_t seq = blockIdx.x; seq < n_seq; seq += gridDim.x) {
    __syncwarp();             // every lane is done with the previous sequence's tiles
    fetch_issue(Q, q + seq * sq * ldq + col, ldq, sq, lane);
    fetch_issue(K, k + seq * sk * ldk + col, ldk, sk, lane);
    fetch_issue(V, v + seq * sk * ldv + col, ldv, sk, lane);
    cp_async_wait_all();
    fetch_round(Q, sq, lane);
    fetch_round(K, sk, lane);
    fetch_round(V, sk, lane);
    __syncwarp();
    const int jmax = key_limit(lengths, seq, sq, sk);
#pragma unroll 1
    for (int m0 = 0; m0 < rq; m0 += 16) {
      Row a;
      zero(a);
      gemm_nt(a, Q, m0, K, nkb, g, t);
      float inv[2];
      softmax_rows(a, t, inv, jmax);
      Out o;
      zero(o);
      gemm_frag_n<false>(o, a, V, nkb, g, t);
      if (DROPOUT) {
        // a lane pair (t, t ^ 1) holds two columns of one aligned group of four in two rows: the even lane draws row
        // g's group, the odd lane row g + 8's, and each hands its partner the half it needs (as attn_mma.cu's amma50)
        const int odd = t & 1;
#pragma unroll
        for (int nt = 0; nt < 3; ++nt) {
          const float4 m = dropout_mask4((uint64_t)(seq * sq + m0 + g + 8 * odd) * D + col + nt * 8 + (t >> 1) * 4,
                                         DROPOUT_STREAM_CTX, dr.p, dr.scale, dr.seed, dr.offset);
          const float r0 = __shfl_xor_sync(0xffffffffu, odd ? m.x : m.z, 1);
          const float r1 = __shfl_xor_sync(0xffffffffu, odd ? m.y : m.w, 1);
          o[nt][0] *= odd ? r0 : m.x;
          o[nt][1] *= odd ? r1 : m.y;
          o[nt][2] *= odd ? m.z : r0;
          o[nt][3] *= odd ? m.w : r1;
        }
      }
      store_rows(ctx + seq * sq * D + col, D, o, m0, sq, g, t);
    }
  }
}

// dq / dk / dv are written with the pitches of q / k / v (the projection layout the weight contractions read)
template <bool DROPOUT>
__global__ void __launch_bounds__(32)
mha_bwd_kernel(const float* __restrict__ q, int64_t ldq, const float* __restrict__ k, int64_t ldk,
               const float* __restrict__ v, int64_t ldv, const float* __restrict__ d_ctx, float* __restrict__ dq,
               float* __restrict__ dk, float* __restrict__ dv, int64_t n_seq, int sq, int sk,
               const int32_t* __restrict__ lengths, Drop dr) {
  extern __shared__ __align__(16) float smem[];
  const int lane = threadIdx.x, g = lane >> 2, t = lane & 3;
  const int rq = round16(sq), rk = round16(sk);
  for (int f = lane; f < (2 * rq + 2 * rk) * ST + 2 * ZS; f += 32) smem[f] = 0.f;
  __syncwarp();
  float* Q = smem;
  float* G = Q + rq * ST;
  float* K = G + rq * ST;
  float* V = K + rk * ST;
  float* zinv = V + rk * ST;
  float* delta = zinv + ZS;
  const int col = blockIdx.y * DH;
  const int nkb = (sk + 7) / 8, nqb = (sq + 7) / 8;
  for (int64_t seq = blockIdx.x; seq < n_seq; seq += gridDim.x) {
    __syncwarp();             // every lane is done with the previous sequence's tiles and row vectors
    fetch_issue(Q, q + seq * sq * ldq + col, ldq, sq, lane);
    fetch_issue(G, d_ctx + seq * sq * D + col, D, sq, lane);
    fetch_issue(K, k + seq * sk * ldk + col, ldk, sk, lane);
    fetch_issue(V, v + seq * sk * ldv + col, ldv, sk, lane);
    cp_async_wait_all();
    fetch_round(Q, sq, lane);
    if (DROPOUT) fetch_round_masked(G, sq, lane, seq * sq, col, dr);
    else fetch_round(G, sq, lane);
    fetch_round(K, sk, lane);
    fetch_round(V, sk, lane);
    __syncwarp();
    const int jmax = key_limit(lengths, seq, sq, sk);
    // ---- pass 1: query tiles -> dQ, row vectors ----
#pragma unroll 1
    for (int m0 = 0; m0 < rq; m0 += 16) {
      Row a, dp;
      zero(a);
      gemm_nt(a, Q, m0, K, nkb, g, t);
      float inv[2];
      softmax_rows(a, t, inv, jmax);          // a = attn
      zero(dp);
      gemm_nt(dp, G, m0, V, nkb, g, t);       // dp = dO V^T
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        float dl = 0.f;
#pragma unroll
        for (int nt = 0; nt < NT; ++nt)
#pragma unroll
          for (int e = 0; e < 2; ++e) dl = fmaf(a[nt][half * 2 + e], dp[nt][half * 2 + e], dl);
        dl += __shfl_xor_sync(0xffffffffu, dl, 1);
        dl += __shfl_xor_sync(0xffffffffu, dl, 2);
#pragma unroll
        for (int nt = 0; nt < NT; ++nt)
#pragma unroll
          for (int e = 0; e < 2; ++e) dp[nt][half * 2 + e] = a[nt][half * 2 + e] * (dp[nt][half * 2 + e] - dl) * INV_SQRT_DH;
        const int row = m0 + g + 8 * half;
        if (t == 0 && row < sq) {
          zinv[row] = inv[half];
          delta[row] = dl;
        }
      }
      Out r;
      zero(r);
      gemm_frag_n<false>(r, dp, K, nkb, g, t);     // dQ = dS K
      store_rows(dq + seq * sq * ldq + col, ldq, r, m0, sq, g, t);
    }
    __syncwarp();             // the row vectors are visible to every lane
    // ---- pass 2: key tiles -> dK, dV ----
#pragma unroll 1
    for (int k0 = 0; k0 < rk; k0 += 16) {
      Row a, dp;
      zero(a);
      gemm_nt(a, K, k0, Q, nqb, g, t);        // S^T: rows = keys, columns = queries
      zero(dp);
      gemm_nt(dp, V, k0, G, nqb, g, t);       // dP^T = V dO^T
#pragma unroll
      for (int nt = 0; nt < NT; ++nt)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int qc = nt * 8 + 2 * t + e;
          const float z = qc < sq ? zinv[qc] : 0.f, dl = qc < sq ? delta[qc] : 0.f;
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            const bool keep = qc < sq && k0 + g + 8 * half < jmax;                        // query column, key row
            const float at = keep ? ex2(a[nt][half * 2 + e] * SCALE_LOG2E) * z : 0.f;
            a[nt][half * 2 + e] = at;                                                     // attn^T
            dp[nt][half * 2 + e] = at * (dp[nt][half * 2 + e] - dl) * INV_SQRT_DH;        // dS^T
          }
        }
      Out r;
      zero(r);
      gemm_frag_n<true>(r, dp, Q, nqb, g, t);      // dK = (dS_hi + dS_lo)^T Q
      store_rows(dk + seq * sk * ldk + col, ldk, r, k0, sk, g, t);
      zero(r);
      gemm_frag_n<false>(r, a, G, nqb, g, t);      // dV = attn^T dO
      store_rows(dv + seq * sk * ldv + col, ldv, r, k0, sk, g, t);
    }
  }
}

}  // namespace amha

// ---- FP32 mode --------------------------------------------------------------------------------------------------------
constexpr int MHA_MAXS = 64;
constexpr int MHA_HC_FWD = 5;    // heads per CTA: K and V of 5 heads at 64 keys = 51 KB of shared memory
constexpr int MHA_HC_BWD = 3;    // Q, dO, K, V and the two [3*Sq][Sk+1] score planes: 161 KB at 64 x 64

// CTA = (sequence, chunk of HC heads); thread = (head, query i)
template <int HC, bool DROPOUT>
__global__ void __launch_bounds__(HC * MHA_MAXS)
attn_cross_fwd_kernel(const float* __restrict__ q, int64_t ldq, const float* __restrict__ k, int64_t ldk,
                      const float* __restrict__ v, int64_t ldv, float* __restrict__ ctx, int64_t n_seq, int sq, int sk,
                      const int32_t* __restrict__ lengths, amha::Drop dr) {
  constexpr int W = HC * DH, W4 = W / 4;
  extern __shared__ __align__(16) float smem[];
  float* Ks = smem;            // [sk][W]
  float* Vs = smem + sk * W;   // [sk][W]
  const int tid = threadIdx.x;
  const int hl = tid / sq, i = tid % sq;
  const bool active = tid < sq * HC;
  const int cw = blockIdx.y * W;
  for (int64_t seq = blockIdx.x; seq < n_seq; seq += gridDim.x) {
    __syncthreads();
    for (int f = tid; f < sk * W4 * 2; f += blockDim.x) {
      const int which = f / (sk * W4), r = f % (sk * W4), j = r / W4, c4 = r % W4;
      const float* src = which ? v + (seq * sk + j) * ldv : k + (seq * sk + j) * ldk;
      *reinterpret_cast<float4*>((which ? Vs : Ks) + j * W + c4 * 4) = *reinterpret_cast<const float4*>(src + cw + c4 * 4);
    }
    __syncthreads();
    if (!active) continue;
    float qr[DH], acc[DH];
    {
      const float4* qp = reinterpret_cast<const float4*>(q + (seq * sq + i) * ldq + cw + hl * DH);
#pragma unroll
      for (int c = 0; c < DH / 4; ++c) {
        const float4 x = qp[c];
        qr[4 * c] = x.x; qr[4 * c + 1] = x.y; qr[4 * c + 2] = x.z; qr[4 * c + 3] = x.w;
      }
    }
#pragma unroll
    for (int d = 0; d < DH; ++d) acc[d] = 0.f;
    float Z = 0.f;
    const int jmax = amha::key_limit(lengths, seq, sq, sk);
#pragma unroll 4
    for (int j = 0; j < jmax; ++j) {
      const float4* kp = reinterpret_cast<const float4*>(Ks + j * W + hl * DH);
      float sp[DH / 4];
#pragma unroll
      for (int c = 0; c < DH / 4; ++c) {
        const float4 kk = kp[c];
        sp[c] = fmaf(qr[4 * c + 3], kk.w, fmaf(qr[4 * c + 2], kk.z, fmaf(qr[4 * c + 1], kk.y, qr[4 * c] * kk.x)));
      }
      const float s = ((sp[0] + sp[1]) + (sp[2] + sp[3])) + sp[4];
      const float e = expf(s / amha::SQRT_DH);
      Z += e;
      const float4* vp = reinterpret_cast<const float4*>(Vs + j * W + hl * DH);
#pragma unroll
      for (int c = 0; c < DH / 4; ++c) {
        const float4 vv = vp[c];
        acc[4 * c] = fmaf(e, vv.x, acc[4 * c]); acc[4 * c + 1] = fmaf(e, vv.y, acc[4 * c + 1]);
        acc[4 * c + 2] = fmaf(e, vv.z, acc[4 * c + 2]); acc[4 * c + 3] = fmaf(e, vv.w, acc[4 * c + 3]);
      }
    }
    const float inv = 1.f / (Z + amha::ATTN_EPS);
    float4* op = reinterpret_cast<float4*>(ctx + (seq * sq + i) * D + cw + hl * DH);
#pragma unroll
    for (int c = 0; c < DH / 4; ++c) {
      float4 o = make_float4(acc[4 * c] * inv, acc[4 * c + 1] * inv, acc[4 * c + 2] * inv, acc[4 * c + 3] * inv);
      if (DROPOUT) {
        const float4 m = dropout_mask4((uint64_t)(seq * sq + i) * D + cw + hl * DH + 4 * c, amha::DROPOUT_STREAM_CTX, dr.p,
                                       dr.scale, dr.seed, dr.offset);
        o.x *= m.x; o.y *= m.y; o.z *= m.z; o.w *= m.w;
      }
      op[c] = o;
    }
  }
}

// Phase 1: thread (h, query i) computes row i of the scores (e_ij, da_ij = g_i . v_j), its 1 / (Z + eps) and delta, then
// dQ_i, leaving attn_ij and ds_ij in shared memory (zero for masked keys).  Phase 2: thread (h, key j) reads column j
// and accumulates dK_j and dV_j.  Score planes have a pitch of sk + 1 words.
template <int HC, bool DROPOUT>
__global__ void __launch_bounds__(HC * MHA_MAXS)
attn_cross_bwd_kernel(const float* __restrict__ q, int64_t ldq, const float* __restrict__ k, int64_t ldk,
                      const float* __restrict__ v, int64_t ldv, const float* __restrict__ d_ctx, float* __restrict__ dq,
                      float* __restrict__ dk, float* __restrict__ dv, int64_t n_seq, int sq, int sk,
                      const int32_t* __restrict__ lengths, amha::Drop dr) {
  constexpr int W = HC * DH, W4 = W / 4;
  const int sp1 = sk + 1;
  extern __shared__ __align__(16) float smem[];
  float* Qs = smem;               // [sq][W]
  float* Gs = Qs + sq * W;        // [sq][W]
  float* Ks = Gs + sq * W;        // [sk][W]
  float* Vs = Ks + sk * W;        // [sk][W]
  float* Ps = Vs + sk * W;        // [HC*sq][sk+1] e, then attn
  float* Ds = Ps + HC * sq * sp1; // [HC*sq][sk+1] da, then ds
  const int tid = threadIdx.x;
  const int cw = blockIdx.y * W;
  for (int64_t seq = blockIdx.x; seq < n_seq; seq += gridDim.x) {
    __syncthreads();
    for (int f = tid; f < (sq + sk) * W4 * 2; f += blockDim.x) {
      const int nq = sq * W4;
      const float* src;
      float* dst;
      if (f < 2 * nq) {
        const int which = f / nq, r = f % nq, j = r / W4, c4 = r % W4;
        src = (which ? d_ctx + (seq * sq + j) * D : q + (seq * sq + j) * ldq) + cw + c4 * 4;
        dst = (which ? Gs : Qs) + j * W + c4 * 4;
        if (DROPOUT && which) {      // d_ctx through the dropout-2 mask
          float4 x = *reinterpret_cast<const float4*>(src);
          const float4 m = dropout_mask4((uint64_t)(seq * sq + j) * D + cw + c4 * 4, amha::DROPOUT_STREAM_CTX, dr.p,
                                         dr.scale, dr.seed, dr.offset);
          x.x *= m.x; x.y *= m.y; x.z *= m.z; x.w *= m.w;
          *reinterpret_cast<float4*>(dst) = x;
          continue;
        }
      } else {
        const int f2 = f - 2 * nq, nk = sk * W4;
        const int which = f2 / nk, r = f2 % nk, j = r / W4, c4 = r % W4;
        src = (which ? v + (seq * sk + j) * ldv : k + (seq * sk + j) * ldk) + cw + c4 * 4;
        dst = (which ? Vs : Ks) + j * W + c4 * 4;
      }
      *reinterpret_cast<float4*>(dst) = *reinterpret_cast<const float4*>(src);
    }
    __syncthreads();
    const int jmax = amha::key_limit(lengths, seq, sq, sk);
    float a[DH], b[DH], r[DH];
    // ---- phase 1 ----
    if (tid < sq * HC) {
      const int hl = tid / sq, i = tid % sq;
      float* prow = Ps + (hl * sq + i) * sp1;
      float* drow = Ds + (hl * sq + i) * sp1;
#pragma unroll
      for (int d = 0; d < DH; ++d) { a[d] = Qs[i * W + hl * DH + d]; b[d] = Gs[i * W + hl * DH + d]; r[d] = 0.f; }
      float Z = 0.f, num = 0.f;
#pragma unroll 4
      for (int j = 0; j < jmax; ++j) {
        const float4* kp = reinterpret_cast<const float4*>(Ks + j * W + hl * DH);
        const float4* vp = reinterpret_cast<const float4*>(Vs + j * W + hl * DH);
        float sp[DH / 4], dp[DH / 4];      // five independent 4-term chains per dot product, in the forward's order
#pragma unroll
        for (int c = 0; c < DH / 4; ++c) {
          const float4 kk = kp[c], vv = vp[c];
          sp[c] = fmaf(a[4 * c + 3], kk.w, fmaf(a[4 * c + 2], kk.z, fmaf(a[4 * c + 1], kk.y, a[4 * c] * kk.x)));
          dp[c] = fmaf(b[4 * c + 3], vv.w, fmaf(b[4 * c + 2], vv.z, fmaf(b[4 * c + 1], vv.y, b[4 * c] * vv.x)));
        }
        const float s = ((sp[0] + sp[1]) + (sp[2] + sp[3])) + sp[4];
        const float da = ((dp[0] + dp[1]) + (dp[2] + dp[3])) + dp[4];
        const float e = expf(s / amha::SQRT_DH);      // same expression as the forward kernel
        Z += e;
        num = fmaf(e, da, num);
        prow[j] = e;
        drow[j] = da;
      }
      const float zinv = 1.f / (Z + amha::ATTN_EPS);
      const float delta = num * zinv;
#pragma unroll 4
      for (int j = 0; j < jmax; ++j) {
        const float4* kp = reinterpret_cast<const float4*>(Ks + j * W + hl * DH);
        const float at = prow[j] * zinv;
        const float ds = at * (drow[j] - delta) * amha::INV_SQRT_DH;
        prow[j] = at;
        drow[j] = ds;
#pragma unroll
        for (int c = 0; c < DH / 4; ++c) {
          const float4 kk = kp[c];
          r[4 * c] = fmaf(ds, kk.x, r[4 * c]); r[4 * c + 1] = fmaf(ds, kk.y, r[4 * c + 1]);
          r[4 * c + 2] = fmaf(ds, kk.z, r[4 * c + 2]); r[4 * c + 3] = fmaf(ds, kk.w, r[4 * c + 3]);
        }
      }
      for (int j = jmax; j < sk; ++j) prow[j] = drow[j] = 0.f;
      float4* op = reinterpret_cast<float4*>(dq + (seq * sq + i) * ldq + cw + hl * DH);
#pragma unroll
      for (int c = 0; c < DH / 4; ++c) op[c] = make_float4(r[4 * c], r[4 * c + 1], r[4 * c + 2], r[4 * c + 3]);
    }
    __syncthreads();
    // ---- phase 2 ----
    if (tid < sk * HC) {
      const int hl = tid / sk, j = tid % sk;
      const float* pcol = Ps + hl * sq * sp1 + j;
      const float* dcol = Ds + hl * sq * sp1 + j;
#pragma unroll
      for (int d = 0; d < DH; ++d) { a[d] = 0.f; b[d] = 0.f; }     // a = dK_j, b = dV_j
#pragma unroll 4
      for (int ii = 0; ii < sq; ++ii) {
        const float4* qp = reinterpret_cast<const float4*>(Qs + ii * W + hl * DH);
        const float4* gp = reinterpret_cast<const float4*>(Gs + ii * W + hl * DH);
        const float at = pcol[ii * sp1];
        const float ds = dcol[ii * sp1];
#pragma unroll
        for (int c = 0; c < DH / 4; ++c) {
          const float4 qv = qp[c], gv = gp[c];
          a[4 * c] = fmaf(ds, qv.x, a[4 * c]); a[4 * c + 1] = fmaf(ds, qv.y, a[4 * c + 1]);
          a[4 * c + 2] = fmaf(ds, qv.z, a[4 * c + 2]); a[4 * c + 3] = fmaf(ds, qv.w, a[4 * c + 3]);
          b[4 * c] = fmaf(at, gv.x, b[4 * c]); b[4 * c + 1] = fmaf(at, gv.y, b[4 * c + 1]);
          b[4 * c + 2] = fmaf(at, gv.z, b[4 * c + 2]); b[4 * c + 3] = fmaf(at, gv.w, b[4 * c + 3]);
        }
      }
      float4* ok = reinterpret_cast<float4*>(dk + (seq * sk + j) * ldk + cw + hl * DH);
      float4* ov = reinterpret_cast<float4*>(dv + (seq * sk + j) * ldv + cw + hl * DH);
#pragma unroll
      for (int c = 0; c < DH / 4; ++c) {
        ok[c] = make_float4(a[4 * c], a[4 * c + 1], a[4 * c + 2], a[4 * c + 3]);
        ov[c] = make_float4(b[4 * c], b[4 * c + 1], b[4 * c + 2], b[4 * c + 3]);
      }
    }
  }
}

static unsigned mha_grid_x(int64_t n_seq, int per_sm) {
  return (unsigned)(n_seq < (int64_t)num_sms() * per_sm ? n_seq : (int64_t)num_sms() * per_sm);
}

int mha_attn_fwd(const MhaOperands& in, float* ctx, int64_t n_seq, int sq, int sk, const int32_t* lengths, int mode,
                 cudaStream_t st, float p, uint64_t seed, uint64_t offset) {
  if (n_seq == 0) return NRMS_OK;
  const amha::Drop dr{p, p > 0.f ? 1.f / (1.f - p) : 1.f, seed, offset};
  if (mode == NRMS_MODE_TF32) {
    const size_t smem = (size_t)(amha::round16(sq) + 2 * amha::round16(sk)) * amha::ST * sizeof(float);
    const dim3 grid(mha_grid_x(n_seq, 16), H);
    if (p > 0.f)
      amha::mha_fwd_kernel<true><<<grid, 32, smem, st>>>(in.q, in.ldq, in.k, in.ldk, in.v, in.ldv, ctx, n_seq, sq, sk,
                                                         lengths, dr);
    else
      amha::mha_fwd_kernel<false><<<grid, 32, smem, st>>>(in.q, in.ldq, in.k, in.ldk, in.v, in.ldv, ctx, n_seq, sq, sk,
                                                          lengths, dr);
    NRMS_LAUNCH_CHECK("mha_fwd");
    return NRMS_OK;
  }
  constexpr int HC = MHA_HC_FWD;
  const size_t smem = (size_t)2 * sk * HC * DH * sizeof(float);
  const dim3 grid(mha_grid_x(n_seq, 8), H / HC);
  const int threads = (sq * HC + 31) / 32 * 32;
  const int max_smem = 2 * MHA_MAXS * HC * DH * (int)sizeof(float);
  if (p > 0.f) {
    static bool configured[64] = {false};
    if (cudaError_t e = set_max_dynamic_smem(attn_cross_fwd_kernel<HC, true>, max_smem, configured))
      return cuda_fail(e, "attn_cross_fwd attr");
    attn_cross_fwd_kernel<HC, true><<<grid, threads, smem, st>>>(in.q, in.ldq, in.k, in.ldk, in.v, in.ldv, ctx, n_seq, sq,
                                                                 sk, lengths, dr);
  } else {
    static bool configured[64] = {false};
    if (cudaError_t e = set_max_dynamic_smem(attn_cross_fwd_kernel<HC, false>, max_smem, configured))
      return cuda_fail(e, "attn_cross_fwd attr");
    attn_cross_fwd_kernel<HC, false><<<grid, threads, smem, st>>>(in.q, in.ldq, in.k, in.ldk, in.v, in.ldv, ctx, n_seq, sq,
                                                                  sk, lengths, dr);
  }
  NRMS_LAUNCH_CHECK("attn_cross_fwd");
  return NRMS_OK;
}

int mha_attn_bwd(const MhaOperands& in, const float* d_ctx, float* dq, float* dk, float* dv, int64_t n_seq, int sq, int sk,
                 const int32_t* lengths, int mode, cudaStream_t st, float p, uint64_t seed, uint64_t offset) {
  if (n_seq == 0) return NRMS_OK;
  const amha::Drop dr{p, p > 0.f ? 1.f / (1.f - p) : 1.f, seed, offset};
  if (mode == NRMS_MODE_TF32) {
    const size_t smem = ((size_t)(2 * amha::round16(sq) + 2 * amha::round16(sk)) * amha::ST + 2 * amha::ZS) * sizeof(float);
    const dim3 grid(mha_grid_x(n_seq, 16), H);
    if (p > 0.f)
      amha::mha_bwd_kernel<true><<<grid, 32, smem, st>>>(in.q, in.ldq, in.k, in.ldk, in.v, in.ldv, d_ctx, dq, dk, dv, n_seq,
                                                         sq, sk, lengths, dr);
    else
      amha::mha_bwd_kernel<false><<<grid, 32, smem, st>>>(in.q, in.ldq, in.k, in.ldk, in.v, in.ldv, d_ctx, dq, dk, dv,
                                                          n_seq, sq, sk, lengths, dr);
    NRMS_LAUNCH_CHECK("mha_bwd");
    return NRMS_OK;
  }
  constexpr int HC = MHA_HC_BWD;
  auto bytes = [](int a, int b) { return (size_t)(2 * (a + b) * HC * DH + 2 * HC * a * (b + 1)) * sizeof(float); };
  const int rows = sq > sk ? sq : sk;
  const dim3 grid(mha_grid_x(n_seq, 4), H / HC);
  const int threads = (rows * HC + 31) / 32 * 32;
  if (p > 0.f) {
    static bool configured[64] = {false};
    if (cudaError_t e = set_max_dynamic_smem(attn_cross_bwd_kernel<HC, true>, (int)bytes(MHA_MAXS, MHA_MAXS), configured))
      return cuda_fail(e, "attn_cross_bwd attr");
    attn_cross_bwd_kernel<HC, true><<<grid, threads, bytes(sq, sk), st>>>(in.q, in.ldq, in.k, in.ldk, in.v, in.ldv, d_ctx,
                                                                          dq, dk, dv, n_seq, sq, sk, lengths, dr);
  } else {
    static bool configured[64] = {false};
    if (cudaError_t e = set_max_dynamic_smem(attn_cross_bwd_kernel<HC, false>, (int)bytes(MHA_MAXS, MHA_MAXS), configured))
      return cuda_fail(e, "attn_cross_bwd attr");
    attn_cross_bwd_kernel<HC, false><<<grid, threads, bytes(sq, sk), st>>>(in.q, in.ldq, in.k, in.ldk, in.v, in.ldv, d_ctx,
                                                                           dq, dk, dv, n_seq, sq, sk, lengths, dr);
  }
  NRMS_LAUNCH_CHECK("attn_cross_bwd");
  return NRMS_OK;
}

}  // namespace nrms
