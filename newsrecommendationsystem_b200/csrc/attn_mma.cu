// Tensor-mode TRAINING attention over 20-token titles on the tensor cores (mma.sync.m16n8k8 TF32, fp32 accumulate):
// forward and backward of ScaledDotProductAttention inside MultiHeadSelfAttention
// (reference src/model/general/attention/multihead_self.py:15-23 and its autograd), one warp per (title, head).
//
// Why mma.sync and not tcgen05 here: per (title, head) the five contractions of the backward are 20x20x20 each --
// 1/13 of one 128x128x16 tcgen05 tile -- and their operands chain through per-row softmax arithmetic in registers.  The
// CUDA-core kernels this replaces (encoder_kernels.cuh, still the FP32-mode path) spent one shared-memory load per four
// FMAs and ran at 0.8 ms per 7,040 titles in the backward (ncu launch list, profiles/), 20 % of the training step.
//
// Layout.  CTA = (title, chunk of 5 heads), one warp per head.  Per head four shared-memory tiles Q, K, V, G(=dO) of
// [24 rows][28 floats]: rows 20..23 and columns 20..27 stay zero (they pad the 20-long dimensions to MMA shapes: rows to
// 2 x m16 / 3 x n8, the head dimension to 3 x k8), values are rounded to TF32 (cvt.rna) when staged.  The row pitch of 28
// words makes every fragment load conflict-free (pitch mod 32 = 28: the 8 row groups of a fragment land on distinct
// 4-bank groups).
//
//   S = Q K^T            A = Q rows, B = K rows                      ("NT": both operands read along the head dimension)
//   P = exp(S / sqrt 20), attn = P / (sum_j P + 1e-8)                 in the accumulator fragments, quad shuffles
//   O = attn V           A = the attn accumulator fragments, used in place: an accumulator fragment holds columns
//                        (2t, 2t+1) of an 8-column block where an A fragment wants (t, t+4); the contraction index is a
//                        dummy, so V's rows are simply read in the matching order (8b+2t, 8b+2t+1) -- no shuffles
//   backward: dP = G V^T (NT), dS = attn (dP - sum_j attn dP) / sqrt 20, dQ = dS K (fragments in place, like O),
//             dK = dS^T Q and dV = attn^T G read dS / attn back TRANSPOSED from shared memory: they are parked in the V
//             and K tiles, which are dead by then (their padding stays zero: only the 20x20 block is written).
// Global loads: warp-private 16-byte async copies, no block-wide barrier in the title loop (see warp_fetch).
//
// Key mask (the backward's MASKED instantiation, for the standalone block's `length`, multihead_self.py:60-68): the
// exponentials of key columns >= length are 0 where they are formed, so the row sums, attn, dS and delta see nothing
// of them, and the dK / dV rows of masked keys come out exactly zero with no special case (dS hi + lo included: both
// halves are 0).  Query rows past the length are computed like the others.
#include "common.cuh"
#include "tc_api.cuh"

namespace nrms {
namespace amma {

constexpr int S = 20;            // tokens per title
constexpr int RT = 24;           // tile rows (3 x 8)
constexpr int ST = 28;           // tile row pitch in floats
constexpr int TILE = RT * ST;    // floats per tile
constexpr int HC = 5;            // heads per CTA (one warp each)
constexpr int THREADS = HC * 32;
constexpr float SQRT_DH = 4.47213595499957939f;
constexpr float ATTN_EPS = 1e-8f;

// keys of sequence `seq` that the `length` mask keeps: min(max(length, 0), s) (encoder_kernels.cuh, attention_fwd_kernel)
__device__ __forceinline__ int key_limit(const int32_t* __restrict__ lengths, int64_t seq, int s) {
  const int l = lengths[seq];
  return l < 0 ? 0 : (l < s ? l : s);
}
constexpr uint32_t DROPOUT_STREAM_CTX = 2;     // encoder_kernels.cuh
constexpr int NBUF = 1;          // one set of tiles per warp (a second set, filled under the compute, halved the resident warps: slower)

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
// operand load.  The tiles arrive raw (cp.async); their warp rounds them to TF32 in place once (warp_fetch: cvt.rna; a
// bare fp32 pattern would be truncated by the tensor core) -- one conversion per element instead of one per fragment load
__device__ __forceinline__ uint32_t ld(const float* p) { return __float_as_uint(*p); }
__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  const uint32_t s = (uint32_t)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }

#ifdef NRMS_AMMA_TRACE
#define AT(k) do { if (threadIdx.x == 0 && blockIdx.x == 0 && blockIdx.y == 0) tr[k] = clock64(); } while (0)
#else
#define AT(k)
#endif

typedef float Frag[2][3][4];     // [m tile][n tile][accumulator register]

__device__ __forceinline__ void zero(Frag& c) {
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 3; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) c[mt][nt][e] = 0.f;
}

// c[i][j] += sum_d A[i][d] B[j][d]        (A, B: tiles)
__device__ __forceinline__ void gemm_nt(Frag& c, const float* A, const float* B, int g, int t) {
#pragma unroll
  for (int ks = 0; ks < 3; ++ks) {
    uint32_t a[2][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
      const int r0 = mt * 16 + g, r1 = r0 + 8;
      a[mt][0] = ld(A + r0 * ST + ks * 8 + t);
      a[mt][2] = ld(A + r0 * ST + ks * 8 + t + 4);
      a[mt][1] = r1 < RT ? ld(A + r1 * ST + ks * 8 + t) : 0u;
      a[mt][3] = r1 < RT ? ld(A + r1 * ST + ks * 8 + t + 4) : 0u;
    }
#pragma unroll
    for (int nt = 0; nt < 3; ++nt) {
      const uint32_t b0 = ld(B + (nt * 8 + g) * ST + ks * 8 + t), b1 = ld(B + (nt * 8 + g) * ST + ks * 8 + t + 4);
#pragma unroll
      for (int mt = 0; mt < 2; ++mt) mma_tf32(c[mt][nt], a[mt][0], a[mt][1], a[mt][2], a[mt][3], b0, b1);
    }
  }
}

// c[i][d] += sum_j P[i][j] B[j][d]        (P: accumulator fragments used in place as the A operand, B: tile)
__device__ __forceinline__ void gemm_frag_n(Frag& c, const Frag& p, const float* B, int g, int t) {
#pragma unroll
  for (int ks = 0; ks < 3; ++ks) {
    uint32_t a[2][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
      a[mt][0] = __float_as_uint(tf32_round(p[mt][ks][0]));   // (row g,   contraction slot t)     <- column 8ks + 2t
      a[mt][2] = __float_as_uint(tf32_round(p[mt][ks][1]));   // (row g,   contraction slot t + 4) <- column 8ks + 2t + 1
      a[mt][1] = __float_as_uint(tf32_round(p[mt][ks][2]));   // (row g+8, slot t)
      a[mt][3] = __float_as_uint(tf32_round(p[mt][ks][3]));   // (row g+8, slot t + 4)
    }
#pragma unroll
    for (int nt = 0; nt < 3; ++nt) {
      const uint32_t b0 = ld(B + (ks * 8 + 2 * t) * ST + nt * 8 + g), b1 = ld(B + (ks * 8 + 2 * t + 1) * ST + nt * 8 + g);
#pragma unroll
      for (int mt = 0; mt < 2; ++mt) mma_tf32(c[mt][nt], a[mt][0], a[mt][1], a[mt][2], a[mt][3], b0, b1);
    }
  }
}

// c[j][d] += sum_i T[i][j] B[i][d]        (T, B: tiles; T is read transposed)
__device__ __forceinline__ void gemm_tn(Frag& c, const float* T, const float* B, int g, int t) {
#pragma unroll
  for (int ks = 0; ks < 3; ++ks) {
    const int i0 = ks * 8 + t, i1 = i0 + 4;
    uint32_t a[2][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
      const int j0 = mt * 16 + g, j1 = j0 + 8;
      a[mt][0] = ld(T + i0 * ST + j0);
      a[mt][2] = ld(T + i1 * ST + j0);
      a[mt][1] = j1 < RT ? ld(T + i0 * ST + j1) : 0u;
      a[mt][3] = j1 < RT ? ld(T + i1 * ST + j1) : 0u;
    }
#pragma unroll
    for (int nt = 0; nt < 3; ++nt) {
      const uint32_t b0 = ld(B + i0 * ST + nt * 8 + g), b1 = ld(B + i1 * ST + nt * 8 + g);
#pragma unroll
      for (int mt = 0; mt < 2; ++mt) mma_tf32(c[mt][nt], a[mt][0], a[mt][1], a[mt][2], a[mt][3], b0, b1);
    }
  }
}

// raw scores -> attention weights in place: exp(s / sqrt 20) for key columns < jmax (20, or the clamped length of the
// masked backward), 0 for the others, divided by (row sum + 1e-8)  (multihead_self.py:16-20: no max subtraction)
__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void softmax_rows(Frag& c, int t, int jmax = S) {
  constexpr float SCALE_LOG2E = 1.4426950408889634f / SQRT_DH;     // exp(s / sqrt 20) = 2^(s * log2(e) / sqrt 20)
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      float sum = 0.f;
#pragma unroll
      for (int nt = 0; nt < 3; ++nt)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int col = nt * 8 + 2 * t + e;
          const float v = col < jmax ? ex2(c[mt][nt][half * 2 + e] * SCALE_LOG2E) : 0.f;
          c[mt][nt][half * 2 + e] = v;
          sum += v;
        }
      sum += __shfl_xor_sync(0xffffffffu, sum, 1);
      sum += __shfl_xor_sync(0xffffffffu, sum, 2);
      const float inv = 1.f / (sum + ATTN_EPS);
#pragma unroll
      for (int nt = 0; nt < 3; ++nt)
#pragma unroll
        for (int e = 0; e < 2; ++e) c[mt][nt][half * 2 + e] *= inv;
    }
}

// store the 20 x 20 block of a fragment into a tile as [row][col] (TF32-rounded); padding rows / columns are not touched
__device__ __forceinline__ void park(float* T, const Frag& c, int g, int t) {
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 3; ++nt)
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        const int row = mt * 16 + g + 8 * half, col = nt * 8 + 2 * t;
        if (row < S && col < S)
          *reinterpret_cast<float2*>(T + row * ST + col) =
              make_float2(tf32_round(c[mt][nt][half * 2]), tf32_round(c[mt][nt][half * 2 + 1]));
      }
}

// write the 20 x 20 block of a fragment to global rows (pitch ld floats), two floats per store
__device__ __forceinline__ void store_rows(float* dst, int64_t ld_, const Frag& c, int g, int t) {
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 3; ++nt)
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        const int row = mt * 16 + g + 8 * half, col = nt * 8 + 2 * t;
        if (row < S && col < S)
          *reinterpret_cast<float2*>(dst + row * ld_ + col) = make_float2(c[mt][nt][half * 2], c[mt][nt][half * 2 + 1]);
      }
}

// the same 20 x 20 block written TRANSPOSED: dstT[col * ldt + row].  The weight-gradient contraction dW = dQKV^T X reads
// dQKV^T as a K-major operand (tc_gemm.cu); writing it here replaces a 507 MB read + 507 MB write transposition pass per
// step.  The fragment is turned through a dead tile (scratch[col][row], 20 x 20 block only: the padding stays zero) and
// leaves as 16-byte stores: a column of the block is 20 consecutive floats = 80 contiguous, 16-byte aligned bytes of a
// row of dstT.  (Storing the fragments transposed directly -- 72 scalar stores per lane and matrix -- took the kernel
// from 383 to 804 us and 215 registers.)
__device__ __forceinline__ void store_rows_t(float* dstT, int64_t ldt, float* scratch, const Frag& c, int lane, int g, int t) {
  __syncwarp();
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 3; ++nt)
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        const int row = mt * 16 + g + 8 * half, col = nt * 8 + 2 * t;
        if (row < S && col < S) {
          scratch[col * ST + row] = c[mt][nt][half * 2];
          scratch[(col + 1) * ST + row] = c[mt][nt][half * 2 + 1];
        }
      }
  __syncwarp();
  for (int f = lane; f < S * (S / 4); f += 32) {
    const int col = f / (S / 4), r4 = f % (S / 4);
    *reinterpret_cast<float4*>(dstT + (int64_t)col * ldt + 4 * r4) = *reinterpret_cast<const float4*>(scratch + col * ST + 4 * r4);
  }
  __syncwarp();
}

// Warp-private staging: each warp copies the 20 x 20 blocks of its own head's NTILES tiles (tile k <- columns
// [k*300 + head*20, +20) of the title's 20 qkv rows for k < 3, of its d_ctx rows for k == 3) with 16-byte async copies,
// waits for them, and rounds them to TF32 in place (cvt.rna; a bare fp32 pattern would be truncated by the tensor core;
// the d_ctx tile also takes the dropout-2 mask of the forward's Philox stream here).  Every lane converts exactly the 16-byte
// pieces it copied itself, so there is no barrier between the copy and the conversion, and no block-wide barrier at all:
// the warps of a CTA drift apart and hide each other's copy latency.  (The first version staged cooperatively with two
// __syncthreads per title: clock64 stamps showed 4.2k cycles at the barrier, 3k waiting for the copies and 4.5k in a
// rolled conversion loop, against 5.7k of contractions.)
template <int NTILES>
__device__ __forceinline__ void warp_fetch(float* tiles, const float* __restrict__ qkv_head, const float* __restrict__ g_head,
                                           int lane, int64_t row0, int col0, float p, float scale, uint64_t seed,
                                           uint64_t offset) {
  constexpr int PT = 4;                       // 100 sixteen-byte pieces per tile over 32 lanes
  int j[PT], d4[PT];
#pragma unroll
  for (int k = 0; k < PT; ++k) {
    const int f = lane + 32 * k;
    j[k] = f / (DH / 4);
    d4[k] = f % (DH / 4);
  }
#pragma unroll
  for (int w = 0; w < NTILES; ++w)
#pragma unroll
    for (int k = 0; k < PT; ++k)
      if (lane + 32 * k < S * (DH / 4)) {
        const float* src = (w < 3) ? qkv_head + (int64_t)j[k] * D3 + w * D + d4[k] * 4 : g_head + (int64_t)j[k] * D + d4[k] * 4;
        cp_async16(tiles + w * TILE + j[k] * ST + d4[k] * 4, src);
      }
  cp_async_wait_all();
#pragma unroll
  for (int w = 0; w < NTILES; ++w) {
    float4 x[PT];
#pragma unroll
    for (int k = 0; k < PT; ++k)
      if (lane + 32 * k < S * (DH / 4)) x[k] = *reinterpret_cast<const float4*>(tiles + w * TILE + j[k] * ST + d4[k] * 4);
    if (w == 3 && p > 0.f) {
#pragma unroll
      for (int k = 0; k < PT; ++k)
        if (lane + 32 * k < S * (DH / 4)) {
          const float4 m = dropout_mask4((uint64_t)(row0 + j[k]) * D + col0 + d4[k] * 4, DROPOUT_STREAM_CTX, p, scale, seed, offset);
          x[k].x *= m.x; x[k].y *= m.y; x[k].z *= m.z; x[k].w *= m.w;
        }
    }
#pragma unroll
    for (int k = 0; k < PT; ++k)
      if (lane + 32 * k < S * (DH / 4))
        *reinterpret_cast<float4*>(tiles + w * TILE + j[k] * ST + d4[k] * 4) =
            make_float4(tf32_round(x[k].x), tf32_round(x[k].y), tf32_round(x[k].z), tf32_round(x[k].w));
  }
  __syncwarp();
}

__global__ void __launch_bounds__(THREADS)
attn_fwd_kernel(const float* __restrict__ qkv, float* __restrict__ ctx, int64_t n_seq, float p, float scale, uint64_t seed,
                uint64_t offset) {
  extern __shared__ __align__(16) float smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
  const int hc = blockIdx.y;
  for (int f = tid; f < HC * 3 * TILE; f += THREADS) smem[f] = 0.f;
  __syncthreads();
  float* Q = smem + (warp * 3 + 0) * TILE;
  const float* K = Q + TILE;
  const float* V = K + TILE;
  const int colbase = hc * (HC * DH) + warp * DH;
  for (int64_t seq = blockIdx.x; seq < n_seq; seq += gridDim.x) {
    __syncwarp();             // every lane is done with the previous title's tiles
    warp_fetch<3>(Q, qkv + seq * S * D3 + colbase, nullptr, lane, seq * S, colbase, 0.f, 1.f, 0, 0);
    Frag a;
    zero(a);
    gemm_nt(a, Q, K, g, t);
    softmax_rows(a, t);
    Frag o;
    zero(o);
    gemm_frag_n(o, a, V, g, t);
    if (p > 0.f) {
      // dropout-2 masks: 100 aligned groups of four columns = 100 Philox evaluations, 4 per lane, written over the dead
      // Q block (rows / columns < 20 only: the padding stays zero) and read back in accumulator order
      __syncwarp();
      for (int f = lane; f < S * (DH / 4); f += 32) {
        const int j = f / (DH / 4), d4 = f % (DH / 4);
        *reinterpret_cast<float4*>(Q + j * ST + d4 * 4) =
            dropout_mask4((uint64_t)(seq * S + j) * D + colbase + d4 * 4, DROPOUT_STREAM_CTX, p, scale, seed, offset);
      }
      __syncwarp();
#pragma unroll
      for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int nt = 0; nt < 3; ++nt)
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            const int row = mt * 16 + g + 8 * half, col = nt * 8 + 2 * t;
            if (row < S && col < S) {
              const float2 m = *reinterpret_cast<const float2*>(Q + row * ST + col);
              o[mt][nt][half * 2] *= m.x;
              o[mt][nt][half * 2 + 1] *= m.y;
            }
          }
    }
    store_rows(ctx + seq * S * D + colbase, D, o, g, t);
  }
}

// MASKED: keys at positions >= lengths[seq] are left out (see the header); otherwise `lengths` is not read
template <bool MASKED>
__global__ void __launch_bounds__(THREADS)
attn_bwd_kernel(const float* __restrict__ qkv, const float* __restrict__ d_ctx, float* __restrict__ d_qkv,
                float* __restrict__ d_qkv_t, int64_t ldt, int64_t n_seq, float p, float scale, uint64_t seed, uint64_t offset,
                const int32_t* __restrict__ lengths) {
  extern __shared__ __align__(16) float smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
  const int hc = blockIdx.y;
  for (int f = tid; f < HC * 4 * TILE; f += THREADS) smem[f] = 0.f;
  __syncthreads();
  constexpr float INV_SQRT_DH = 1.f / SQRT_DH;
  float* Q = smem + (warp * 4 + 0) * TILE;
  float* K = Q + TILE;
  float* V = K + TILE;
  float* G = V + TILE;
  const int colbase = hc * (HC * DH) + warp * DH;
#ifdef NRMS_AMMA_TRACE
  long long tr[12] = {0};
#endif
  for (int64_t seq = blockIdx.x; seq < n_seq; seq += gridDim.x) {
    AT(0);
    __syncwarp();             // every lane is done with the previous title's tiles
    AT(1);
    AT(2);
    warp_fetch<4>(Q, qkv + seq * S * D3 + colbase, d_ctx + seq * S * D + colbase, lane, seq * S, colbase, p, scale, seed, offset);
    AT(3);
    Frag a, dp;
    zero(a);
    gemm_nt(a, Q, K, g, t);
    AT(4);
    softmax_rows(a, t, MASKED ? key_limit(lengths, seq, S) : S);       // a = attn (masked key columns 0)
    AT(5);
    zero(dp);
    gemm_nt(dp, G, V, g, t);                  // dp = dO V^T
    AT(6);
    // ds = attn (dp - sum_j attn dp) / sqrt 20, in place over dp
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        float delta = 0.f;
#pragma unroll
        for (int nt = 0; nt < 3; ++nt)
#pragma unroll
          for (int e = 0; e < 2; ++e) delta = fmaf(a[mt][nt][half * 2 + e], dp[mt][nt][half * 2 + e], delta);
        delta += __shfl_xor_sync(0xffffffffu, delta, 1);
        delta += __shfl_xor_sync(0xffffffffu, delta, 2);
#pragma unroll
        for (int nt = 0; nt < 3; ++nt)
#pragma unroll
          for (int e = 0; e < 2; ++e)
            dp[mt][nt][half * 2 + e] = a[mt][nt][half * 2 + e] * (dp[mt][nt][half * 2 + e] - delta) * INV_SQRT_DH;
      }
    float* out = d_qkv + seq * S * D3 + colbase;
    float* out_t = d_qkv_t ? d_qkv_t + (int64_t)colbase * ldt + seq * S : nullptr;     // [900, ldt]: row = column of dQKV
    __syncwarp();
    park(V, dp, g, t);                        // V is dead: dS (TF32-rounded) parked as [i][j]
    Frag r;
    zero(r);
    gemm_frag_n(r, dp, K, g, t);              // dQ = dS K
    store_rows(out, D3, r, g, t);
    if (out_t) store_rows_t(out_t, ldt, K, r, lane, g, t);       // K is dead from here on
    AT(7);
    __syncwarp();
    // K is dead: the rounding residue dS - tf32(dS) goes there.  The rows of dS sum to ~0 (the softmax Jacobian), and
    // the K-bias gradient is exactly that sum: with dS = hi + lo in the dK contraction it cancels to fp32 accuracy
    // instead of leaving 2^-11-sized rounding noise.
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int nt = 0; nt < 3; ++nt)
#pragma unroll
        for (int e = 0; e < 4; ++e) dp[mt][nt][e] -= tf32_round(dp[mt][nt][e]);
    park(K, dp, g, t);
    __syncwarp();
    zero(r);
    gemm_tn(r, V, Q, g, t);                   // dK = (dS_hi + dS_lo)^T Q
    gemm_tn(r, K, Q, g, t);
    store_rows(out + D, D3, r, g, t);
    if (out_t) store_rows_t(out_t + (int64_t)D * ldt, ldt, K, r, lane, g, t);       // dS_lo in K is dead
    AT(8);
    __syncwarp();
    park(V, a, g, t);                         // dS is dead: attn parked as [i][j]
    __syncwarp();
    zero(r);
    gemm_tn(r, V, G, g, t);                   // dV = attn^T dO
    store_rows(out + 2 * D, D3, r, g, t);
    if (out_t) store_rows_t(out_t + (int64_t)2 * D * ldt, ldt, K, r, lane, g, t);
    AT(9);
#ifdef NRMS_AMMA_TRACE
    if (threadIdx.x == 0 && blockIdx.x == 0 && blockIdx.y == 0 && seq == (int64_t)gridDim.x * 2) {
      printf("attn_bwd sync+issue/wait/round/S/softmax/dP/dS+dQ/dK/dV cycles:");
      for (int k_ = 1; k_ < 10; ++k_) printf(" %lld", tr[k_] - tr[k_ - 1]);
      printf("\n");
    }
#endif
  }
}

}  // namespace amma

// ---- 50-token texts (the abstract encoder of model/Exp1) ------------------------------------------------------------
// Same contractions and semantics as the title kernels above, but their layout does not carry over: per (text, head) the
// scores are 50 x 50, so a whole score fragment per warp would not fit the registers, and dS / attn (50 x 50) no longer
// fit the dead K / V tiles the title backward parks them in.
//
// Layout.  One warp per (text, head); tiles Q, K, V (and G = dO in the backward) of [56 rows][28 floats]: keys pad to 7
// n8 tiles (rows 50..55 stay zero), queries to 4 m16 tiles (rows 56..63 are not stored: their fragment loads read zero),
// the head dimension to 3 k8 steps (columns 20..27 stay zero).  The tiles are read-only once staged.
//   forward:  per 16-query tile, S = Q K^T (28 accumulators), attn, O = attn V (12 accumulators), dropout-2 mask drawn
//             in registers (one Philox evaluation per lane and 8-column block, halves exchanged between lane pairs)
//   backward, pass 1, per 16-query tile:  S = Q K^T, attn, dP = G V^T, dS, dQ = dS K; 1 / (sum + eps) and
//             delta = sum_j attn dP of every query row are kept in shared memory (2 x 64 floats per head)
//   backward, pass 2, per 16-key tile:    S^T = K Q^T, attn^T = exp(S^T / sqrt 20) / (sum + eps) of the query column,
//             dP^T = V G^T, dS^T = attn^T (dP^T - delta) / sqrt 20, dK = dS^T Q (dS split hi + lo, as in the title
//             kernel: the K-bias gradient is a sum that cancels), dV = attn^T G
// So the scores and exponentials are computed twice (seven 64 x 56 x 24 contractions instead of five) rather than parking
// two 50 x 50 matrices per head in shared memory.  Heads per CTA: 3 in the forward (56 KB, 4 CTAs per SM), 1 in the
// backward (25.6 KB, 8 CTAs per SM); the warps never wait for each other, so a CTA of one warp loses nothing.
// The backward's MASKED instantiation zeroes the exponentials of masked keys in both passes: key columns in pass 1,
// key rows of the transposed tile in pass 2 (see the key mask of the title kernels).
namespace amma50 {

constexpr int S = 50;            // tokens per text
constexpr int RT = 56;           // tile rows (7 x 8)
constexpr int ST = 28;           // tile row pitch in floats (conflict-free fragment loads, see amma)
constexpr int TILE = RT * ST;
constexpr int MT = 4;            // 16-row tiles over the queries (64 >= 50)
constexpr int NT = 7;            // 8-column tiles over the keys (56 >= 50)
constexpr int HC_FWD = 3, HC_BWD = 1;
constexpr int ZS = 64;           // floats per per-row vector (1 / (sum + eps), delta) of the backward

typedef float Row[NT][4];        // accumulators of 16 rows x 56 columns
typedef float Out[3][4];         // accumulators of 16 rows x 24 columns (the head dimension)

template <typename F>
__device__ __forceinline__ void zero(F& c) {
  float* f = &c[0][0];
#pragma unroll
  for (int i = 0; i < (int)(sizeof(F) / sizeof(float)); ++i) f[i] = 0.f;
}

// c[i][j] += sum_d A[m0 + i][d] B[j][d]     (16 rows of tile A from row m0, the 56 rows of tile B)
__device__ __forceinline__ void gemm_nt(Row& c, const float* A, int m0, const float* B, int g, int t) {
  const int r0 = m0 + g, r1 = r0 + 8;
#pragma unroll
  for (int ks = 0; ks < 3; ++ks) {
    const uint32_t a0 = amma::ld(A + r0 * ST + ks * 8 + t), a2 = amma::ld(A + r0 * ST + ks * 8 + t + 4);
    const uint32_t a1 = r1 < RT ? amma::ld(A + r1 * ST + ks * 8 + t) : 0u;
    const uint32_t a3 = r1 < RT ? amma::ld(A + r1 * ST + ks * 8 + t + 4) : 0u;
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      const uint32_t b0 = amma::ld(B + (nt * 8 + g) * ST + ks * 8 + t), b1 = amma::ld(B + (nt * 8 + g) * ST + ks * 8 + t + 4);
      amma::mma_tf32(c[nt], a0, a1, a2, a3, b0, b1);
    }
  }
}

// c[i][d] += sum_j P[i][j] B[j][d]          (P: accumulators used in place as the A operand, see amma::gemm_frag_n)
// SPLIT: P is taken as tf32(P) + tf32(P - tf32(P)), two products per step
template <bool SPLIT>
__device__ __forceinline__ void gemm_frag_n(Out& c, const Row& p, const float* B, int g, int t) {
#pragma unroll
  for (int ks = 0; ks < NT; ++ks) {
    float hi[4], lo[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      hi[e] = amma::tf32_round(p[ks][e]);
      lo[e] = SPLIT ? amma::tf32_round(p[ks][e] - hi[e]) : 0.f;
    }
#pragma unroll
    for (int nt = 0; nt < 3; ++nt) {
      const uint32_t b0 = amma::ld(B + (ks * 8 + 2 * t) * ST + nt * 8 + g), b1 = amma::ld(B + (ks * 8 + 2 * t + 1) * ST + nt * 8 + g);
      amma::mma_tf32(c[nt], __float_as_uint(hi[0]), __float_as_uint(hi[2]), __float_as_uint(hi[1]), __float_as_uint(hi[3]), b0, b1);
      if (SPLIT)
        amma::mma_tf32(c[nt], __float_as_uint(lo[0]), __float_as_uint(lo[2]), __float_as_uint(lo[1]), __float_as_uint(lo[3]), b0, b1);
    }
  }
}

constexpr float SCALE_LOG2E = 1.4426950408889634f / amma::SQRT_DH;     // exp(s / sqrt 20) = 2^(s * log2(e) / sqrt 20)
constexpr float INV_SQRT_DH = 1.f / amma::SQRT_DH;

// raw scores -> attention weights in place (key columns >= jmax -> 0; jmax = 50 or the clamped length);
// inv[half] = 1 / (row sum + 1e-8) of row g + 8 half
__device__ __forceinline__ void softmax_rows(Row& c, int t, float (&inv)[2], int jmax = S) {
#pragma unroll
  for (int half = 0; half < 2; ++half) {
    float sum = 0.f;
#pragma unroll
    for (int nt = 0; nt < NT; ++nt)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int col = nt * 8 + 2 * t + e;
        const float v = col < jmax ? amma::ex2(c[nt][half * 2 + e] * SCALE_LOG2E) : 0.f;
        c[nt][half * 2 + e] = v;
        sum += v;
      }
    sum += __shfl_xor_sync(0xffffffffu, sum, 1);
    sum += __shfl_xor_sync(0xffffffffu, sum, 2);
    inv[half] = 1.f / (sum + amma::ATTN_EPS);
#pragma unroll
    for (int nt = 0; nt < NT; ++nt)
#pragma unroll
      for (int e = 0; e < 2; ++e) c[nt][half * 2 + e] *= inv[half];
  }
}

// rows m0 .. m0 + 15 (those < 50) of an Out fragment to global rows of pitch ld_ (two floats per store)
__device__ __forceinline__ void store_rows(float* dst, int64_t ld_, const Out& c, int m0, int g, int t) {
#pragma unroll
  for (int nt = 0; nt < 3; ++nt)
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      const int row = m0 + g + 8 * half, col = nt * 8 + 2 * t;
      if (row < S && col < DH)
        *reinterpret_cast<float2*>(dst + row * ld_ + col) = make_float2(c[nt][half * 2], c[nt][half * 2 + 1]);
    }
}

// the same rows written transposed, dstT[col * ldt + row] (the K-major operand of the dWqkv contraction).  A column of a
// 16-row tile is 64 contiguous bytes of dstT, and each store instruction of the warp fills four 32-byte sectors (eight
// consecutive rows of four columns), so the scalar stores waste no bandwidth.
__device__ __forceinline__ void store_cols(float* dstT, int64_t ldt, const Out& c, int m0, int g, int t) {
#pragma unroll
  for (int nt = 0; nt < 3; ++nt)
#pragma unroll
    for (int half = 0; half < 2; ++half)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int row = m0 + g + 8 * half, col = nt * 8 + 2 * t + e;
        if (row < S && col < DH) dstT[(int64_t)col * ldt + row] = c[nt][half * 2 + e];
      }
}

// warp-private staging as amma::warp_fetch: tile w <- columns [w*300 + col0, +20) of the text's 50 qkv rows for w < 3,
// of its d_ctx rows (times the dropout-2 mask) for w == 3; 250 sixteen-byte pieces per tile, rounded to TF32 in place
template <int NTILES>
__device__ __forceinline__ void fetch(float* tiles, const float* __restrict__ qkv_head, const float* __restrict__ g_head,
                                      int lane, int64_t row0, int col0, float p, float scale, uint64_t seed, uint64_t offset) {
  constexpr int PIECES = S * (DH / 4);
  constexpr int PT = (PIECES + 31) / 32;
#pragma unroll
  for (int w = 0; w < NTILES; ++w)
#pragma unroll
    for (int k = 0; k < PT; ++k) {
      const int f = lane + 32 * k, j = f / (DH / 4), d4 = f % (DH / 4);
      if (f < PIECES) {
        const float* src = (w < 3) ? qkv_head + (int64_t)j * D3 + w * D + d4 * 4 : g_head + (int64_t)j * D + d4 * 4;
        amma::cp_async16(tiles + w * TILE + j * ST + d4 * 4, src);
      }
    }
  amma::cp_async_wait_all();
#pragma unroll
  for (int w = 0; w < NTILES; ++w)
#pragma unroll
    for (int k = 0; k < PT; ++k) {
      const int f = lane + 32 * k, j = f / (DH / 4), d4 = f % (DH / 4);
      if (f < PIECES) {
        float4* q = reinterpret_cast<float4*>(tiles + w * TILE + j * ST + d4 * 4);
        float4 x = *q;
        if (w == 3 && p > 0.f) {
          const float4 m = dropout_mask4((uint64_t)(row0 + j) * D + col0 + d4 * 4, amma::DROPOUT_STREAM_CTX, p, scale, seed, offset);
          x.x *= m.x; x.y *= m.y; x.z *= m.z; x.w *= m.w;
        }
        *q = make_float4(amma::tf32_round(x.x), amma::tf32_round(x.y), amma::tf32_round(x.z), amma::tf32_round(x.w));
      }
    }
  __syncwarp();
}

__global__ void __launch_bounds__(HC_FWD * 32)
attn50_fwd_kernel(const float* __restrict__ qkv, float* __restrict__ ctx, int64_t n_seq, float p, float scale, uint64_t seed,
                  uint64_t offset) {
  extern __shared__ __align__(16) float smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
  for (int f = tid; f < HC_FWD * 3 * TILE; f += blockDim.x) smem[f] = 0.f;
  __syncthreads();
  float* Q = smem + warp * 3 * TILE;
  const float* K = Q + TILE;
  const float* V = K + TILE;
  const int colbase = blockIdx.y * (HC_FWD * DH) + warp * DH;
  for (int64_t seq = blockIdx.x; seq < n_seq; seq += gridDim.x) {
    __syncwarp();             // every lane is done with the previous text's tiles
    fetch<3>(Q, qkv + seq * S * D3 + colbase, nullptr, lane, seq * S, colbase, 0.f, 1.f, 0, 0);
#pragma unroll 1
    for (int mt = 0; mt < MT; ++mt) {
      Row a;
      zero(a);
      gemm_nt(a, Q, mt * 16, K, g, t);
      float inv[2];
      softmax_rows(a, t, inv);
      Out o;
      zero(o);
      gemm_frag_n<false>(o, a, V, g, t);
      if (p > 0.f) {
        // dropout-2 mask of element (seq*50 + row) * 300 + col: a Philox evaluation yields an aligned group of four
        // columns, and a lane pair (t, t^1) holds two columns of one group in two rows.  The even lane draws row g's
        // group, the odd lane row g + 8's, and each hands its partner the half it needs.
#pragma unroll
        for (int nt = 0; nt < 3; ++nt) {
          const int odd = t & 1;
          const float4 m = dropout_mask4((uint64_t)(seq * S + mt * 16 + g + 8 * odd) * D + colbase + nt * 8 + (t >> 1) * 4,
                                         amma::DROPOUT_STREAM_CTX, p, scale, seed, offset);
          const float r0 = __shfl_xor_sync(0xffffffffu, odd ? m.x : m.z, 1);
          const float r1 = __shfl_xor_sync(0xffffffffu, odd ? m.y : m.w, 1);
          o[nt][0] *= odd ? r0 : m.x;
          o[nt][1] *= odd ? r1 : m.y;
          o[nt][2] *= odd ? m.z : r0;
          o[nt][3] *= odd ? m.w : r1;
        }
      }
      store_rows(ctx + seq * S * D + colbase, D, o, mt * 16, g, t);
    }
  }
}

template <bool MASKED>
__global__ void __launch_bounds__(HC_BWD * 32)
attn50_bwd_kernel(const float* __restrict__ qkv, const float* __restrict__ d_ctx, float* __restrict__ d_qkv,
                  float* __restrict__ d_qkv_t, int64_t ldt, int64_t n_seq, float p, float scale, uint64_t seed,
                  uint64_t offset, const int32_t* __restrict__ lengths) {
  extern __shared__ __align__(16) float smem[];
  constexpr int PER_WARP = 4 * TILE + 2 * ZS;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
  for (int f = tid; f < HC_BWD * PER_WARP; f += blockDim.x) smem[f] = 0.f;
  __syncthreads();
  float* Q = smem + warp * PER_WARP;
  const float* K = Q + TILE;
  const float* V = K + TILE;
  const float* G = V + TILE;
  float* zinv = Q + 4 * TILE;
  float* delta = zinv + ZS;
  const int colbase = blockIdx.y * (HC_BWD * DH) + warp * DH;
  for (int64_t seq = blockIdx.x; seq < n_seq; seq += gridDim.x) {
    __syncwarp();             // every lane is done with the previous text's tiles and row vectors
    fetch<4>(Q, qkv + seq * S * D3 + colbase, d_ctx + seq * S * D + colbase, lane, seq * S, colbase, p, scale, seed, offset);
    float* out = d_qkv + seq * S * D3 + colbase;
    float* out_t = d_qkv_t ? d_qkv_t + (int64_t)colbase * ldt + seq * S : nullptr;     // [900, ldt]: row = column of dQKV
    const int jmax = MASKED ? amma::key_limit(lengths, seq, S) : S;
    // ---- pass 1: query tiles -> dQ, row vectors ----
#pragma unroll 1
    for (int mt = 0; mt < MT; ++mt) {
      Row a, dp;
      zero(a);
      gemm_nt(a, Q, mt * 16, K, g, t);
      float inv[2];
      softmax_rows(a, t, inv, jmax);          // a = attn
      zero(dp);
      gemm_nt(dp, G, mt * 16, V, g, t);       // dp = dO V^T
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
        const int row = mt * 16 + g + 8 * half;
        if (t == 0 && row < S) {
          zinv[row] = inv[half];
          delta[row] = dl;
        }
      }
      Out r;
      zero(r);
      gemm_frag_n<false>(r, dp, K, g, t);     // dQ = dS K
      store_rows(out, D3, r, mt * 16, g, t);
      if (out_t) store_cols(out_t, ldt, r, mt * 16, g, t);
    }
    __syncwarp();             // the row vectors are visible to every lane
    // ---- pass 2: key tiles -> dK, dV ----
#pragma unroll 1
    for (int kt = 0; kt < MT; ++kt) {
      Row a, dp;
      zero(a);
      gemm_nt(a, K, kt * 16, Q, g, t);        // S^T: rows = keys, columns = queries
      zero(dp);
      gemm_nt(dp, V, kt * 16, G, g, t);       // dP^T = V dO^T
#pragma unroll
      for (int nt = 0; nt < NT; ++nt)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int col = nt * 8 + 2 * t + e;
          const float z = col < S ? zinv[col] : 0.f, dl = col < S ? delta[col] : 0.f;
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            const bool keep = col < S && (!MASKED || kt * 16 + g + 8 * half < jmax);        // query column, key row
            const float at = keep ? amma::ex2(a[nt][half * 2 + e] * SCALE_LOG2E) * z : 0.f;
            a[nt][half * 2 + e] = at;                                                     // attn^T
            dp[nt][half * 2 + e] = at * (dp[nt][half * 2 + e] - dl) * INV_SQRT_DH;        // dS^T
          }
        }
      Out r;
      zero(r);
      gemm_frag_n<true>(r, dp, Q, g, t);      // dK = (dS_hi + dS_lo)^T Q
      store_rows(out + D, D3, r, kt * 16, g, t);
      if (out_t) store_cols(out_t + (int64_t)D * ldt, ldt, r, kt * 16, g, t);
      zero(r);
      gemm_frag_n<false>(r, a, G, g, t);      // dV = attn^T dO
      store_rows(out + 2 * D, D3, r, kt * 16, g, t);
      if (out_t) store_cols(out_t + (int64_t)2 * D * ldt, ldt, r, kt * 16, g, t);
    }
  }
}

}  // namespace amma50

int attn_mma50_fwd(const float* qkv, float* ctx, int64_t n_seq, float p, uint64_t seed, uint64_t offset, cudaStream_t st) {
  const size_t smem = (size_t)amma50::HC_FWD * 3 * amma50::TILE * sizeof(float);
  static bool configured[64] = {false};
  if (cudaError_t e = set_max_dynamic_smem(amma50::attn50_fwd_kernel, (int)smem, configured)) return cuda_fail(e, "attn_mma50_fwd attr");
  int64_t gx = n_seq < (int64_t)num_sms() * 8 ? n_seq : (int64_t)num_sms() * 8;
  const float scale = p > 0.f ? 1.f / (1.f - p) : 1.f;
  amma50::attn50_fwd_kernel<<<dim3((unsigned)gx, H / amma50::HC_FWD), amma50::HC_FWD * 32, smem, st>>>(qkv, ctx, n_seq, p, scale,
                                                                                                   seed, offset);
  NRMS_LAUNCH_CHECK("attn_mma50_fwd");
  return NRMS_OK;
}

template <bool MASKED>
static int attn_mma50_bwd_launch(const float* qkv, const float* d_ctx, float* d_qkv, float* d_qkv_t, int64_t ldt,
                                 int64_t n_seq, float p, uint64_t seed, uint64_t offset, cudaStream_t st,
                                 const int32_t* lengths) {
  const size_t smem = (size_t)amma50::HC_BWD * (4 * amma50::TILE + 2 * amma50::ZS) * sizeof(float);
  static bool configured[64] = {false};
  if (cudaError_t e = set_max_dynamic_smem(amma50::attn50_bwd_kernel<MASKED>, (int)smem, configured))
    return cuda_fail(e, "attn_mma50_bwd attr");
  int64_t gx = n_seq < (int64_t)num_sms() * 8 ? n_seq : (int64_t)num_sms() * 8;
  const float scale = p > 0.f ? 1.f / (1.f - p) : 1.f;
  amma50::attn50_bwd_kernel<MASKED><<<dim3((unsigned)gx, H / amma50::HC_BWD), amma50::HC_BWD * 32, smem, st>>>(
      qkv, d_ctx, d_qkv, d_qkv_t, ldt, n_seq, p, scale, seed, offset, lengths);
  NRMS_LAUNCH_CHECK("attn_mma50_bwd");
  return NRMS_OK;
}

int attn_mma50_bwd(const float* qkv, const float* d_ctx, float* d_qkv, float* d_qkv_t, int64_t ldt, int64_t n_seq, float p,
                   uint64_t seed, uint64_t offset, cudaStream_t st, const int32_t* lengths) {
  return lengths ? attn_mma50_bwd_launch<true>(qkv, d_ctx, d_qkv, d_qkv_t, ldt, n_seq, p, seed, offset, st, lengths)
                 : attn_mma50_bwd_launch<false>(qkv, d_ctx, d_qkv, d_qkv_t, ldt, n_seq, p, seed, offset, st, nullptr);
}

int attn_mma_fwd(const float* qkv, float* ctx, int64_t n_seq, float p, uint64_t seed, uint64_t offset, cudaStream_t st) {
  const size_t smem = amma::NBUF * (size_t)amma::HC * 3 * amma::TILE * sizeof(float);
  static bool configured[64] = {false};
  if (cudaError_t e = set_max_dynamic_smem(amma::attn_fwd_kernel, (int)smem, configured)) return cuda_fail(e, "attn_mma_fwd attr");
  int64_t gx = n_seq < (int64_t)num_sms() * 8 ? n_seq : (int64_t)num_sms() * 8;
  const float scale = p > 0.f ? 1.f / (1.f - p) : 1.f;
  amma::attn_fwd_kernel<<<dim3((unsigned)gx, H / amma::HC), amma::THREADS, smem, st>>>(qkv, ctx, n_seq, p, scale, seed, offset);
  NRMS_LAUNCH_CHECK("attn_mma_fwd");
  return NRMS_OK;
}

template <bool MASKED>
static int attn_mma_bwd_launch(const float* qkv, const float* d_ctx, float* d_qkv, float* d_qkv_t, int64_t ldt, int64_t n_seq,
                               float p, uint64_t seed, uint64_t offset, cudaStream_t st, const int32_t* lengths) {
  const size_t smem = amma::NBUF * (size_t)amma::HC * 4 * amma::TILE * sizeof(float);
  static bool configured[64] = {false};
  if (cudaError_t e = set_max_dynamic_smem(amma::attn_bwd_kernel<MASKED>, (int)smem, configured))
    return cuda_fail(e, "attn_mma_bwd attr");
  int64_t gx = n_seq < (int64_t)num_sms() * 8 ? n_seq : (int64_t)num_sms() * 8;
  const float scale = p > 0.f ? 1.f / (1.f - p) : 1.f;
  amma::attn_bwd_kernel<MASKED><<<dim3((unsigned)gx, H / amma::HC), amma::THREADS, smem, st>>>(
      qkv, d_ctx, d_qkv, d_qkv_t, ldt, n_seq, p, scale, seed, offset, lengths);
  NRMS_LAUNCH_CHECK("attn_mma_bwd");
  return NRMS_OK;
}

int attn_mma_bwd(const float* qkv, const float* d_ctx, float* d_qkv, float* d_qkv_t, int64_t ldt, int64_t n_seq, float p,
                 uint64_t seed, uint64_t offset, cudaStream_t st, const int32_t* lengths) {
  return lengths ? attn_mma_bwd_launch<true>(qkv, d_ctx, d_qkv, d_qkv_t, ldt, n_seq, p, seed, offset, st, lengths)
                 : attn_mma_bwd_launch<false>(qkv, d_ctx, d_qkv, d_qkv_t, ldt, n_seq, p, seed, offset, st, nullptr);
}

}  // namespace nrms
