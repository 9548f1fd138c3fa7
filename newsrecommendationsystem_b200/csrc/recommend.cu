// Single-user latency path (SURVEY 8 f4): what reference src/recommend.py:245-341 does for its one target user --
//   user_vector = model.get_user_vector(stack(news2vector[x] for x in clicked_news))      recommend.py:264-279
//   click_probability = model.get_prediction(stack(news2vector[c] for c in impression), user_vector)   :301-315
//   order = np.argsort(-(click_probability + 1) / 2)                                                    :338-340
// -- as TWO launches of thread-block clusters instead of ~25 batched-op launches over a batch of one.  FP32 on the
// CUDA cores throughout (reference arithmetic up to summation order): at one user the whole encoder is 16.5 M MACs
// and what matters is how many SMs share it and how few times they meet.
//
// Kernel A (15 clusters x 8 CTAs, one cluster per attention head): CTA r of cluster h projects history rows r, r+8, ..
// onto the head's 60 q|k|v columns, hands its k|v rows to the other seven CTAs through distributed shared memory, runs
// exp-softmax attention for its own rows, and writes (a) the head's slice of its context rows and (b) that slice's
// contribution to the additive layer, tpart[h][i][:] = C_h[i] Wa[:, 20h:20h+20]^T -- the additive linear map is a sum
// over heads, so no CTA ever needs a whole context row.
// Kernel B (one cluster of 8 CTAs): CTA r sums the 15 partials for 25 of the 200 additive units, adds the bias, takes
// tanh and the dot with the query; the eight partial scores per row meet in every CTA's shared memory; each CTA then
// knows the softmax weights, forms the user vector (the context rows were copied into shared memory while the partials
// were in flight), scores every 8th candidate and hands its scores to all eight CTAs; each CTA then ranks an eighth of
// the candidates by counting (rank = number of candidates that sort before it), so no CTA sorts alone.
// Both kernels are written for latency, not throughput: every phase issues all of its global loads before it uses any
// (measured with clock64 stamps, -DNRMS_LAT_TRACE: the first version spent 16k of its 36k cycles in five dependent
// rounds of partial-sum loads and 9k in fifty dependent context loads).
#include <cooperative_groups.h>
#include "common.cuh"

namespace cg = cooperative_groups;

namespace nrms {
namespace lat {

constexpr int S = 50;           // config.num_clicked_news_a_user
constexpr int CL = 8;           // CTAs per cluster (portable maximum)
constexpr int RMAX = 7;         // history rows per CTA: ceil(50 / 8)
constexpr int XS = 308;         // padded row stride (floats): 16-byte aligned, conflict-free for strided float4 reads
constexpr int THREADS = 256;
constexpr float SQRT_DH = 4.47213595499957939f;
constexpr int MAX_SORT = 4096;

struct SmemA {
  float x[RMAX][XS];            // this CTA's history rows
  float w[3 * DH][XS];          // the head's q|k|v weight rows: j = 20 * {q,k,v} + column
  float bias[64];
  float q[RMAX][DH];
  float kv[S][2 * DH];          // k (0..19) | v (20..39) of all 50 rows; every CTA of the cluster writes its rows here
  float e[RMAX][S + 2];
  float ctx[RMAX][DH];
  float part[4][RMAX][64];      // projection partial sums of the four K quarters
  float kvl[RMAX][2 * DH];      // k | v of my rows before they are handed out
};

#ifdef NRMS_LAT_TRACE
#define LAT_T(k) do { if (threadIdx.x == 0 && blockIdx.x == 0) tr[k] = clock64(); } while (0)
#define LAT_DECL long long tr[12] = {0}
#define LAT_PRINT(name, n) do { if (threadIdx.x == 0 && blockIdx.x == 0) { printf(name); for (int k_ = 1; k_ < n; ++k_) printf(" %lld", tr[k_] - tr[k_ - 1]); printf("\n"); } } while (0)
#else
#define LAT_T(k)
#define LAT_DECL
#define LAT_PRINT(name, n)
#endif

// Ranking key of a score: unsigned order = score order, -0 == +0, and NaN (key 0) below every number, -inf included.
__device__ __forceinline__ uint32_t rank_key(float s) {
  if (s != s) return 0u;
  const uint32_t u = __float_as_uint(s == 0.f ? 0.f : s);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  const uint32_t s = (uint32_t)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }

__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(THREADS)
head_kernel(const float* __restrict__ table, int64_t n_rows, const int32_t* __restrict__ hist,
            const float* __restrict__ wqkv, const float* __restrict__ bqkv, const float* __restrict__ wa,
            float* __restrict__ ctx_g, float* __restrict__ tpart) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  SmemA& sm = *reinterpret_cast<SmemA*>(smem_raw);
  cg::cluster_group cluster = cg::this_cluster();
  const int r = (int)cluster.block_rank();
  const int h = blockIdx.x / CL;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n_mine = (S - r + CL - 1) / CL;      // rows r, r + 8, ... < 50
  LAT_DECL;
  LAT_T(0);

  // ---- stage this CTA's history rows (index load, then the row: the longer dependent chain goes first) and the head's
  //      weight rows, as 16-byte async copies ----
  for (int f = tid; f < RMAX * DV4; f += THREADS) {
    const int ii = f / DV4, l = f % DV4;
    if (ii < n_mine) {
      int64_t src = hist[r + CL * ii];
      if (src < 0 || src >= n_rows) src = n_rows - 1;     // callers pass the zero PADDED_NEWS row last; see the header
      cp_async16(&sm.x[ii][4 * l], table + src * D + 4 * l);
    } else {
      *reinterpret_cast<float4*>(&sm.x[ii][4 * l]) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
  for (int f = tid; f < 3 * DH * DV4; f += THREADS) {
    const int j = f / DV4, l = f % DV4;
    const int64_t row = (int64_t)(j / DH) * D + h * DH + (j % DH);
    cp_async16(&sm.w[j][4 * l], wqkv + row * D + 4 * l);
  }
  if (tid < 3 * DH) sm.bias[tid] = bqkv[(tid / DH) * D + h * DH + (tid % DH)];
  // the slice of W_a this thread needs at the end (unit q = tid, columns 20h .. 20h+19), fetched early
  float4 wa4[DH / 4];
  if (tid < QD) {
#pragma unroll
    for (int k = 0; k < DH / 4; ++k) wa4[k] = __ldg(reinterpret_cast<const float4*>(wa + (int64_t)tid * D + h * DH) + k);
  }
  cp_async_wait_all();
  __syncthreads();
  LAT_T(1);

  // ---- projection: warp = (column half, quarter of the 300-long dot product); x reads are warp broadcasts ----
  {
    const int j = (warp & 1) * 32 + lane, lq = warp >> 1;
    const int jc = j < 3 * DH ? j : 3 * DH - 1;
    const int l0 = lq * 19, l1 = (l0 + 19 < DV4) ? l0 + 19 : DV4;
    float acc[RMAX];
#pragma unroll
    for (int ii = 0; ii < RMAX; ++ii) acc[ii] = 0.f;
#pragma unroll 4
    for (int l = l0; l < l1; ++l) {
      const float4 wv = *reinterpret_cast<const float4*>(&sm.w[jc][4 * l]);
#pragma unroll
      for (int ii = 0; ii < RMAX; ++ii) {
        const float4 xv = *reinterpret_cast<const float4*>(&sm.x[ii][4 * l]);
        acc[ii] = fmaf(xv.w, wv.w, fmaf(xv.z, wv.z, fmaf(xv.y, wv.y, fmaf(xv.x, wv.x, acc[ii]))));
      }
    }
#pragma unroll
    for (int ii = 0; ii < RMAX; ++ii) sm.part[lq][ii][j] = acc[ii];
  }
  __syncthreads();
  for (int f = tid; f < RMAX * 3 * DH; f += THREADS) {
    const int ii = f / (3 * DH), j = f % (3 * DH);
    const float v = sm.bias[j] + ((sm.part[0][ii][j] + sm.part[1][ii][j]) + (sm.part[2][ii][j] + sm.part[3][ii][j]));
    if (j < DH) sm.q[ii][j] = v;
    else sm.kvl[ii][j - DH] = v;
  }
  __syncthreads();
  // k | v of my rows go to every CTA of the cluster (distributed shared memory, 16-byte stores)
  for (int f = tid; f < CL * RMAX * (2 * DH / 4); f += THREADS) {
    const int dst = f / (RMAX * 10), rem = f % (RMAX * 10), ii = rem / 10, c4 = rem % 10;
    if (ii < n_mine) {
      float* remote = cluster.map_shared_rank(&sm.kv[0][0], dst);
      *reinterpret_cast<float4*>(remote + (r + CL * ii) * (2 * DH) + 4 * c4) = *reinterpret_cast<const float4*>(&sm.kvl[ii][4 * c4]);
    }
  }
  LAT_T(2);
  cluster.sync();
  LAT_T(3);

  // ---- attention of my rows over all 50 keys (multihead_self.py:15-23: exp, no shift, eps in the denominator) ----
  for (int f = tid; f < n_mine * S; f += THREADS) {
    const int ii = f / S, j = f % S;
    float dp[DH / 4];
#pragma unroll
    for (int c = 0; c < DH / 4; ++c) {
      const float4 qv = *reinterpret_cast<const float4*>(&sm.q[ii][4 * c]);
      const float4 kv = *reinterpret_cast<const float4*>(&sm.kv[j][4 * c]);
      dp[c] = fmaf(qv.w, kv.w, fmaf(qv.z, kv.z, fmaf(qv.y, kv.y, qv.x * kv.x)));
    }
    sm.e[ii][j] = expf((((dp[0] + dp[1]) + (dp[2] + dp[3])) + dp[4]) / SQRT_DH);
  }
  __syncthreads();
  if (warp < n_mine) {          // one warp per row: Z, then attn = e / (Z + 1e-8) in place
    const float e0 = sm.e[warp][lane], e1 = (lane + 32 < S) ? sm.e[warp][lane + 32] : 0.f;
    const float den = warp_sum(e0 + e1) + 1e-8f;
    sm.e[warp][lane] = e0 / den;
    if (lane + 32 < S) sm.e[warp][lane + 32] = e1 / den;
  }
  __syncthreads();
  if (tid < n_mine * DH) {
    const int ii = tid / DH, d = tid % DH;
    float a0 = 0.f, a1 = 0.f;
#pragma unroll 5
    for (int j = 0; j < S; j += 2) {
      a0 = fmaf(sm.e[ii][j], sm.kv[j][DH + d], a0);
      a1 = fmaf(sm.e[ii][j + 1], sm.kv[j + 1][DH + d], a1);
    }
    const float acc = a0 + a1;
    sm.ctx[ii][d] = acc;
    ctx_g[(int64_t)(r + CL * ii) * D + h * DH + d] = acc;
  }
  __syncthreads();
  LAT_T(4);

  // ---- this head's share of the additive layer for my rows ----
  if (tid < QD) {
    for (int ii = 0; ii < n_mine; ++ii) {
      float acc = 0.f;
#pragma unroll
      for (int k = 0; k < DH / 4; ++k) {
        acc = fmaf(sm.ctx[ii][4 * k + 0], wa4[k].x, acc);
        acc = fmaf(sm.ctx[ii][4 * k + 1], wa4[k].y, acc);
        acc = fmaf(sm.ctx[ii][4 * k + 2], wa4[k].z, acc);
        acc = fmaf(sm.ctx[ii][4 * k + 3], wa4[k].w, acc);
      }
      tpart[((int64_t)h * S + (r + CL * ii)) * QD + tid] = acc;
    }
  }
  LAT_T(5);
  LAT_PRINT("head_kernel stage/project/sync/attention/additive cycles:", 6);
  // no CTA may exit while a peer can still write into its shared memory: all remote stores precede the first
  // cluster.sync(), and none follow it
}

struct SmemB {
  float sp[CL][S];              // partial pooling scores of the 8 unit slices (filled by all CTAs)
  float srow[S];
  float wrow[S];
  float user[D + 4];
  float ctx[S][D];              // the context rows (copied in while the partials are in flight)
};

__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(THREADS)
pool_score_kernel(const float* __restrict__ table, int64_t n_rows, const int32_t* __restrict__ cand, int C,
                  const float* __restrict__ ba, const float* __restrict__ qa, const float* __restrict__ ctx_g,
                  const float* __restrict__ tpart, float* __restrict__ user_vec, float* __restrict__ scores,
                  int32_t* __restrict__ order) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  SmemB& sm = *reinterpret_cast<SmemB*>(smem_raw);
  uint32_t* sc = reinterpret_cast<uint32_t*>(smem_raw + sizeof(SmemB));   // [C rounded up to 4]: every rank_key(score)
  cg::cluster_group cluster = cg::this_cluster();
  const int r = (int)cluster.block_rank();
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int QS = QD / CL;   // 25 additive units per CTA
  LAT_DECL;
  LAT_T(0);

  for (int f = tid; f < S * DV4; f += THREADS) cp_async16(&sm.ctx[0][0] + 4 * f, ctx_g + 4 * f);
  if (order != nullptr && tid < 4) sc[((C + 3) & ~3) - 1 - tid] = 0u;   // pad entries (j >= C) never sort before anything
  // warp = history rows warp, warp + 8, ..; lane = additive unit (25 of 32 lanes).  The loads of a batch of rows are all
  // issued before the first is used, and the row sums come from shuffles (shared-memory float atomics on one address
  // per row serialise: 13k of the first version's 16k cycles).
  {
    const int q = r * QS + (lane < QS ? lane : 0);
    const float bq = ba[q], qq = qa[q];
#pragma unroll
    for (int batch = 0; batch < 2; ++batch) {
      constexpr int RB = 4;
      float v[RB][H];
#pragma unroll
      for (int k = 0; k < RB; ++k) {
        const int i = warp + 8 * (batch * RB + k);
        const int ic = i < S ? i : 0;
#pragma unroll
        for (int hh = 0; hh < H; ++hh) v[k][hh] = __ldg(tpart + ((int64_t)hh * S + ic) * QD + q);
      }
#pragma unroll
      for (int k = 0; k < RB; ++k) {
        const int i = warp + 8 * (batch * RB + k);
        float t = bq;
#pragma unroll
        for (int hh = 0; hh < H; ++hh) t += v[k][hh];
        const float part = warp_sum(lane < QS ? tanhf(t) * qq : 0.f);
        if (lane == 0 && i < S) sm.srow[i] = part;
      }
    }
  }
  __syncthreads();
  if (tid < S) {
    const float x = sm.srow[tid];
    for (int dst = 0; dst < CL; ++dst) cluster.map_shared_rank(&sm.sp[0][0], dst)[r * S + tid] = x;
  }
  LAT_T(1);
  cluster.sync();
  LAT_T(2);

  // every CTA: softmax over the 50 rows (additive.py:37-39), then the user vector
  if (warp == 0) {
    float sv[2];
    float m = -INFINITY;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int i = lane + 32 * k;
      float a = 0.f;
      if (i < S) {
#pragma unroll
        for (int c = 0; c < CL; ++c) a += sm.sp[c][i];
        m = fmaxf(m, a);
      }
      sv[k] = a;
    }
    m = warp_max(m);
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int i = lane + 32 * k;
      sv[k] = (i < S) ? expf(sv[k] - m) : 0.f;
      sum += sv[k];
    }
    sum = warp_sum(sum);
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int i = lane + 32 * k;
      if (i < S) sm.wrow[i] = sv[k] / sum;
    }
  }
  cp_async_wait_all();
  __syncthreads();
  for (int d = tid; d < D; d += THREADS) {
    float a0 = 0.f, a1 = 0.f;
#pragma unroll 5
    for (int i = 0; i < S; i += 2) {
      a0 = fmaf(sm.wrow[i], sm.ctx[i][d], a0);
      a1 = fmaf(sm.wrow[i + 1], sm.ctx[i + 1][d], a1);
    }
    sm.user[d] = a0 + a1;
    if (r == 0) user_vec[d] = a0 + a1;
  }
  __syncthreads();
  LAT_T(3);

  // scores: warp per candidate, candidates r*8 + warp, + 64, ...; four rows in flight per warp.  With a ranking every
  // score also goes to all eight CTAs' shared memory (lane k stores to CTA k).
  {
    float4 u[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const int l = lane + 32 * k;
      u[k] = (l < DV4) ? *reinterpret_cast<const float4*>(&sm.user[4 * l]) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    uint32_t* sc_remote = (order != nullptr && lane < CL) ? cluster.map_shared_rank(sc, lane) : nullptr;
    constexpr int INF = 4;
    for (int c0 = r * 8 + warp; c0 < C; c0 += INF * CL * 8) {
      float4 a[INF][3];
#pragma unroll
      for (int t = 0; t < INF; ++t) {
        const int c = c0 + t * CL * 8;
        int64_t row = c < C ? cand[c] : 0;
        if (row < 0 || row >= n_rows) row = n_rows - 1;
        const float4* p = reinterpret_cast<const float4*>(table + row * D);
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          const int l = lane + 32 * k;
          a[t][k] = (l < DV4 && c < C) ? __ldg(p + l) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
#pragma unroll
      for (int t = 0; t < INF; ++t) {
        const int c = c0 + t * CL * 8;
        float s0 = 0.f;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          s0 = fmaf(a[t][k].x, u[k].x, s0); s0 = fmaf(a[t][k].y, u[k].y, s0);
          s0 = fmaf(a[t][k].z, u[k].z, s0); s0 = fmaf(a[t][k].w, u[k].w, s0);
        }
        s0 = warp_sum(s0);
        if (c < C) {
          if (lane == 0) scores[c] = s0;
          if (sc_remote != nullptr) sc_remote[c] = rank_key(s0);
        }
      }
    }
  }
  LAT_T(4);
  if (order == nullptr) return;
  cluster.sync();
  LAT_T(5);

  // rank by counting: candidate i goes to position #{j : k_j > k_i or (k_j == k_i and j < i)} over the keys k = rank_key(s)
  // -- descending score, equal scores in ascending candidate position, NaN last and in candidate order (np.argsort(-y) of
  // recommend.py:339 on a stable sort).  CTA r ranks the candidates i = r (mod 8); every comparison reads shared memory
  // as a warp broadcast.
  const int C4 = (C + 3) & ~3;
  for (int i = r + CL * tid; i < C; i += CL * THREADS) {
    const uint32_t si = sc[i];
    int before = 0;
    for (int j = 0; j < C4; j += 4) {
      const uint4 sj = *reinterpret_cast<const uint4*>(sc + j);
      before += (sj.x > si || (sj.x == si && j < i)) ? 1 : 0;
      before += (sj.y > si || (sj.y == si && j + 1 < i)) ? 1 : 0;
      before += (sj.z > si || (sj.z == si && j + 2 < i)) ? 1 : 0;
      before += (sj.w > si || (sj.w == si && j + 3 < i)) ? 1 : 0;
    }
    order[before] = i;
  }
  LAT_T(6);
  LAT_PRINT("pool_score_kernel partials/sync/user/score/sync/rank cycles:", 7);
}

}  // namespace lat
}  // namespace nrms

using namespace nrms;

extern "C" {

size_t nrms_recommend_workspace_bytes(void) {
  return align_up((size_t)lat::S * D * sizeof(float), 256) + (size_t)H * lat::S * QD * sizeof(float);
}

int nrms_recommend_user(const float* table, int64_t n_rows, const int32_t* hist_rows, const int32_t* cand_rows, int C,
                        const float* wqkv, const float* bqkv, const float* wa, const float* ba, const float* qa,
                        float* user_vec, float* scores, int32_t* order, void* workspace, size_t workspace_bytes,
                        void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  NRMS_CHECK_ARG(n_rows > 0 && C >= 0, NRMS_E_INVALID, "bad sizes");
  NRMS_CHECK_ARG(table && hist_rows && wqkv && bqkv && wa && ba && qa && user_vec, NRMS_E_INVALID, "null pointer");
  NRMS_CHECK_ARG(C == 0 || (cand_rows && scores), NRMS_E_INVALID, "null candidate / score pointer");
  NRMS_CHECK_ARG(aligned16(table) && aligned16(wqkv) && aligned16(wa), NRMS_E_INVALID, "pointers must be 16-byte aligned");
  NRMS_CHECK_ARG(order == nullptr || C <= lat::MAX_SORT, NRMS_E_UNSUPPORTED,
                 "the in-kernel ranking holds at most %d candidates (pass order = NULL for scores only)", lat::MAX_SORT);
  NRMS_CHECK_ARG(workspace && aligned16(workspace) && workspace_bytes >= nrms_recommend_workspace_bytes(),
                 NRMS_E_WORKSPACE, "workspace too small: need %zu bytes", nrms_recommend_workspace_bytes());
  float* ctx_g = reinterpret_cast<float*>(workspace);
  float* tpart = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + align_up((size_t)lat::S * D * sizeof(float), 256));
  static bool cfg_a[64] = {false}, cfg_b[64] = {false};
  if (cudaError_t e = set_max_dynamic_smem(lat::head_kernel, (int)sizeof(lat::SmemA), cfg_a)) return cuda_fail(e, "head_kernel attr");
  lat::head_kernel<<<H * lat::CL, lat::THREADS, sizeof(lat::SmemA), st>>>(table, n_rows, hist_rows, wqkv, bqkv, wa, ctx_g, tpart);
  NRMS_LAUNCH_CHECK("recommend head_kernel");
  const bool rank = order != nullptr && C > 0;
  const size_t smem_b = sizeof(lat::SmemB) + (rank ? (size_t)((C + 3) & ~3) * sizeof(float) : 0);
  if (cudaError_t e = set_max_dynamic_smem(lat::pool_score_kernel, (int)(sizeof(lat::SmemB) + lat::MAX_SORT * sizeof(float)), cfg_b))
    return cuda_fail(e, "pool_score_kernel attr");
  lat::pool_score_kernel<<<lat::CL, lat::THREADS, smem_b, st>>>(table, n_rows, cand_rows, C, ba, qa, ctx_g, tpart, user_vec,
                                                                scores, rank ? order : nullptr);
  NRMS_LAUNCH_CHECK("recommend pool_score_kernel");
  return NRMS_OK;
}

}  // extern "C"
