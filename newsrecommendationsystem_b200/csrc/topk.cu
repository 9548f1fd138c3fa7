// Top-k news of the whole table per user (nrms_topk_news): which k rows of the news-vector table score highest against
// each user vector, excluding rows the user already read -- without ever writing the [n_users, n_news] score matrix.
//
// Tensor mode, two launches after a small user conversion:
//   score pass (topk_score_kernel): a tcgen05 kind::f16 GEMM in the warp-specialised shape of tc_gemm_nt_kernel<true>.
//     Work item = (block of 128 users, split = a contiguous range of 256-row news tiles).  The users' fp16 rows are the
//     A operand, resident in shared memory for the item (5 chunks of 128 rows x 128 B); the news rows stream through a
//     4-stage TMA ring as the B operand; two 256-column TMEM accumulators let the epilogue of one tile overlap the MMAs
//     of the next.  The epilogue does not store scores: thread = TMEM lane = user row, and every score above the row's
//     running threshold is appended to that (row, split)'s candidate list in the workspace (select_push16).
//   merge (topk_merge_kernel): one CTA per user merges the lists of all splits, drops the excluded rows and writes the
//     k best in (score desc, row asc) order.
// FP32 mode: the same selection and merge over score blocks written by the CUDA-core sgemm (reference arithmetic).
//
// Selection.  A list holds at most `cap` entries; k' = k + n_exclude is what each list must keep for the merge to be
// exact (up to n_exclude of a split's best rows can be excluded afterwards).  When an append could overflow a list the
// warp compacts it cooperatively (radix select of the k'-th largest score over the list, then a stable compaction) and
// the row's threshold rises to that score.  Entries of a list are appended in ascending row order and compaction is
// stable, so among equal scores the smallest rows survive: a later row with a score equal to the threshold ranks below
// every kept entry and is not appended.  Scores travel as order-preserving 32-bit keys; NaN scores are never appended.
#include <cuda.h>
#include <cuda_fp16.h>
#include "tc_common.cuh"
#include "sgemm.cuh"

namespace nrms {

int make_tmap_k_major_f16(CUtensorMap* out, const void* base, int64_t rows, int cols, int64_t ld, int box_rows);

namespace topk {
using namespace tc;

constexpr int BM = 128, BN = 256;            // users per block, news rows per tile
constexpr int LD16 = 320;                    // halfs per packed row (300 values, table: 1.0 in column 300)
constexpr int KCH = LD16 / 64;               // 128-byte K chunks per row: 5
constexpr int A_CHUNK = BM * 128;            // 16 KB
constexpr int B_STAGE = BN * 128;            // 32 KB
constexpr int STAGES = 4;
constexpr int THREADS = 192;
constexpr int HIST_OFF = KCH * A_CHUNK + STAGES * B_STAGE;          // 4 epilogue warps x 256 bins
constexpr int BAR_OFF = HIST_OFF + 4 * 256 * 4;
constexpr int SMEM = BAR_OFF + 256 + 1024;
static_assert(SMEM <= 232448, "shared memory");
constexpr int MAX_K = 256, MAX_EXCL = 64;
constexpr int FP32_UC = 2048, FP32_NC = 16384;                    // FP32 mode: users x news per score block
constexpr int MERGE_THREADS = 256;
constexpr int MAX_SPLITS = 1024;

// order-preserving key: larger score -> larger key (-inf -> 0x007FFFFF); key 0 marks an excluded entry in the merge.
// -0 and +0 are one score (the tie rule then orders them by row).
__device__ __forceinline__ uint32_t score_key(float s) {
  const uint32_t u = __float_as_uint(s == 0.f ? 0.f : s);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key_score(uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k);
}
__device__ __forceinline__ uint32_t lanemask_lt() {
  uint32_t m;
  asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
  return m;
}

// Digit search of one radix-select pass: hist[256] holds the counts of the candidates matching the current prefix;
// returns the digit d holding the need-th largest candidate and sets `above` to the count in digits > d.  Whole warp.
__device__ __forceinline__ int radix_digit(const uint32_t* hist, int need, int& above, int lane) {
  int c[8], tot = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    c[j] = (int)hist[255 - 8 * lane - j];      // lane 0 owns the highest bins
    tot += c[j];
  }
  int incl = tot;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  const int excl = incl - tot;
  const uint32_t bl = __ballot_sync(0xffffffffu, excl < need && need <= incl);
  const int src = __ffs(bl) - 1;
  int digit = 0, ab = 0;
  if (lane == src) {
    int a = excl;
    bool found = false;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (!found && a + c[j] >= need) {
        digit = 255 - 8 * lane - j;
        ab = a;
        found = true;
      }
      a += c[j];
    }
  }
  above = __shfl_sync(0xffffffffu, ab, src);
  return __shfl_sync(0xffffffffu, digit, src);
}

// Whole warp: keep the kp best of the n > kp entries of one list (stable), return the kp-th largest key.  The list is
// read once into registers (entry 32 j + lane in slot j); the radix passes and the compaction work from there.
constexpr int CJ = 21;                       // register slots per lane: list_cap(MAX_K + MAX_EXCL) / 32
__device__ __noinline__ uint32_t warp_compact(uint32_t* keys, int32_t* rows, int n, int kp, uint32_t* hist, int lane) {
  uint32_t kr[CJ];
  int32_t rr[CJ];
#pragma unroll
  for (int j = 0; j < CJ; ++j) {
    const int i = 32 * j + lane;
    kr[j] = i < n ? keys[i] : 0u;
    rr[j] = i < n ? rows[i] : 0;
  }
  uint32_t prefix = 0, mask = 0;
  int need = kp;
#pragma unroll 1
  for (int shift = 24; shift >= 0; shift -= 8) {
    for (int b = lane; b < 256; b += 32) hist[b] = 0;
    __syncwarp();
#pragma unroll
    for (int j = 0; j < CJ; ++j)
      if (32 * j + lane < n && (kr[j] & mask) == prefix) atomicAdd(&hist[(kr[j] >> shift) & 255u], 1u);
    __syncwarp();
    int above;
    const int d = radix_digit(hist, need, above, lane);
    need -= above;
    prefix |= (uint32_t)d << shift;
    mask |= 255u << shift;
    __syncwarp();
  }
  // prefix = the kp-th largest key; keep every larger entry and the first `need` entries equal to it, in list order
  int out = 0, eq_seen = 0;
#pragma unroll
  for (int j = 0; j < CJ; ++j) {
    const bool in = 32 * j + lane < n;
    const bool eq = in && kr[j] == prefix;
    const uint32_t be = __ballot_sync(0xffffffffu, eq);
    const bool keep = (in && kr[j] > prefix) || (eq && eq_seen + __popc(be & lanemask_lt()) < need);
    const uint32_t bk = __ballot_sync(0xffffffffu, keep);
    if (keep) {
      const int p = out + __popc(bk & lanemask_lt());
      keys[p] = kr[j];
      rows[p] = rr[j];
    }
    out += __popc(bk);
    eq_seen += __popc(be);
  }
  __syncwarp();
  return prefix;
}

// One row's selection state; `list` is the element offset of its (row, split) list.
struct Sel {
  int64_t list;
  int cnt;
  uint32_t thr;
  bool full;      // false until the first compaction: every non-NaN score is taken
};

// Whole warp, converged: offer 16 consecutive scores of news rows n0 + j, which load(v) fetches (rows >= n_lim and
// inactive lanes are skipped).  The fused epilogue and the FP32 selection kernel both call this.  The lists are made
// room for before the scores are loaded, so no score stays live across a compaction.
template <class Load>
__device__ __forceinline__ void select_push16(Load load, int n0, int n_lim, bool active, Sel& st, uint32_t* keys,
                                              int32_t* rows, int kp, int cap, uint32_t* hist, int lane) {
  uint32_t need = __ballot_sync(0xffffffffu, st.cnt > cap - 16);
  while (need) {
    const int src = __ffs(need) - 1;
    need &= need - 1;
    const int64_t base = __shfl_sync(0xffffffffu, st.list, src);
    const int n = __shfl_sync(0xffffffffu, st.cnt, src);
    const uint32_t t = warp_compact(keys + base, rows + base, n, kp, hist, lane);
    if (lane == src) {
      st.cnt = kp;
      st.thr = t;
      st.full = true;
    }
  }
  float v[16];
  load(v);
  float vmax = v[0];               // fmaxf skips NaN; a chunk whose best score is not above the threshold adds nothing
#pragma unroll
  for (int j = 1; j < 16; ++j) vmax = fmaxf(vmax, v[j]);
  if (active && (!st.full || score_key(vmax) > st.thr)) {
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const float s = v[j];
      const uint32_t k = score_key(s);
      if (n0 + j < n_lim && s == s && (!st.full || k > st.thr)) {
        keys[st.list + st.cnt] = k;
        rows[st.list + st.cnt] = n0 + j;
        ++st.cnt;
      }
    }
  }
}

// Whole warp, converged, after a row's last scores: compact every list still longer than kp (less for the merge to read).
__device__ __forceinline__ void select_finish(Sel& st, uint32_t* keys, int32_t* rows, int kp, uint32_t* hist, int lane) {
  uint32_t need = __ballot_sync(0xffffffffu, st.cnt > kp);
  while (need) {
    const int src = __ffs(need) - 1;
    need &= need - 1;
    const int64_t base = __shfl_sync(0xffffffffu, st.list, src);
    const int n = __shfl_sync(0xffffffffu, st.cnt, src);
    warp_compact(keys + base, rows + base, n, kp, hist, lane);
    if (lane == src) st.cnt = kp;
  }
}

// ---- tensor mode ------------------------------------------------------------------------------------------------
// users fp32 [U, 300] -> fp16 [U_pad, 320], zero columns 300..319 (they meet the table's 1.0 bias column) and zero rows
__global__ void __launch_bounds__(256) users_to_f16_kernel(const float* __restrict__ u, int64_t U, int64_t U_pad,
                                                           __half* __restrict__ out) {
  const int64_t total = U_pad * (LD16 / 2);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / (LD16 / 2);
    const int c = 2 * (int)(i - r * (LD16 / 2));
    float a = 0.f, b = 0.f;
    if (r < U && c < D) {
      a = u[r * D + c];
      b = u[r * D + c + 1];
    }
    reinterpret_cast<__half2*>(out)[i] = __floats2half2_rn(a, b);
  }
}

__device__ __forceinline__ void tma_load_2d(uint32_t dst_smem, const CUtensorMap* tmap, int c0, int c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
      ::"r"(dst_smem), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(c0), "r"(c1), "r"(bar)
      : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("{ .reg .b64 st; mbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1; }" ::"r"(bar), "r"(bytes)
               : "memory");
}

// Work item w (the host's split rule, restated by tests/test_topk.py): user block w / splits, split w % splits owning
// news tiles [split * tps, min(n_tiles, (split + 1) * tps)); CTA b takes items b, b + gridDim.x, ...
__global__ void __launch_bounds__(THREADS, 1)
topk_score_kernel(const __grid_constant__ CUtensorMap tmap_u, const __grid_constant__ CUtensorMap tmap_t, int64_t U,
                  int n_news, int splits, int tps, uint32_t b_tx_bytes, uint32_t* __restrict__ lkeys,
                  int32_t* __restrict__ lrows, int32_t* __restrict__ counts, int kp, int cap) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* base_ptr = smem_raw + (base - raw);
  const uint32_t a_smem = base, b_smem = base + KCH * A_CHUNK;
  const uint32_t bars = base + BAR_OFF;
  const uint32_t full_bar = bars;                       // [STAGES]
  const uint32_t empty_bar = bars + 8 * STAGES;         // [STAGES]
  const uint32_t tfull_bar = bars + 16 * STAGES;        // [2]
  const uint32_t tempty_bar = tfull_bar + 16;           // [2]
  const uint32_t afull_bar = tempty_bar + 16;
  const uint32_t aempty_bar = afull_bar + 8;
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(base_ptr + BAR_OFF + 16 * STAGES + 64);

  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int n_tiles = (n_news + BN - 1) / BN;
  const int64_t items = ((U + BM - 1) / BM) * splits;
  const int64_t my_items = (int64_t)blockIdx.x < items ? (items - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  auto tile_range = [&](int64_t w, int& t0, int& t1) {
    t0 = (int)(w % splits) * tps;
    t1 = t0 + tps < n_tiles ? t0 + tps : n_tiles;
  };

  if (tid == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar + 8 * s, 1);
      mbar_init(empty_bar + 8 * s, 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar + 8 * a, 1);
      mbar_init(tempty_bar + 8 * a, 4);
    }
    mbar_init(afull_bar, 1);
    mbar_init(aempty_bar, 1);
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc(smem_u32((const void*)tmem_ptr_smem), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp == 0) {
    // ------------------------------ TMA producer ------------------------------
    if (lane == 0) {
      uint32_t it = 0;
      for (int64_t i = 0; i < my_items; ++i) {
        const int64_t w = blockIdx.x + i * gridDim.x;
        const int m0 = (int)(w / splits) * BM;
        int t0, t1;
        tile_range(w, t0, t1);
        mbar_wait(aempty_bar, ((uint32_t)i & 1u) ^ 1u);          // the previous item's MMAs have read the users
        mbar_expect_tx(afull_bar, KCH * A_CHUNK);
        for (int kc = 0; kc < KCH; ++kc) tma_load_2d(a_smem + kc * A_CHUNK, &tmap_u, kc * 64, m0, afull_bar);
        for (int t = t0; t < t1; ++t)
          for (int kc = 0; kc < KCH; ++kc, ++it) {
            const int s = it % STAGES;
            const uint32_t ph = (it / STAGES) & 1;
            mbar_wait(empty_bar + 8 * s, ph ^ 1);
            mbar_expect_tx(full_bar + 8 * s, b_tx_bytes);
            tma_load_2d(b_smem + s * B_STAGE, &tmap_t, kc * 64, t * BN, full_bar + 8 * s);
          }
      }
    }
  } else if (warp == 1) {
    // ------------------------------ MMA issuer (converged warp, predicated issue) ------------------------------
    const uint32_t el = elect_one_u32();
    const uint64_t desc0 = umma_desc_k_sw128(0);
    uint32_t it = 0, tile_it = 0;
    for (int64_t i = 0; i < my_items; ++i) {
      const int64_t w = blockIdx.x + i * gridDim.x;
      int t0, t1;
      tile_range(w, t0, t1);
      mbar_wait(afull_bar, (uint32_t)i & 1u);
      tc_fence_after();
      for (int t = t0; t < t1; ++t, ++tile_it) {
        int n_valid = n_news - t * BN;
        if (n_valid > BN) n_valid = BN;
        const uint32_t idesc = umma_idesc_f16(BM, (n_valid + 15) & ~15);
        const uint32_t as = tile_it & 1;
        mbar_wait(tempty_bar + 8 * as, ((tile_it >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + as * BN;
        for (int kc = 0; kc < KCH; ++kc, ++it) {
          const int s = it % STAGES;
          const uint32_t ph = (it / STAGES) & 1;
          mbar_wait(full_bar + 8 * s, ph);
          tc_fence_after();
          const uint32_t sa = (a_smem + kc * A_CHUNK) >> 4;
          const uint32_t sb = (b_smem + s * B_STAGE) >> 4;
#pragma unroll
          for (int ks = 0; ks < 4; ++ks)
            umma_f16_ss_p(d_tmem, desc0 | (uint64_t)((sa + 2 * ks) & 0x3FFF), desc0 | (uint64_t)((sb + 2 * ks) & 0x3FFF),
                          idesc, (kc || ks) ? 1u : 0u, el);
          umma_commit_p(empty_bar + 8 * s, el);
        }
        umma_commit_p(tfull_bar + 8 * as, el);
      }
      umma_commit_p(aempty_bar, el);
    }
  } else {
    // ------------------------------ selection epilogue (warps 2..5) ------------------------------
    const int q = warp & 3;                       // TMEM lane quarter this warp may access
    uint32_t* hist = reinterpret_cast<uint32_t*>(base_ptr + HIST_OFF) + (warp - 2) * 256;
    uint32_t tile_it = 0;
    for (int64_t i = 0; i < my_items; ++i) {
      const int64_t w = blockIdx.x + i * gridDim.x;
      const int64_t m = (w / splits) * BM + q * 32 + lane;
      const int sp = (int)(w % splits);
      const bool active = m < U;
      int t0, t1;
      tile_range(w, t0, t1);
      Sel st{(m * splits + sp) * (int64_t)cap, 0, 0u, false};
      for (int t = t0; t < t1; ++t, ++tile_it) {
        const int n0 = t * BN;
        int n_valid = n_news - n0;
        if (n_valid > BN) n_valid = BN;
        const uint32_t as = tile_it & 1;
        mbar_wait(tfull_bar + 8 * as, (tile_it >> 1) & 1);
        tc_fence_after();
        const uint32_t trow = tmem_base + as * BN + ((uint32_t)(q * 32) << 16);
        for (int col = 0; col < n_valid; col += 16) {
          select_push16([&](float* v) { tmem_ld16(trow + col, v); }, n0 + col, n_news, active, st, lkeys, lrows, kp, cap,
                        hist, lane);
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(tempty_bar + 8 * as);
      }
      select_finish(st, lkeys, lrows, kp, hist, lane);
      if (active) counts[m * splits + sp] = st.cnt;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// ---- FP32 mode: selection over a score block S [rows, ldc] (row r = user u0 + r, column c = news n0 + c) ----------
__global__ void __launch_bounds__(128) topk_select_block_kernel(const float* __restrict__ S, int64_t ldc, int rows_in,
                                                               int n_cols, int n0, int n_news, int split, int splits,
                                                               uint32_t* __restrict__ lkeys, int32_t* __restrict__ lrows,
                                                               int32_t* __restrict__ counts, int kp, int cap) {
  __shared__ uint32_t hist_all[4][256];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t r = (int64_t)blockIdx.x * 128 + threadIdx.x;
  const bool active = r < rows_in;
  Sel st{(r * splits + split) * (int64_t)cap, 0, 0u, false};
  for (int col = 0; col < n_cols; col += 16) {
    auto load = [&](float* v) {
      if (active) {
        const float4* p = reinterpret_cast<const float4*>(S + r * ldc + col);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 x = p[j];
          v[4 * j] = x.x; v[4 * j + 1] = x.y; v[4 * j + 2] = x.z; v[4 * j + 3] = x.w;
        }
      }
    };
    select_push16(load, n0 + col, n0 + n_cols < n_news ? n0 + n_cols : n_news, active, st, lkeys, lrows, kp, cap,
                  hist_all[warp], lane);
  }
  select_finish(st, lkeys, lrows, kp, hist_all[warp], lane);
  if (active) counts[r * splits + split] = st.cnt;
}

// ---- merge: one CTA per user --------------------------------------------------------------------------------------
// Lists of user u (local index u - u0): (u_local * splits + sp) * cap, counts[u_local * splits + sp].
__global__ void __launch_bounds__(MERGE_THREADS) topk_merge_kernel(uint32_t* __restrict__ lkeys, const int32_t* __restrict__ lrows,
                                                                  const int32_t* __restrict__ counts, int splits, int cap,
                                                                  int64_t u0, const int32_t* __restrict__ excl, int n_excl,
                                                                  int k, float* __restrict__ top_scores,
                                                                  int32_t* __restrict__ top_rows) {
  __shared__ int32_t s_excl[MAX_EXCL];
  __shared__ int32_t s_cnt[MAX_SPLITS];
  __shared__ uint32_t hist[256];
  __shared__ unsigned long long sel[MAX_K];
  __shared__ int s_valid, s_nsel, s_digit, s_above;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t ul = blockIdx.x;
  const int64_t u = u0 + ul;
  if (tid < n_excl) s_excl[tid] = excl[u * n_excl + tid];
  for (int s = tid; s < splits; s += MERGE_THREADS) s_cnt[s] = counts[ul * splits + s];
  if (tid == 0) { s_valid = 0; s_nsel = 0; }
  __syncthreads();
  uint32_t* keys = lkeys + ul * splits * (int64_t)cap;
  const int32_t* rows = lrows + ul * splits * (int64_t)cap;
  // composite 64-bit key: score key, then the smaller row first -- unique per user, so the top k is one set
  auto ck = [&](int64_t e) -> unsigned long long {
    return ((unsigned long long)keys[e] << 32) | (0xFFFFFFFFu - (uint32_t)rows[e]);
  };
  // pass 0: excluded entries get key 0; count the rest
  const int64_t n_slots = (int64_t)splits * cap;
  int valid = 0;
  for (int64_t e = tid; e < n_slots; e += MERGE_THREADS) {
    if (e % cap >= s_cnt[e / cap]) continue;
    const int32_t r = rows[e];
    bool ex = false;
    for (int j = 0; j < n_excl; ++j) ex |= s_excl[j] == r;
    if (ex) keys[e] = 0u;
    else ++valid;
  }
  valid = __reduce_add_sync(0xffffffffu, valid);
  if (lane == 0) atomicAdd(&s_valid, valid);
  __syncthreads();
  const int need_total = s_valid < k ? s_valid : k;
  unsigned long long prefix = 0ull, mask = 0ull;
  if (need_total < s_valid) {
    int need = need_total;
    for (int shift = 56; shift >= 0; shift -= 8) {
      hist[tid] = 0u;                      // MERGE_THREADS == 256 bins
      __syncthreads();
      for (int64_t e = tid; e < n_slots; e += MERGE_THREADS) {
        if (e % cap >= s_cnt[e / cap] || keys[e] == 0u) continue;
        const unsigned long long c = ck(e);
        if ((c & mask) == prefix) atomicAdd(&hist[(c >> shift) & 255u], 1u);
      }
      __syncthreads();
      if (warp == 0) {
        int above;
        const int d = radix_digit(hist, need, above, lane);
        if (lane == 0) { s_digit = d; s_above = above; }
      }
      __syncthreads();
      const int d = s_digit;
      need -= s_above;
      prefix |= (unsigned long long)d << shift;
      mask |= 255ull << shift;
      const bool done = (int)hist[d] == need;      // every candidate with this prefix is in
      __syncthreads();
      if (done) break;
    }
  }
  // collect the selected entries ((c & mask) >= prefix: exactly need_total of them), then rank by counting
  for (int64_t e = tid; e < n_slots; e += MERGE_THREADS) {
    if (e % cap >= s_cnt[e / cap] || keys[e] == 0u) continue;
    const unsigned long long c = ck(e);
    if ((c & mask) >= prefix) sel[atomicAdd(&s_nsel, 1)] = c;
  }
  __syncthreads();
  const int nsel = s_nsel;
  for (int t = tid; t < k; t += MERGE_THREADS) {
    if (t < nsel) {
      const unsigned long long c = sel[t];
      int rank = 0;
      for (int j = 0; j < nsel; ++j) rank += sel[j] > c ? 1 : 0;
      top_scores[u * k + rank] = key_score((uint32_t)(c >> 32));
      top_rows[u * k + rank] = (int32_t)(0xFFFFFFFFu - (uint32_t)c);
    } else {
      top_scores[u * k + t] = -INFINITY;
      top_rows[u * k + t] = -1;
    }
  }
}

// ---- host ----------------------------------------------------------------------------------------------------------
inline int list_cap(int kp) { return ((2 * kp + 31) / 32) * 32 + 32; }
static_assert(((2 * (MAX_K + MAX_EXCL) + 31) / 32) * 32 + 32 <= 32 * CJ, "list capacity exceeds the compaction registers");

struct Plan {
  int64_t U_pad;      // tensor mode: users rounded up to the 128-row block
  int n_tiles, splits, tps;
  int64_t list_users; // users whose lists live in the workspace at once
};

// Tensor mode: split the news tiles so that (user blocks x splits) fills the SMs -- one split when the user blocks alone
// do (each CTA walks the whole table), about one split per SM for a single user.  Every split owns >= 1 tile.
// FP32 mode: splits are the FP32_NC-row score blocks; lists for FP32_UC users at a time.
inline Plan make_plan(int64_t U, int64_t n_news, int mode, int sms) {
  Plan p;
  if (mode == NRMS_MODE_TF32) {
    p.U_pad = (U + BM - 1) / BM * BM;
    p.n_tiles = (int)((n_news + BN - 1) / BN);
    const int64_t ublocks = p.U_pad / BM;
    int64_t s = ublocks > 0 ? sms / ublocks : 1;
    if (s < 1) s = 1;
    if (s > p.n_tiles) s = p.n_tiles;
    p.tps = (int)((p.n_tiles + s - 1) / s);
    p.splits = (p.n_tiles + p.tps - 1) / p.tps;
    p.list_users = U;
  } else {
    p.U_pad = U;
    p.n_tiles = (int)((n_news + FP32_NC - 1) / FP32_NC);
    p.splits = p.n_tiles;
    p.tps = 1;
    p.list_users = U < FP32_UC ? U : FP32_UC;
  }
  return p;
}

struct Layout {
  size_t users16, scores, keys, rows, counts, total;
};
inline Layout make_layout(const Plan& p, int64_t n_news, int cap, int mode) {
  Layout l;
  size_t off = 0;
  auto take = [&](size_t bytes) { const size_t o = off; off += align_up(bytes, 256); return o; };
  const int64_t nc = n_news < FP32_NC ? n_news : FP32_NC;
  l.users16 = take(mode == NRMS_MODE_TF32 ? (size_t)p.U_pad * LD16 * 2 : 0);
  l.scores = take(mode == NRMS_MODE_FP32 ? (size_t)p.list_users * (size_t)((nc + 63) / 64 * 64) * 4 : 0);
  const size_t entries = (size_t)p.list_users * p.splits * cap;
  l.keys = take(entries * 4);
  l.rows = take(entries * 4);
  l.counts = take((size_t)p.list_users * p.splits * 4);
  l.total = off;
  return l;
}

}  // namespace topk
}  // namespace nrms

using namespace nrms;

extern "C" {

size_t nrms_topk_workspace_bytes(int64_t n_users, int64_t n_news, int k, int n_exclude, int mode) {
  if (n_users <= 0 || n_news <= 0 || k < 1 || k > topk::MAX_K || n_exclude < 0 || n_exclude > topk::MAX_EXCL ||
      (mode != NRMS_MODE_FP32 && mode != NRMS_MODE_TF32))
    return 0;
  const topk::Plan p = topk::make_plan(n_users, n_news, mode, num_sms());
  return topk::make_layout(p, n_news, topk::list_cap(k + n_exclude), mode).total;
}

int nrms_topk_news(const void* table, int64_t n_news, const float* user_vec, int64_t n_users,
                   const int32_t* exclude_rows, int n_exclude, int k, float* top_scores, int32_t* top_rows,
                   void* workspace, size_t workspace_bytes, int mode, void* stream) {
  using namespace topk;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  NRMS_CHECK_ARG(k >= 1 && k <= MAX_K, NRMS_E_UNSUPPORTED, "k = %d: the selection keeps 1 <= k <= %d rows", k, MAX_K);
  NRMS_CHECK_ARG(n_exclude <= MAX_EXCL, NRMS_E_UNSUPPORTED, "n_exclude = %d: at most %d exclusions per user", n_exclude,
                 MAX_EXCL);
  NRMS_CHECK_ARG(n_exclude >= 0 && n_users >= 0 && n_news > 0 && n_news < (1ll << 31), NRMS_E_INVALID, "bad sizes");
  NRMS_CHECK_ARG(mode == NRMS_MODE_FP32 || mode == NRMS_MODE_TF32, NRMS_E_INVALID, "unknown mode %d", mode);
  NRMS_CHECK_ARG(table && user_vec && top_scores && top_rows && workspace, NRMS_E_INVALID, "null pointer");
  NRMS_CHECK_ARG(n_exclude == 0 || exclude_rows, NRMS_E_INVALID, "null exclude_rows with n_exclude = %d", n_exclude);
  NRMS_CHECK_ARG(aligned16(table) && aligned16(user_vec) && (reinterpret_cast<uintptr_t>(workspace) & 255) == 0 &&
                     (reinterpret_cast<uintptr_t>(top_scores) & 3) == 0 && (reinterpret_cast<uintptr_t>(top_rows) & 3) == 0 &&
                     (reinterpret_cast<uintptr_t>(exclude_rows) & 3) == 0,
                 NRMS_E_INVALID, "misaligned pointer (table / user_vec 16 bytes, workspace 256 bytes)");
  if (n_users == 0) return NRMS_OK;
  const int ne = exclude_rows ? n_exclude : 0;
  const int kp = k + ne, cap = list_cap(kp);
  const int sms = num_sms();
  const Plan p = make_plan(n_users, n_news, mode, sms);
  NRMS_CHECK_ARG(p.splits <= MAX_SPLITS, NRMS_E_UNSUPPORTED, "table too large (%d splits)", p.splits);
  const Layout l = make_layout(p, n_news, cap, mode);
  NRMS_CHECK_ARG(workspace_bytes >= l.total, NRMS_E_WORKSPACE, "workspace too small: need %zu bytes", l.total);
  char* ws = reinterpret_cast<char*>(workspace);
  uint32_t* lkeys = reinterpret_cast<uint32_t*>(ws + l.keys);
  int32_t* lrows = reinterpret_cast<int32_t*>(ws + l.rows);
  int32_t* counts = reinterpret_cast<int32_t*>(ws + l.counts);

  if (mode == NRMS_MODE_TF32) {
    NRMS_CHECK_ARG(p.U_pad < (1ll << 31), NRMS_E_UNSUPPORTED, "too many users for one tensor map");
    void* users16 = ws + l.users16;
    {
      const int64_t total = p.U_pad * (LD16 / 2);
      int64_t gb = (total + 255) / 256;
      if (gb > (int64_t)sms * 16) gb = (int64_t)sms * 16;
      users_to_f16_kernel<<<(unsigned)gb, 256, 0, st>>>(user_vec, n_users, p.U_pad, reinterpret_cast<__half*>(users16));
      NRMS_LAUNCH_CHECK("topk users_to_f16_kernel");
    }
    alignas(64) CUtensorMap tu, tt;
    if (int rc = make_tmap_k_major_f16(&tu, users16, p.U_pad, LD16, LD16, BM)) return rc;
    const int box_t = n_news < BN ? (int)n_news : BN;
    if (int rc = make_tmap_k_major_f16(&tt, table, n_news, LD16, LD16, box_t)) return rc;
    static bool cfg[64] = {false};
    if (cudaError_t e = set_max_dynamic_smem(topk_score_kernel, SMEM, cfg)) return cuda_fail(e, "topk_score_kernel attr");
    const int64_t items = (p.U_pad / BM) * p.splits;
    const int grid = items < sms ? (int)items : sms;
    topk_score_kernel<<<grid, THREADS, SMEM, st>>>(tu, tt, n_users, (int)n_news, p.splits, p.tps, (uint32_t)box_t * 128,
                                                   lkeys, lrows, counts, kp, cap);
    NRMS_LAUNCH_CHECK("topk_score_kernel");
    NRMS_CHECK_ARG(n_users < (1ll << 31), NRMS_E_UNSUPPORTED, "too many users for one merge grid");
    topk_merge_kernel<<<(unsigned)n_users, MERGE_THREADS, 0, st>>>(lkeys, lrows, counts, p.splits, cap, 0, exclude_rows, ne,
                                                                   k, top_scores, top_rows);
    NRMS_LAUNCH_CHECK("topk_merge_kernel");
    return NRMS_OK;
  }

  // FP32: for each block of users, score blocks of FP32_NC news rows with the CUDA-core sgemm, select, then merge
  const float* table32 = reinterpret_cast<const float*>(table);
  float* S = reinterpret_cast<float*>(ws + l.scores);
  const int64_t nc_max = n_news < FP32_NC ? n_news : FP32_NC;
  const int64_t ldc = (nc_max + 63) / 64 * 64;
  for (int64_t u0 = 0; u0 < n_users; u0 += p.list_users) {
    const int64_t un = n_users - u0 < p.list_users ? n_users - u0 : p.list_users;
    for (int c = 0; c < p.splits; ++c) {
      const int64_t n0 = (int64_t)c * FP32_NC;
      const int nn = (int)(n_news - n0 < FP32_NC ? n_news - n0 : FP32_NC);
      NRMS_CUDA((sgemm_launch<0, 0, EPI_STORE>(user_vec + u0 * D, D, table32 + n0 * D, D, nullptr, S, ldc, un, nn, D, 1, st)));
      topk_select_block_kernel<<<(unsigned)((un + 127) / 128), 128, 0, st>>>(S, ldc, (int)un, nn, (int)n0, (int)n_news, c,
                                                                             p.splits, lkeys, lrows, counts, kp, cap);
      NRMS_LAUNCH_CHECK("topk_select_block_kernel");
    }
    topk_merge_kernel<<<(unsigned)un, MERGE_THREADS, 0, st>>>(lkeys, lrows, counts, p.splits, cap, u0, exclude_rows, ne, k,
                                                              top_scores, top_rows);
    NRMS_LAUNCH_CHECK("topk_merge_kernel");
  }
  return NRMS_OK;
}

}  // extern "C"
