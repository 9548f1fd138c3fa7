// Click predictor (dense + CSR), cross-entropy(label 0), fused Adam/AdamW, row gather,
// ranking metrics, and the error plumbing of the C-ABI.
#include <cuda_fp16.h>
#include "common.cuh"
#include "encoder_kernels.cuh"
#include <math.h>
#include <atomic>

namespace nrms {
int pack_rows16(const float* src, int64_t n_rows, void* src16, cudaStream_t st);   // pack.cu

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

static std::atomic<long long> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

int cuda_fail(cudaError_t e, const char* what) {
  set_error("CUDA error in %s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
  return NRMS_E_CUDA;
}

// ---- a8: scores[b,c] = cand[b,c,:] . user[b,:]  (one warp per (b,c)) -----------------------
__global__ void __launch_bounds__(256)
score_fwd_kernel(const float* __restrict__ cand, const float* __restrict__ user, int64_t BC, int C, int X,
                 float* __restrict__ scores) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  const int X4 = X >> 2;
  for (int64_t bc = warp; bc < BC; bc += nwarps) {
    const float4* cp = reinterpret_cast<const float4*>(cand + bc * X);
    const float4* up = reinterpret_cast<const float4*>(user + (bc / C) * X);
    float acc = 0.f;
    for (int l = lane; l < X4; l += 32) {
      float4 a = cp[l], u = up[l];
      acc = fmaf(a.x, u.x, acc); acc = fmaf(a.y, u.y, acc); acc = fmaf(a.z, u.z, acc); acc = fmaf(a.w, u.w, acc);
    }
    acc = warp_sum(acc);
    if (lane == 0) scores[bc] = acc;
  }
}

// d_cand[b,c,:] = d_s[b,c] * user[b,:] ; d_user[b,:] = sum_c d_s[b,c] * cand[b,c,:]   (block per b)
__global__ void __launch_bounds__(128)
score_bwd_kernel(const float* __restrict__ d_scores, const float* __restrict__ cand, const float* __restrict__ user,
                 int C, int X, float* __restrict__ d_cand, float* __restrict__ d_user) {
  const int64_t b = blockIdx.x;
  for (int x = threadIdx.x; x < X; x += blockDim.x) {
    const float u = user[b * X + x];
    float acc = 0.f;
    for (int c = 0; c < C; ++c) {
      const float ds = d_scores[b * C + c];
      d_cand[(b * C + c) * X + x] = ds * u;
      acc = fmaf(ds, cand[(b * C + c) * X + x], acc);
    }
    d_user[b * X + x] = acc;
  }
}

// ---- evaluate scoring on CSR impressions: warp per impression, 8 lanes per candidate --------
// Rows of DVEC float4 (300 wide: DVEC = 75; LSTUR's 900-wide vectors: 225).  Up to 80 float4 per row, the user vector
// lives in registers (10 float4 per lane) and each 8-lane group streams one row with coalesced float4 loads and reduces
// with 3 shuffles.  Wider rows are walked in chunks of 80 float4, the user chunk reloaded next to the row chunk.
template <int DVEC>
__global__ void __launch_bounds__(256)
score_csr_kernel(const float* __restrict__ table, const int32_t* __restrict__ cand_rows,
                 const int64_t* __restrict__ offsets, const float* __restrict__ user_vec, int64_t n_imp,
                 float* __restrict__ scores) {
  constexpr int NCH = (DVEC + 79) / 80;
  const int lane = threadIdx.x & 31;
  const int g = lane & 7, grp = lane >> 3;
  const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t imp = warp; imp < n_imp; imp += nwarps) {
    const float4* up = reinterpret_cast<const float4*>(user_vec + imp * 4 * DVEC);
    float4 u[10];
    if (NCH == 1) {
#pragma unroll
      for (int k = 0; k < 10; ++k) {
        const int idx = g + 8 * k;
        u[k] = (idx < DVEC) ? __ldg(up + idx) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
    const int64_t beg = offsets[imp], end = offsets[imp + 1];
    for (int64_t c0 = beg; c0 < end; c0 += 4) {
      const int64_t c = c0 + grp;
      float acc = 0.f;
      if (c < end) {
        const float4* rp = reinterpret_cast<const float4*>(table + (int64_t)cand_rows[c] * 4 * DVEC);
        for (int ch = 0; ch < NCH; ++ch) {
          float4 v[10];
#pragma unroll
          for (int k = 0; k < 10; ++k) {
            const int idx = ch * 80 + g + 8 * k;
            v[k] = (idx < DVEC) ? __ldg(rp + idx) : make_float4(0.f, 0.f, 0.f, 0.f);
            if (NCH > 1) u[k] = (idx < DVEC) ? __ldg(up + idx) : make_float4(0.f, 0.f, 0.f, 0.f);
          }
#pragma unroll
          for (int k = 0; k < 10; ++k) {
            acc = fmaf(v[k].x, u[k].x, acc); acc = fmaf(v[k].y, u[k].y, acc);
            acc = fmaf(v[k].z, u[k].z, acc); acc = fmaf(v[k].w, u[k].w, acc);
          }
        }
      }
      acc += __shfl_xor_sync(0xffffffffu, acc, 4);
      acc += __shfl_xor_sync(0xffffffffu, acc, 2);
      acc += __shfl_xor_sync(0xffffffffu, acc, 1);
      if (g == 0 && c < end) scores[c] = acc;
    }
  }
}

// Tensor-mode variant: the candidate rows come from an fp16 copy of the news-vector table ([rows][320] halfs, the
// same layout the user encoder gathers from: values 0..299, 1.0 at 300, zeros after), fp32 accumulation.  Half the
// bytes per candidate (640 B); the 42 MB table stays L2-resident.  8 lanes per row, 5 x 16 bytes per lane.
__global__ void __launch_bounds__(256)
score_csr_f16_kernel(const __half* __restrict__ table16, const int32_t* __restrict__ cand_rows,
                     const int64_t* __restrict__ offsets, const float* __restrict__ user_vec, int64_t n_imp,
                     float* __restrict__ scores) {
  const int lane = threadIdx.x & 31;
  const int g = lane & 7, grp = lane >> 3;
  const int64_t warp = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int64_t nwarps = (int64_t)gridDim.x * (blockDim.x >> 5);
  for (int64_t imp = warp; imp < n_imp; imp += nwarps) {
    // lane g owns the 8-element chunks g, g+8, ..., g+32 of the 320-wide row (chunks 37.5.. are the 1.0 / zero tail)
    const float4* up = reinterpret_cast<const float4*>(user_vec + imp * D);
    float4 u[5][2];
#pragma unroll
    for (int k = 0; k < 5; ++k) {
      const int ch = g + 8 * k;                 // 8 floats = 2 float4 at 2*ch, 2*ch+1 (valid below 75)
      u[k][0] = (2 * ch < DV4) ? __ldg(up + 2 * ch) : make_float4(0.f, 0.f, 0.f, 0.f);
      u[k][1] = (2 * ch + 1 < DV4) ? __ldg(up + 2 * ch + 1) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    const int64_t beg = offsets[imp], end = offsets[imp + 1];
    for (int64_t c0 = beg; c0 < end; c0 += 4) {
      const int64_t c = c0 + grp;
      float acc = 0.f;
      if (c < end) {
        const uint4* rp = reinterpret_cast<const uint4*>(table16 + (int64_t)cand_rows[c] * 320);
        uint4 v[5];
#pragma unroll
        for (int k = 0; k < 5; ++k) v[k] = __ldg(rp + g + 8 * k);
#pragma unroll
        for (int k = 0; k < 5; ++k) {
          const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&v[k].x));
          const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&v[k].y));
          const float2 cc = __half22float2(*reinterpret_cast<const __half2*>(&v[k].z));
          const float2 d = __half22float2(*reinterpret_cast<const __half2*>(&v[k].w));
          acc = fmaf(a.x, u[k][0].x, acc); acc = fmaf(a.y, u[k][0].y, acc);
          acc = fmaf(b.x, u[k][0].z, acc); acc = fmaf(b.y, u[k][0].w, acc);
          acc = fmaf(cc.x, u[k][1].x, acc); acc = fmaf(cc.y, u[k][1].y, acc);
          acc = fmaf(d.x, u[k][1].z, acc); acc = fmaf(d.y, u[k][1].w, acc);
        }
      }
      acc += __shfl_xor_sync(0xffffffffu, acc, 4);
      acc += __shfl_xor_sync(0xffffffffu, acc, 2);
      acc += __shfl_xor_sync(0xffffffffu, acc, 1);
      if (g == 0 && c < end) scores[c] = acc;
    }
  }
}

// ---- a11: CE with label 0, mean over batch (single block; B*C is tiny) ---------------------
__global__ void __launch_bounds__(256)
ce_loss_kernel(const float* __restrict__ logits, int64_t B, int C, float grad_scale, float* __restrict__ loss,
               float* __restrict__ d_logits) {
  __shared__ float red[8];
  float local = 0.f;
  const float invB = 1.f / (float)B;
  for (int64_t b = threadIdx.x; b < B; b += blockDim.x) {
    const float* row = logits + b * C;
    float m = row[0];
    for (int c = 1; c < C; ++c) m = fmaxf(m, row[c]);
    float sum = 0.f;
    for (int c = 0; c < C; ++c) sum += expf(row[c] - m);
    const float lse = logf(sum);
    local += -(row[0] - m - lse);
    if (d_logits) {
      for (int c = 0; c < C; ++c) {
        float pr = expf(row[c] - m - lse);
        d_logits[b * C + c] = (pr - (c == 0 ? 1.f : 0.f)) * invB * grad_scale;
      }
    }
  }
  local = warp_sum(local);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = local;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
    *loss = t * invB;
  }
}

// ---- a12: Adam / AdamW, 4 elements per thread ------------------------------------------------
__global__ void __launch_bounds__(256)
adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
            int64_t n, float lr, float b1, float b2, float eps, float wd, int decoupled, float step_size,
            float inv_bc2_sqrt, float grad_scale) {
  const int64_t n4 = n >> 2;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  auto upd = [&](float& pp, float gg, float& mm, float& vv) {
    gg *= grad_scale;
    if (wd != 0.f) {
      if (decoupled) pp *= (1.f - lr * wd);
      else gg = fmaf(wd, pp, gg);
    }
    mm = b1 * mm + (1.f - b1) * gg;
    vv = b2 * vv + (1.f - b2) * gg * gg;
    const float denom = sqrtf(vv) * inv_bc2_sqrt + eps;
    pp -= step_size * (mm / denom);
  };
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 pp = reinterpret_cast<float4*>(p)[i];
    float4 gg = reinterpret_cast<const float4*>(g)[i];
    float4 mm = reinterpret_cast<float4*>(m)[i];
    float4 vv = reinterpret_cast<float4*>(v)[i];
    upd(pp.x, gg.x, mm.x, vv.x); upd(pp.y, gg.y, mm.y, vv.y);
    upd(pp.z, gg.z, mm.z, vv.z); upd(pp.w, gg.w, mm.w, vv.w);
    reinterpret_cast<float4*>(p)[i] = pp;
    reinterpret_cast<float4*>(m)[i] = mm;
    reinterpret_cast<float4*>(v)[i] = vv;
  }
  for (int64_t i = (n4 << 2) + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    float pp = p[i], mm = m[i], vv = v[i];
    upd(pp, g[i], mm, vv);
    p[i] = pp; m[i] = mm; v[i] = vv;
  }
}

// ---- a14: ranking metrics, one warp per impression --------------------------------------------
// order = descending score, exact ties by descending index (reversed stable argsort; the
// reference's np.argsort()[::-1] leaves exact ties unspecified).  AUC counts ties 1/2 (sklearn).
constexpr int METRIC_CAP = 512;  // candidates staged in smem per warp; longer lists read global
// 1 / log2(rank + 1) for rank = 1..10 (only ranks <= 10 enter nDCG@5/@10): fp64 log2 is a long software sequence on
// a GPU whose fp64 pipe is vestigial, and it was called ~3 times per impression.  Values = 1.0 / numpy.log2(r + 1.0).
__constant__ double c_inv_log2[10] = {1.0, 0.6309297535714575, 0.5, 0.43067655807339306, 0.38685280723454163, 0.3562071871080222, 0.3333333333333333, 0.31546487678572877, 0.3010299956639812, 0.2890648263178879};
__global__ void __launch_bounds__(128)
rank_metrics_kernel(const float* __restrict__ scores, const int8_t* __restrict__ labels,
                    const int64_t* __restrict__ offsets, int64_t n_imp, double* __restrict__ per) {
  __shared__ float s_sc[4][METRIC_CAP];
  __shared__ int8_t s_lb[4][METRIC_CAP];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int64_t warp = (int64_t)blockIdx.x * 4 + wib;
  const int64_t nwarps = (int64_t)gridDim.x * 4;
  for (int64_t imp = warp; imp < n_imp; imp += nwarps) {
    const int64_t beg = offsets[imp];
    const int C = (int)(offsets[imp + 1] - beg);
    const float* sc = scores + beg;
    const int8_t* lb = labels + beg;
    const bool staged = C <= METRIC_CAP;
    __syncwarp();
    if (staged) {
      for (int j = lane; j < C; j += 32) { s_sc[wib][j] = sc[j]; s_lb[wib][j] = lb[j]; }
      __syncwarp();
      sc = s_sc[wib];
      lb = s_lb[wib];
    }
    int npos_l = 0;
    for (int j = lane; j < C; j += 32) npos_l += (lb[j] != 0);
    int npos = npos_l;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) npos += __shfl_xor_sync(0xffffffffu, npos, o);
    const int nneg = C - npos;
    // positives are few (~4 % of the candidates): the warp takes them one at a time and splits the O(C) rank
    // count over its lanes (all lanes end up with the same totals; no fp64 reduction needed)
    double auc = 0.0, mrr = 0.0, d5 = 0.0, d10 = 0.0;
    for (int i0 = 0; i0 < C; i0 += 32) {
      const int ii = i0 + lane;
      unsigned pos_mask = __ballot_sync(0xffffffffu, ii < C && lb[ii] != 0);
      while (pos_mask) {
        const int i = i0 + __ffs(pos_mask) - 1;
        pos_mask &= pos_mask - 1;
        const float si = sc[i];
        int above = 0, neg_below = 0, neg_tie = 0;
        for (int j = lane; j < C; j += 32) {
          const float sj = sc[j];
          const bool isneg = lb[j] == 0;
          above += (sj > si) || (sj == si && j > i);
          neg_below += isneg && (sj < si);
          neg_tie += isneg && (sj == si);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          above += __shfl_xor_sync(0xffffffffu, above, o);
          neg_below += __shfl_xor_sync(0xffffffffu, neg_below, o);
          neg_tie += __shfl_xor_sync(0xffffffffu, neg_tie, o);
        }
        const int rank = above + 1;
        auc += (double)neg_below + 0.5 * (double)neg_tie;
        mrr += 1.0 / (double)rank;
        if (rank <= 10) {
          const double dg = c_inv_log2[rank - 1];
          if (rank <= 5) d5 += dg;
          d10 += dg;
        }
      }
    }
    if (lane == 0) {
      double* o = per + imp * 4;
      if (npos == 0 || nneg == 0) {
        const double nan = __longlong_as_double(0x7ff8000000000000LL);
        o[0] = o[1] = o[2] = o[3] = nan;
      } else {
        double i5 = 0.0, i10 = 0.0;
        for (int r = 1; r <= 10 && r <= npos; ++r) {
          const double dg = c_inv_log2[r - 1];
          if (r <= 5) i5 += dg;
          i10 += dg;
        }
        o[0] = auc / ((double)npos * (double)nneg);
        o[1] = mrr / (double)npos;
        o[2] = d5 / i5;
        o[3] = d10 / i10;
      }
    }
  }
}

// nanmean numerators/denominators: one block, fixed-order tree reduction (deterministic)
__global__ void __launch_bounds__(1024)
metric_reduce_kernel(const double* __restrict__ per, int64_t n_imp, double* __restrict__ sums_counts) {
  __shared__ double red[8][32];
  double s[4] = {0, 0, 0, 0}, c[4] = {0, 0, 0, 0};
  for (int64_t i = threadIdx.x; i < n_imp; i += blockDim.x) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const double v = per[i * 4 + k];
      if (v == v) { s[k] += v; c[k] += 1.0; }
    }
  }
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 4; ++k) { s[k] = warp_sum_d(s[k]); c[k] = warp_sum_d(c[k]); }
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < 4; ++k) { red[k][w] = s[k]; red[4 + k][w] = c[k]; }
  }
  __syncthreads();
  if (w < 8) {
    double v = (lane < (int)(blockDim.x >> 5)) ? red[w][lane] : 0.0;
    v = warp_sum_d(v);
    if (lane == 0) sums_counts[w] = v;
  }
}

}  // namespace nrms

using namespace nrms;

extern "C" {

const char* nrms_last_error(void) { return g_err; }
int nrms_abi_version(void) { return 2; }
int64_t nrms_launch_count(void) { return (int64_t)g_launches.load(std::memory_order_relaxed); }

int nrms_score_fwd(const float* cand, const float* user, int64_t B, int C, int X, float* scores, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  NRMS_CHECK_ARG(B >= 0 && C > 0 && X > 0 && X % 4 == 0, NRMS_E_INVALID, "bad sizes (X must be a multiple of 4)");
  if (B == 0) return NRMS_OK;
  NRMS_CHECK_ARG(cand && user && scores && aligned16(cand) && aligned16(user), NRMS_E_INVALID, "null/misaligned pointer");
  const int64_t BC = B * C;
  int64_t gb = (BC + 7) / 8;
  if (gb > (int64_t)num_sms() * 16) gb = (int64_t)num_sms() * 16;
  score_fwd_kernel<<<(unsigned)gb, 256, 0, st>>>(cand, user, BC, C, X, scores);
  NRMS_LAUNCH_CHECK("score_fwd");
  return NRMS_OK;
}

int nrms_score_bwd(const float* d_scores, const float* cand, const float* user, int64_t B, int C, int X,
                   float* d_cand, float* d_user, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  NRMS_CHECK_ARG(B >= 0 && C > 0 && X > 0, NRMS_E_INVALID, "bad sizes");
  if (B == 0) return NRMS_OK;
  NRMS_CHECK_ARG(d_scores && cand && user && d_cand && d_user, NRMS_E_INVALID, "null pointer");
  NRMS_CHECK_ARG(B < (1ll << 31), NRMS_E_UNSUPPORTED, "B too large");
  score_bwd_kernel<<<(unsigned)B, 128, 0, st>>>(d_scores, cand, user, C, X, d_cand, d_user);
  NRMS_LAUNCH_CHECK("score_bwd");
  return NRMS_OK;
}

int nrms_score_csr_width(const float* table, const int32_t* cand_rows, const int64_t* offsets, const float* user_vec,
                         int64_t n_impressions, int width, float* scores, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  NRMS_CHECK_ARG(width == D || width == 3 * D, NRMS_E_UNSUPPORTED, "score width %d unsupported (300 or 900)", width);
  NRMS_CHECK_ARG(n_impressions >= 0, NRMS_E_INVALID, "bad sizes");
  if (n_impressions == 0) return NRMS_OK;
  NRMS_CHECK_ARG(table && cand_rows && offsets && user_vec && scores && aligned16(table) && aligned16(user_vec),
                 NRMS_E_INVALID, "null/misaligned pointer");
  int64_t gb = (n_impressions + 7) / 8;
  if (gb > (int64_t)num_sms() * 8) gb = (int64_t)num_sms() * 8;
  if (width == D)
    score_csr_kernel<DV4><<<(unsigned)gb, 256, 0, st>>>(table, cand_rows, offsets, user_vec, n_impressions, scores);
  else
    score_csr_kernel<3 * DV4><<<(unsigned)gb, 256, 0, st>>>(table, cand_rows, offsets, user_vec, n_impressions, scores);
  NRMS_LAUNCH_CHECK("score_csr");
  return NRMS_OK;
}

int nrms_score_csr(const float* table, const int32_t* cand_rows, const int64_t* offsets, const float* user_vec,
                   int64_t n_impressions, float* scores, void* stream) {
  return nrms_score_csr_width(table, cand_rows, offsets, user_vec, n_impressions, D, scores, stream);
}

int nrms_pack_rows_f16(const float* src, int64_t n_rows, void* dst16, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  NRMS_CHECK_ARG(n_rows >= 0, NRMS_E_INVALID, "bad sizes");
  NRMS_CHECK_ARG(src && dst16 && aligned16(src) && aligned16(dst16), NRMS_E_INVALID, "null/misaligned pointer");
  return pack_rows16(src, n_rows, dst16, st);
}

int nrms_score_csr_f16(const void* table16, const int32_t* cand_rows, const int64_t* offsets, const float* user_vec,
                       int64_t n_impressions, float* scores, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  NRMS_CHECK_ARG(n_impressions >= 0, NRMS_E_INVALID, "bad sizes");
  if (n_impressions == 0) return NRMS_OK;
  NRMS_CHECK_ARG(table16 && cand_rows && offsets && user_vec && scores && aligned16(table16) && aligned16(user_vec),
                 NRMS_E_INVALID, "null/misaligned pointer");
  int64_t gb = (n_impressions + 7) / 8;
  if (gb > (int64_t)num_sms() * 8) gb = (int64_t)num_sms() * 8;
  score_csr_f16_kernel<<<(unsigned)gb, 256, 0, st>>>(reinterpret_cast<const __half*>(table16), cand_rows, offsets,
                                                    user_vec, n_impressions, scores);
  NRMS_LAUNCH_CHECK("score_csr_f16");
  return NRMS_OK;
}

int nrms_ce_loss_fwd_bwd(const float* logits, int64_t B, int C, float grad_scale, float* loss, float* d_logits,
                         void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  NRMS_CHECK_ARG(B > 0 && C > 0, NRMS_E_INVALID, "bad sizes");
  NRMS_CHECK_ARG(logits && loss, NRMS_E_INVALID, "null pointer");
  ce_loss_kernel<<<1, 256, 0, st>>>(logits, B, C, grad_scale, loss, d_logits);
  NRMS_LAUNCH_CHECK("ce_loss");
  return NRMS_OK;
}

int nrms_adam_step(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
                   float eps, float weight_decay, int decoupled, int64_t step, float grad_scale, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  NRMS_CHECK_ARG(n >= 0 && step >= 1, NRMS_E_INVALID, "bad sizes (step is 1-based)");
  if (n == 0) return NRMS_OK;
  NRMS_CHECK_ARG(p && g && m && v && aligned16(p) && aligned16(g) && aligned16(m) && aligned16(v), NRMS_E_INVALID,
                 "null/misaligned pointer");
  const double bc1 = 1.0 - pow((double)beta1, (double)step);
  const double bc2 = 1.0 - pow((double)beta2, (double)step);
  const float step_size = (float)((double)lr / bc1);
  const float inv_bc2_sqrt = (float)(1.0 / sqrt(bc2));
  int64_t gb = ((n >> 2) + 255) / 256;
  if (gb > (int64_t)num_sms() * 16) gb = (int64_t)num_sms() * 16;
  if (gb < 1) gb = 1;
  adam_kernel<<<(unsigned)gb, 256, 0, st>>>(p, g, m, v, n, lr, beta1, beta2, eps, weight_decay, decoupled, step_size,
                                            inv_bc2_sqrt, grad_scale);
  NRMS_LAUNCH_CHECK("adam");
  return NRMS_OK;
}

int nrms_gather_rows(const float* src, const int64_t* rows, int64_t n, int width, float* dst, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  NRMS_CHECK_ARG(n >= 0 && width > 0 && width % 4 == 0, NRMS_E_INVALID, "bad sizes (width must be a multiple of 4)");
  if (n == 0) return NRMS_OK;
  NRMS_CHECK_ARG(src && rows && dst && aligned16(src) && aligned16(dst), NRMS_E_INVALID, "null/misaligned pointer");
  int64_t gb = (n + 7) / 8;
  if (gb > (int64_t)num_sms() * 16) gb = (int64_t)num_sms() * 16;
  gather_rows_kernel<int64_t><<<(unsigned)gb, 256, 0, st>>>(src, rows, n, width / 4, dst);
  NRMS_LAUNCH_CHECK("gather_rows");
  return NRMS_OK;
}

int nrms_rank_metrics(const float* scores, const int8_t* labels, const int64_t* offsets, int64_t n_impressions,
                      double* per_impression, double* sums_counts, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  NRMS_CHECK_ARG(n_impressions >= 0, NRMS_E_INVALID, "bad sizes");
  if (n_impressions == 0) {
    if (sums_counts) NRMS_CUDA(cudaMemsetAsync(sums_counts, 0, 8 * sizeof(double), st));
    return NRMS_OK;
  }
  NRMS_CHECK_ARG(per_impression != nullptr, NRMS_E_INVALID, "per_impression buffer [n,4] is required");
  if (n_impressions > 0) {
    NRMS_CHECK_ARG(scores && labels && offsets, NRMS_E_INVALID, "null pointer");
    int64_t gb = (n_impressions + 3) / 4;
    if (gb > (int64_t)num_sms() * 16) gb = (int64_t)num_sms() * 16;
    rank_metrics_kernel<<<(unsigned)gb, 128, 0, st>>>(scores, labels, offsets, n_impressions, per_impression);
    NRMS_LAUNCH_CHECK("rank_metrics");
  }
  if (sums_counts) {
    metric_reduce_kernel<<<1, 1024, 0, st>>>(per_impression, n_impressions, sums_counts);
    NRMS_LAUNCH_CHECK("metric_reduce");
  }
  return NRMS_OK;
}

}  // extern "C"
