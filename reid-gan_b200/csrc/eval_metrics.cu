// f3 (SURVEY.md 8f) -- evaluation metrics: clustercontrast/evaluators.py pairwise_distance :71-88 and
// clustercontrast/evaluation_metrics/ranking.py mean_ap :82-115, cmc :18-79.
//
// The reference argsorts every query row (n ~ 16k..82k gallery items) and then only looks at where the few
// positives (same id, allowed camera) landed.  Here no row is ever sorted: one CTA per query collects its positives
// (ordered compaction, so the list is deterministic), and for every positive p counts over the valid gallery items
//   le(p)  = #{ d <= d_p }                 -> precision denominator of average_precision_score (ties share a threshold)
//   pos(p) = #{ (d, index) < (d_p, p) }    -> its 0-based position in the sorted valid list (CMC)
// plus tp(p) = #{ positives with d <= d_p }.  AP = sum_p tp(p) / le(p) / P  (sklearn's uninterpolated AP).
#include "common.cuh"

namespace reid {

// ---- pairwise_distance: ||x||^2 + ||y||^2 - 2 x.y^T, fp32 ----------------------------------------------------
__global__ void __launch_bounds__(256) row_sqnorm_kernel(const float* __restrict__ x, int64_t n_rows, int64_t D,
                                                         float* __restrict__ out) {
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= n_rows) return;
  float s = 0.f;
  for (int64_t d = lane_id(); d < D; d += 32) {
    const float v = x[row * D + d];
    s = fmaf(v, v, s);
  }
  s = warp_sum(s);
  if (lane_id() == 0) out[row] = s;
}

constexpr int PT = 64, PK = 16;   // 64 x 64 output tile, 4 x 4 per thread, K step 16

__global__ void __launch_bounds__(256) pairwise_dist_kernel(const float* __restrict__ x, const float* __restrict__ y,
                                                            const float* __restrict__ xx, const float* __restrict__ yy,
                                                            int64_t m, int64_t n, int64_t D, float* __restrict__ out) {
  __shared__ float As[PK][PT + 1];
  __shared__ float Bs[PK][PT + 1];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int64_t r0 = (int64_t)blockIdx.y * PT, c0 = (int64_t)blockIdx.x * PT;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  for (int64_t k0 = 0; k0 < D; k0 += PK) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {                  // 64 rows x 16 k = 1024 elements per operand, 4 per thread
      const int lin = threadIdx.x + e * 256;
      const int rr = lin >> 4, kk = lin & 15;
      const int64_t kd = k0 + kk;
      As[kk][rr] = (r0 + rr < m && kd < D) ? x[(r0 + rr) * D + kd] : 0.f;
      Bs[kk][rr] = (c0 + rr < n && kd < D) ? y[(c0 + rr) * D + kd] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < PK; ++kk) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = As[kk][ty + 16 * i];
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = Bs[kk][tx + 16 * j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t r = r0 + ty + 16 * i;
    if (r >= m) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int64_t c = c0 + tx + 16 * j;
      // dist_m = (xx + yy), then addmm_(x, y^T, beta=1, alpha=-2)   (evaluators.py:84-86)
      if (c < n) out[r * n + c] = __fadd_rn(__fadd_rn(xx[r], yy[c]), __fmul_rn(-2.0f, acc[i][j]));
    }
  }
}

// ---- mean_ap / cmc ------------------------------------------------------------------------------------------------
constexpr int kPosCap = 2048;      // positives per query handled (a query with more is reported through has_pos = -1)
constexpr int kRankThreads = 256;

__global__ void __launch_bounds__(kRankThreads) rank_metrics_kernel(
    const float* __restrict__ dist, int64_t ld, const int64_t* __restrict__ q_ids, const int64_t* __restrict__ g_ids,
    const int64_t* __restrict__ q_cams, const int64_t* __restrict__ g_cams, int64_t n, int separate_camera_set, int topk,
    int first_match_break, double* __restrict__ ap_out, int32_t* __restrict__ has_pos, double* __restrict__ contrib) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  unsigned* s_valid = reinterpret_cast<unsigned*>(smem_raw);                       // [(n + 31) / 32] bit mask of valid items
  int32_t* s_pidx = reinterpret_cast<int32_t*>(s_valid + ((n + 31) >> 5));          // [kPosCap]
  float* s_pd = reinterpret_cast<float*>(s_pidx + kPosCap);                         // [kPosCap]
  int32_t* s_le = reinterpret_cast<int32_t*>(s_pd + kPosCap);                       // [kPosCap]
  int32_t* s_pos = s_le + kPosCap;                                                  // [kPosCap]
  int32_t* s_sorted = s_pos + kPosCap;                                              // [kPosCap]
  __shared__ int s_warp[kRankThreads / 32];
  __shared__ int s_base;
  const int64_t i = blockIdx.x;
  const int t = threadIdx.x, lane = t & 31, w = t >> 5;
  const float* d = dist + i * ld;
  const int64_t qid = q_ids[i], qcam = q_cams[i];
  if (t == 0) s_base = 0;
  __syncthreads();
  // phase 1: valid mask + ordered list of the positives
  for (int64_t base = 0; base < n; base += kRankThreads) {
    const int64_t j = base + t;
    bool valid = false, posv = false;
    if (j < n) {
      const int64_t gid = g_ids[j], gcam = g_cams[j];
      valid = (gid != qid) || (gcam != qcam);                      // ranking.py:47-48 / 108-109
      if (separate_camera_set) valid = valid && (gcam != qcam);    // :49-51
      posv = valid && gid == qid;
    }
    const unsigned vb = __ballot_sync(kFull, valid);
    if (lane == 0 && base + (int64_t)w * 32 < n) s_valid[(base >> 5) + w] = vb;
    const unsigned pb = __ballot_sync(kFull, posv);
    if (lane == 0) s_warp[w] = __popc(pb);
    __syncthreads();
    int before = s_base;
    for (int ww = 0; ww < w; ++ww) before += s_warp[ww];
    if (posv) {
      const int p = before + __popc(pb & ((1u << lane) - 1u));
      if (p < kPosCap) {
        s_pidx[p] = (int32_t)j;
        s_pd[p] = d[j];
      }
    }
    __syncthreads();
    if (t == 0) {
      int tot = 0;
      for (int ww = 0; ww < kRankThreads / 32; ++ww) tot += s_warp[ww];
      s_base += tot;
    }
    __syncthreads();
  }
  const int P = s_base;
  if (P == 0 || P > kPosCap) {
    if (t == 0) {
      has_pos[i] = P == 0 ? 0 : -1;
      ap_out[i] = 0.0;
    }
    return;
  }
  // phase 2: le / pos of every positive, eight positives per sweep of the row
  for (int p0 = 0; p0 < P; p0 += 8) {
    float pd[8];
    int32_t pi[8];
    int le[8], ps[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const bool ok = p0 + u < P;
      pd[u] = ok ? s_pd[p0 + u] : -INFINITY;
      pi[u] = ok ? s_pidx[p0 + u] : -1;
      le[u] = ps[u] = 0;
    }
    for (int64_t j = t; j < n; j += kRankThreads) {
      if (!((s_valid[j >> 5] >> (j & 31)) & 1u)) continue;
      const float dj = d[j];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        le[u] += dj <= pd[u];
        ps[u] += (dj < pd[u]) || (dj == pd[u] && (int32_t)j < pi[u]);
      }
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      le[u] = __reduce_add_sync(kFull, le[u]);
      ps[u] = __reduce_add_sync(kFull, ps[u]);
    }
    __syncthreads();
    if (t < 16) (t < 8 ? s_le : s_pos)[p0 + (t & 7)] = 0;          // 16 >= possible overrun inside the arrays: p0 + 7 < kPosCap + 8
    __syncthreads();
    if (lane == 0) {
#pragma unroll
      for (int u = 0; u < 8; ++u)
        if (p0 + u < P) {
          atomicAdd(&s_le[p0 + u], le[u]);
          atomicAdd(&s_pos[p0 + u], ps[u]);
        }
    }
    __syncthreads();
  }
  // phase 3: sort the positions (rank by counting: they are distinct), AP and the CMC contribution of this query
  for (int p = t; p < P; p += kRankThreads) {
    const int me = s_pos[p];
    int r = 0;
    for (int u = 0; u < P; ++u) r += s_pos[u] < me;
    s_sorted[r] = me;
  }
  __syncthreads();
  if (t == 0) {
    double ap = 0.0;
    for (int p = 0; p < P; ++p) {
      int tp = 0;
      const float dp = s_pd[p];
      for (int u = 0; u < P; ++u) tp += s_pd[u] <= dp;
      ap += (double)tp / (double)s_le[p];
    }
    ap_out[i] = ap / (double)P;
    has_pos[i] = 1;
    if (contrib) {
      double* c = contrib + i * (int64_t)topk;
      const double delta = 1.0 / (double)P;                        // ranking.py:69 (repeat == 1)
      for (int j = 0; j < P; ++j) {                                // :70-75
        const int k = s_sorted[j];
        if (k - j >= topk) break;
        if (first_match_break) {
          c[k - j] += 1.0;
          break;
        }
        c[k - j] += delta;
      }
    }
  }
}

// ret[k] = sum over the queries in order (the reference's sequential accumulation, ranking.py:72-75)
__global__ void cmc_reduce_kernel(const double* __restrict__ contrib, int64_t m, int topk, double* __restrict__ ret) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= topk) return;
  double s = 0.0;
  for (int64_t i = 0; i < m; ++i) s += contrib[i * topk + k];
  ret[k] = s;
}

}  // namespace reid

extern "C" {

int reid_pairwise_distance(const float* x, const float* y, int64_t m, int64_t n, int64_t D, float* scratch_norms,
                           float* out, void* stream) {
  using namespace reid;
  REID_CHECK_ARG(x && y && scratch_norms && out && m >= 1 && n >= 1 && D >= 1, "reid_pairwise_distance: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  float* xx = scratch_norms;
  float* yy = scratch_norms + m;
  row_sqnorm_kernel<<<(unsigned)((m + 7) / 8), 256, 0, st>>>(x, m, D, xx);
  REID_LAUNCH_CHECK();
  row_sqnorm_kernel<<<(unsigned)((n + 7) / 8), 256, 0, st>>>(y, n, D, yy);
  REID_LAUNCH_CHECK();
  pairwise_dist_kernel<<<dim3((unsigned)((n + PT - 1) / PT), (unsigned)((m + PT - 1) / PT)), 256, 0, st>>>(x, y, xx, yy, m, n, D,
                                                                                                         out);
  REID_LAUNCH_CHECK();
  return REID_OK;
}

size_t reid_rank_metrics_smem_bytes(int64_t n) {
  return (size_t)((n + 31) / 32) * 4 + (size_t)reid::kPosCap * 20;
}

int reid_rank_metrics(const float* dist, int64_t m, int64_t n, int64_t ld, const int64_t* q_ids, const int64_t* g_ids,
                      const int64_t* q_cams, const int64_t* g_cams, int separate_camera_set, int topk, int first_match_break,
                      double* ap_out, int32_t* has_pos, double* cmc_contrib, double* cmc_ret, void* stream) {
  using namespace reid;
  REID_CHECK_ARG(dist && q_ids && g_ids && q_cams && g_cams && ap_out && has_pos && m >= 1 && n >= 1 && ld >= n,
                 "reid_rank_metrics: bad arguments");
  REID_CHECK_ARG((cmc_contrib == nullptr) == (cmc_ret == nullptr) && (cmc_contrib == nullptr || topk >= 1),
                 "reid_rank_metrics: cmc buffers go together (topk >= 1)");
  const size_t smem = reid_rank_metrics_smem_bytes(n);
  REID_CHECK_ARG(smem <= 200 * 1024, "reid_rank_metrics: gallery of %lld items needs %zu B of shared memory", (long long)n, smem);
  cudaStream_t st = (cudaStream_t)stream;
  if (cmc_contrib) REID_CUDA(cudaMemsetAsync(cmc_contrib, 0, sizeof(double) * (size_t)m * (size_t)topk, st));
  REID_CUDA(cudaFuncSetAttribute(rank_metrics_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  rank_metrics_kernel<<<(unsigned)m, kRankThreads, smem, st>>>(dist, ld, q_ids, g_ids, q_cams, g_cams, n, separate_camera_set,
                                                              topk, first_match_break, ap_out, has_pos, cmc_contrib);
  REID_LAUNCH_CHECK();
  if (cmc_contrib) {
    cmc_reduce_kernel<<<(unsigned)((topk + 127) / 128), 128, 0, st>>>(cmc_contrib, m, topk, cmc_ret);
    REID_LAUNCH_CHECK();
  }
  return REID_OK;
}

int reid_cmc_reduce(const double* cmc_contrib, int64_t m, int topk, double* cmc_ret, void* stream) {
  using namespace reid;
  REID_CHECK_ARG(cmc_contrib && cmc_ret && m >= 1 && topk >= 1, "reid_cmc_reduce: bad arguments");
  cmc_reduce_kernel<<<(unsigned)((topk + 127) / 128), 128, 0, (cudaStream_t)stream>>>(cmc_contrib, m, topk, cmc_ret);
  REID_LAUNCH_CHECK();
  return REID_OK;
}
}
