// f2 from features -- the evaluation-time re-ranking (utils/rerank.py re_ranking :31-97) computed from the (Q+G) x D
// features instead of three dense distance matrices.  With orig(r, c) = pairwise(x_r, x_c)^2 over the union and
// colmax[c] = max_r orig(r, c), the dense path's dist[i, j] = orig(j, i) / colmax[i]: a row of dist is a row of orig
// times a constant.  So the neighbour lists are the squared-L2 kNN of the union (reid_knn_*), and what is specific
// here is colmax (a farthest-neighbour search), the weights of the expansion sets from gathered feature rows and the
// blend against the Q x G distance block.  No M x M matrix exists.
//
// Distance arithmetic of every kernel here: n_i = sum_d x_id^2 and x_i.x_j accumulated in fp64 in one fixed order
// (lane-strided over d, then a warp butterfly), sq(i, j) = fp32((n_i + n_j) - 2 x_i.x_j) computed in fp64, and
// orig = fp32(sq * sq) (np.power(original_dist, 2) of float32, :40).  sq(i, j) and sq(j, i) are the same bits.
#include <math.h>

#include "common.cuh"

namespace reid {

constexpr int kFcWarps = 4;
constexpr int kFcWinMax = 128;     // window members re-scored per row at most; a larger window un-certifies the row
constexpr int kFxRows = 8;         // query rows per CTA of the exact scan
constexpr int kFxThreads = 256;

// fp64 dot of two rows, the lane-strided order every kernel of this file uses; the full sum on every lane
__device__ __forceinline__ double warp_dot64(const float* __restrict__ a, const float* __restrict__ b, int64_t D, int lane) {
  double acc = 0.0;
  for (int64_t d = lane; d < D; d += 32) acc = fma((double)a[d], (double)b[d], acc);
  return warp_sum(acc);
}

__device__ __forceinline__ float pair_sq(double ni, double nj, double dot) { return (float)((ni + nj) - 2.0 * dot); }

// n[i] = sum_d x[i, d]^2 in fp64, one warp per row
__global__ void __launch_bounds__(256) rr_sqnorm64_kernel(const float* __restrict__ x, int64_t n_rows, int64_t D,
                                                          double* __restrict__ out) {
  const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= n_rows) return;
  const float* xr = x + row * D;
  const double s = warp_dot64(xr, xr, D, lane_id());
  if (lane_id() == 0) out[row] = s;
}

// |fp16-GEMM score - exact dot| bound of reid_knn_rescore (knn_rescore.cu reid_tc_err_bound)
__device__ __forceinline__ float fc_err_bound(float max_sqnorm) { return max_sqnorm * (1.02f / 1024.0f) + (1.0f / 16384.0f); }

// Certificate of the farthest row.  The candidate lists score a_j ~ -x_i.x_j (negated operand), |a_j - s_j| <= eps for
// s_j = -x_i.x_j, and every unlisted column scored <= bound.  With a_max the best listed score and norms in
// [nmin, nmax], every column j with a_j < lo = a_max - 2 eps - (nmax - nmin) / 2 has
//   sq_j = n_i + n_j + 2 s_j < n_i + nmax + 2 (lo + eps) = n_i + nmin + 2 (a_max - eps) <= sq of the best listed column,
// so when bound < lo the farthest row is among the listed window members { a_j >= lo }; they are re-scored exactly.
__global__ void __launch_bounds__(kFcWarps * 32) rr_farthest_certify_kernel(
    const float* __restrict__ x, int64_t D, const double* __restrict__ sqn, const unsigned long long* __restrict__ cand,
    const int32_t* __restrict__ cand_cnt, const uint32_t* __restrict__ row_tau, int n_lists, int list_cap,
    int64_t row_begin, int64_t n_rows, const float* __restrict__ range, float* __restrict__ colmax,
    int32_t* __restrict__ flag, unsigned long long* __restrict__ uncert_count) {
  const int lane = lane_id();
  const int64_t lr = (int64_t)blockIdx.x * kFcWarps + (threadIdx.x >> 5);
  if (lr >= n_rows) return;
  const int64_t row = row_begin + lr;
  const float nmax = range[0], nmin = range[1];
  const float eps = fc_err_bound(nmax);
  bool ok = true;
  float amax = -INFINITY;
  for (int q = 0; q < n_lists; ++q) {
    const int64_t li = lr * n_lists + q;
    const int c = cand_cnt[li];
    ok &= c <= list_cap;
    const unsigned long long* src = cand + li * (int64_t)list_cap;
    for (int t = lane; t < min(c, list_cap); t += 32) amax = fmaxf(amax, __uint_as_float((uint32_t)(src[t] >> 32)));
  }
  amax = warp_max(amax);
  // (nmax - nmin) / 2 plus a margin for the fp32 norms of the range against the fp64 norms of the re-score
  const float lo = amax - 2.0f * eps - 0.5f * (nmax - nmin) - 1e-6f * nmax;
  const uint32_t tq = row_tau[lr];
  const float bound = tq ? ord_float(tq) : -INFINITY;
  ok = ok && amax > -INFINITY && bound < lo;
  const float* xi = x + row * D;
  const double ni = sqn[row];
  float best = 0.f;
  int n_win = 0;
  for (int q = 0; q < n_lists && ok; ++q) {
    const int64_t li = lr * n_lists + q;
    const int c = min(cand_cnt[li], list_cap);
    const unsigned long long* src = cand + li * (int64_t)list_cap;
    for (int base = 0; base < c && ok; base += 32) {
      const int t = base + lane;
      const unsigned long long e = t < c ? src[t] : 0ull;
      const float a = __uint_as_float((uint32_t)(e >> 32));
      unsigned b = __ballot_sync(kFull, t < c && a >= lo);
      n_win += __popc(b);
      if (n_win > kFcWinMax) ok = false;
      while (b && ok) {
        const int src_lane = __ffs(b) - 1;
        b &= b - 1;
        const int32_t j = (int32_t)(uint32_t)__shfl_sync(kFull, e, src_lane);
        const float aj = __shfl_sync(kFull, a, src_lane);
        const double dot = warp_dot64(xi, x + (int64_t)j * D, D, lane);
        if (fabsf(aj - (float)(-dot)) > eps) ok = false;      // audit of the fp16 bound: never trust it blindly
        const float s = pair_sq(ni, sqn[j], dot);
        best = fmaxf(best, __fmul_rn(s, s));
      }
    }
  }
  if (lane == 0) {
    colmax[row] = ok ? best : 0.f;      // an uncertified row is zeroed here and filled by reid_rr_farthest_exact
    flag[lr] = ok ? 0 : 1;
    if (!ok && uncert_count) atomicAdd(uncert_count, 1ull);
  }
}

__global__ void rr_zero_rows_kernel(const int32_t* __restrict__ rows, int64_t row_begin, int64_t n_rows, float* __restrict__ colmax) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r < n_rows) colmax[rows ? (int64_t)rows[r] : row_begin + r] = 0.f;
}

// Exact scan: colmax[row] = max_j fp32(sq(row, j)^2) over all M rows.  A CTA parks R <= 8 query rows in shared memory
// and scans the columns [c0, c1) of its split, one column per warp at a time; squares are non-negative, so the float
// bits order like unsigned integers and the splits meet in an atomicMax.
__global__ void __launch_bounds__(kFxThreads) rr_farthest_exact_kernel(const float* __restrict__ x, int64_t M, int64_t D,
                                                                       const double* __restrict__ sqn,
                                                                       const int32_t* __restrict__ rows, int64_t row_begin,
                                                                       int64_t n_rows, int R, int64_t cols_per_split,
                                                                       unsigned* __restrict__ colmax_bits) {
  extern __shared__ float s_q[];        // R x D
  __shared__ unsigned s_max[kFxRows];
  const int w = threadIdx.x >> 5, lane = lane_id();
  const int64_t r0 = (int64_t)blockIdx.x * R;
  const int nr = (int)min((int64_t)R, n_rows - r0);
  int64_t qrow[kFxRows];
  double qn[kFxRows];
#pragma unroll
  for (int r = 0; r < kFxRows; ++r) {
    qrow[r] = r < nr ? (rows ? (int64_t)rows[r0 + r] : row_begin + r0 + r) : 0;
    qn[r] = r < nr ? sqn[qrow[r]] : 0.0;
  }
#pragma unroll
  for (int r = 0; r < kFxRows; ++r)
    if (r < nr)
      for (int64_t d = threadIdx.x; d < D; d += blockDim.x) s_q[r * D + d] = x[qrow[r] * D + d];
  if (threadIdx.x < kFxRows) s_max[threadIdx.x] = 0u;
  __syncthreads();
  float mx[kFxRows];
#pragma unroll
  for (int r = 0; r < kFxRows; ++r) mx[r] = 0.f;
  const int64_t c0 = (int64_t)blockIdx.y * cols_per_split, c1 = min(M, c0 + cols_per_split);
  for (int64_t j = c0 + w; j < c1; j += kFxThreads / 32) {
    const float* xj = x + j * D;
    double acc[kFxRows];
#pragma unroll
    for (int r = 0; r < kFxRows; ++r) acc[r] = 0.0;
    for (int64_t d = lane; d < D; d += 32) {
      const double v = (double)xj[d];
#pragma unroll
      for (int r = 0; r < kFxRows; ++r)
        if (r < nr) acc[r] = fma((double)s_q[r * D + d], v, acc[r]);
    }
    const double nj = sqn[j];
#pragma unroll
    for (int r = 0; r < kFxRows; ++r) {
      if (r < nr) {
        const float s = pair_sq(qn[r], nj, warp_sum(acc[r]));
        mx[r] = fmaxf(mx[r], __fmul_rn(s, s));
      }
    }
  }
  if (lane == 0) {
#pragma unroll
    for (int r = 0; r < kFxRows; ++r)
      if (r < nr) atomicMax(&s_max[r], __float_as_uint(mx[r]));
  }
  __syncthreads();
  if (threadIdx.x < nr) {
    const int64_t t = r0 + threadIdx.x;
    atomicMax(&colmax_bits[rows ? (int64_t)rows[t] : row_begin + t], s_max[threadIdx.x]);
  }
}

// V[i, e] = exp(-orig(e, i) / colmax[i]) / sum_e' (...)   (:66-67) -- the dense path's rr_weights_kernel with the distance
// gathered from the feature rows instead of read from a dist row; the same fp32 summation order.  One warp per row.
__global__ void __launch_bounds__(256) rr_weights_features_kernel(const float* __restrict__ x, int64_t D,
                                                                  const double* __restrict__ sqn,
                                                                  const float* __restrict__ colmax,
                                                                  const int32_t* __restrict__ E_pad, int stride,
                                                                  const int64_t* __restrict__ E_ptr, int64_t n_rows,
                                                                  int32_t* __restrict__ E_idx, float* __restrict__ V_val) {
  const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= n_rows) return;
  const int lane = lane_id();
  const int64_t p0 = E_ptr[row];
  const int n = (int)(E_ptr[row + 1] - p0);
  const int32_t* erow = E_pad + row * (int64_t)stride;
  const float* xi = x + row * D;
  const double ni = sqn[row];
  const float cm = colmax[row];
  float sum = 0.f;
  for (int e0 = 0; e0 < n; e0 += 32) {
    const int32_t mine = e0 + lane < n ? erow[e0 + lane] : 0;
    const int m = min(32, n - e0);
    for (int u = 0; u < m; ++u) {
      const int32_t j = __shfl_sync(kFull, mine, u);
      const double dot = warp_dot64(xi, x + (int64_t)j * D, D, lane);
      const float s = pair_sq(ni, sqn[j], dot);
      const float w = expf(-__fdiv_rn(__fmul_rn(s, s), cm));
      if (lane == u) {
        E_idx[p0 + e0 + u] = j;
        V_val[p0 + e0 + u] = w;
        sum += w;
      }
    }
  }
  sum = warp_sum(sum);
  __syncwarp();
  for (int e = lane; e < n; e += 32) V_val[p0 + e] = __fdiv_rn(V_val[p0 + e], sum);
}

// final[i][g] = J[i - row_begin][Q + g] * (1 - lambda) + (q_g[i][g]^2 / colmax[i]) * lambda  for i in [row_begin, row_end)
// (:95-96 with the dense path's dist[i][Q + g] = q_g[i][g]^2 / colmax[i], same fp32 operations)
__global__ void __launch_bounds__(256) rr_final_qg_kernel(const float* __restrict__ J, int64_t ldJ, const float* __restrict__ qg,
                                                          const float* __restrict__ colmax, int64_t Q, int64_t G, int64_t row_begin,
                                                          float one_minus_lambda, float lambda, float* __restrict__ out) {
  const int64_t r = blockIdx.y, i = row_begin + r;
  const float cm = colmax[i];
  for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < G; g += (int64_t)gridDim.x * blockDim.x) {
    const float v = qg[i * G + g];
    out[i * G + g] = __fadd_rn(__fmul_rn(J[r * ldJ + Q + g], one_minus_lambda), __fmul_rn(__fdiv_rn(__fmul_rn(v, v), cm), lambda));
  }
}

}  // namespace reid

extern "C" {

int reid_rr_row_sqnorm64(const float* x, int64_t n_rows, int64_t D, double* sqnorm, void* stream) {
  using namespace reid;
  REID_CHECK_ARG(x && sqnorm, "reid_rr_row_sqnorm64: NULL pointer");
  REID_CHECK_ARG(n_rows >= 1 && D >= 1, "reid_rr_row_sqnorm64: bad shape");
  rr_sqnorm64_kernel<<<(unsigned)((n_rows + 7) / 8), 256, 0, (cudaStream_t)stream>>>(x, n_rows, D, sqnorm);
  REID_LAUNCH_CHECK();
  return REID_OK;
}

int reid_rr_farthest_certify(const float* x, int64_t M, int64_t D, const double* sqnorm, const uint64_t* cand,
                             const int32_t* cand_cnt, const uint32_t* row_tau, int n_lists, int list_cap, int64_t row_begin,
                             int64_t row_end, const float* sqnorm_range, float* colmax, int32_t* uncertified_flag,
                             uint64_t* uncertified_count, void* stream) {
  using namespace reid;
  REID_CHECK_ARG(x && sqnorm && cand && cand_cnt && row_tau && sqnorm_range && colmax && uncertified_flag,
                 "reid_rr_farthest_certify: NULL pointer");
  REID_CHECK_ARG(M >= 1 && D >= 1 && 0 <= row_begin && row_begin < row_end && row_end <= M,
                 "reid_rr_farthest_certify: bad shape");
  REID_CHECK_ARG(n_lists >= 1 && n_lists <= 2 * REID_TC_MAX_SPLITS && list_cap >= 1,
                 "reid_rr_farthest_certify: n_lists=%d list_cap=%d", n_lists, list_cap);
  const int64_t n = row_end - row_begin;
  rr_farthest_certify_kernel<<<(unsigned)((n + kFcWarps - 1) / kFcWarps), kFcWarps * 32, 0, (cudaStream_t)stream>>>(
      x, D, sqnorm, (const unsigned long long*)cand, cand_cnt, row_tau, n_lists, list_cap, row_begin, n, sqnorm_range, colmax,
      uncertified_flag, (unsigned long long*)uncertified_count);
  REID_LAUNCH_CHECK();
  return REID_OK;
}

int reid_rr_farthest_exact(const float* x, int64_t M, int64_t D, const double* sqnorm, const int32_t* rows, int64_t row_begin,
                           int64_t n_rows, float* colmax, void* stream) {
  using namespace reid;
  REID_CHECK_ARG(x && sqnorm && colmax, "reid_rr_farthest_exact: NULL pointer");
  REID_CHECK_ARG(M >= 1 && D >= 1 && n_rows >= 0 && (rows || (0 <= row_begin && row_begin + n_rows <= M)),
                 "reid_rr_farthest_exact: bad shape");
  const size_t row_bytes = (size_t)D * sizeof(float);
  REID_CHECK_ARG(row_bytes <= 200 * 1024, "reid_rr_farthest_exact: D=%lld too large", (long long)D);
  if (n_rows == 0) return REID_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int R = (int)(row_bytes * kFxRows <= 160 * 1024 ? kFxRows : (160 * 1024) / row_bytes > 0 ? (160 * 1024) / row_bytes : 1);
  const size_t smem = row_bytes * (size_t)R;
  const int64_t row_blocks = (n_rows + R - 1) / R;
  // enough CTAs for a few waves, every split at least 64 columns wide
  int64_t splits = (4LL * num_sms() + row_blocks - 1) / row_blocks;
  splits = splits < 1 ? 1 : splits > (M + 63) / 64 ? (M + 63) / 64 : splits;
  if (splits > 65535) splits = 65535;
  const int64_t cols = (M + splits - 1) / splits;
  REID_CHECK_ARG(row_blocks < (1LL << 31), "reid_rr_farthest_exact: too many rows");
  rr_zero_rows_kernel<<<(unsigned)((n_rows + 255) / 256), 256, 0, st>>>(rows, row_begin, n_rows, colmax);
  REID_LAUNCH_CHECK();
  if (smem > 48 * 1024)
    REID_CUDA(cudaFuncSetAttribute(rr_farthest_exact_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  rr_farthest_exact_kernel<<<dim3((unsigned)row_blocks, (unsigned)((M + cols - 1) / cols)), kFxThreads, smem, st>>>(
      x, M, D, sqnorm, rows, row_begin, n_rows, R, cols, (unsigned*)colmax);
  REID_LAUNCH_CHECK();
  return REID_OK;
}

int reid_rr_weights_features(const float* x, int64_t M, int64_t D, const double* sqnorm, const float* colmax,
                             const int32_t* E_pad, int stride, const int64_t* E_ptr, int64_t n_rows, int32_t* E_idx,
                             float* V_val, void* stream) {
  using namespace reid;
  REID_CHECK_ARG(x && sqnorm && colmax && E_pad && E_ptr && E_idx && V_val, "reid_rr_weights_features: NULL pointer");
  REID_CHECK_ARG(M >= 1 && D >= 1 && stride >= 1 && 0 <= n_rows && n_rows <= M, "reid_rr_weights_features: bad shape");
  if (n_rows == 0) return REID_OK;
  rr_weights_features_kernel<<<(unsigned)((n_rows + 7) / 8), 256, 0, (cudaStream_t)stream>>>(x, D, sqnorm, colmax, E_pad, stride,
                                                                                           E_ptr, n_rows, E_idx, V_val);
  REID_LAUNCH_CHECK();
  return REID_OK;
}

int reid_rr_final_qg(const float* J, int64_t ldJ, const float* q_g, const float* colmax, int64_t Q, int64_t G,
                     int64_t row_begin, int64_t row_end, float one_minus_lambda, float lambda, float* out, void* stream) {
  using namespace reid;
  REID_CHECK_ARG(J && q_g && colmax && out, "reid_rr_final_qg: NULL pointer");
  REID_CHECK_ARG(Q >= 1 && G >= 1 && ldJ >= Q + G && 0 <= row_begin && row_begin < row_end && row_end <= Q &&
                     row_end - row_begin < 65536,
                 "reid_rr_final_qg: bad shape");
  int64_t bx = (G + 255) / 256;
  if (bx > 64) bx = 64;
  rr_final_qg_kernel<<<dim3((unsigned)bx, (unsigned)(row_end - row_begin)), 256, 0, (cudaStream_t)stream>>>(
      J, ldJ, q_g, colmax, Q, G, row_begin, one_minus_lambda, lambda, out);
  REID_LAUNCH_CHECK();
  return REID_OK;
}
}
