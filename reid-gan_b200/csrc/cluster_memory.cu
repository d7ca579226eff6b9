// a10-a12 -- ClusterMemory (clustercontrast/models/cm.py:9-76, 110-137).
// The problem is latency bound (B=256, C~700, D=2048: 1.5 GFLOP, 16 MB), so the design goal is
// few launches and no host synchronisation -- the reference's CM_Hard.backward performs 256
// .cpu() round trips (cm.py:66).  The two GEMMs run on the tensor cores as 3-product TF32 splits (fp32-accurate:
// loss and centroids stay within 1e-4 of the reference's fp32 cuBLAS path), everything else in fp32.
//   forward : split-K GEMM (raw inputs . F^T)  ->  per-row kernel: norm, xhat, z, logsumexp, loss
//   backward: per-row softmax-grad  ->  GEMM (gz . F)  ->  per-row normalize-backward
//   update  : one CTA per distinct label (sequential chain for CM, first-argmin for CM_Hard)
#include "common.cuh"

namespace reid {

constexpr int GM = 64, GN = 64, GK = 16;

// The two contractions (logits = x . F^T, grad = gz . F; 0.73 GFLOP each) run on the tensor cores in TF32 with the
// 3-product split that keeps fp32 accuracy: a = a_hi + a_lo with a_hi = tf32(a), a_lo = tf32(a - a_hi), and
// a.b ~ a_lo.b_hi + a_hi.b_lo + a_hi.b_hi (the dropped a_lo.b_lo term and the representation error are ~2^-22 per
// product; fp32 accumulators).  After the x20 of 1/temp the logits still agree with the reference's fp32 cuBLAS result
// far inside the 1e-4 bar (tests/test_gpu_cm.py: rtol 1e-4, atol 2e-6 on loss, gradient and centroids).  The tiles are
// small (B = 256, C ~ 700: 44 CTAs per split) and the operands need no layout change, so this is the register-operand
// mma.sync.m16n8k8 path rather than a tcgen05 / TMEM pipeline: the stage is latency bound (1.5 GFLOP per step).
__device__ __forceinline__ uint32_t to_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
  hi = to_tf32(x);
  lo = to_tf32(x - __uint_as_float(hi));
}
__device__ __forceinline__ void mma_tf32(float (&c)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile(
      "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

// out[z][m][n] = sum_{k in slice z} A[m][k] * Bop[k][n]
//   kBT = true : B is [Nn x K] row-major (out = A . B^T);  false: B is [K x Nn] row-major (out = A . B)
// 8 warps = 4 (M) x 2 (N); a warp owns a 16 x 32 piece of the 64 x 64 tile = one A fragment x four B fragments per
// 8-wide K step.  Shared-memory rows are padded to 72 floats: the fragment loads (k = t or t + 4, m / n = g) then hit
// 32 different banks.
template <bool kBT>
__global__ void __launch_bounds__(256) gemm_f32_kernel(const float* __restrict__ A, const float* __restrict__ B,
                                                       int64_t M, int64_t Nn, int64_t K, int64_t k_per_split,
                                                       float* __restrict__ out) {
  __shared__ float As[GK][GM + 8];
  __shared__ float Bs[GK][GN + 8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int wm = warp >> 1, wn = warp & 1;
  const int64_t m0 = (int64_t)blockIdx.y * GM, n0 = (int64_t)blockIdx.x * GN;
  const int64_t kb = (int64_t)blockIdx.z * k_per_split;
  const int64_t ke = kb + k_per_split < K ? kb + k_per_split : K;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  for (int64_t k0 = kb; k0 < ke; k0 += GK) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int lin = threadIdx.x + e * 256;  // 1024 elements per operand tile
      {
        const int mm = lin >> 4, kk = lin & 15;  // A: consecutive threads walk k (contiguous)
        const int64_t gm = m0 + mm, gk = k0 + kk;
        As[kk][mm] = (gm < M && gk < ke) ? A[gm * K + gk] : 0.f;
      }
      if (kBT) {
        const int nn = lin >> 4, kk = lin & 15;
        const int64_t gn = n0 + nn, gk = k0 + kk;
        Bs[kk][nn] = (gn < Nn && gk < ke) ? B[gn * K + gk] : 0.f;
      } else {
        const int kk = lin >> 6, nn = lin & 63;  // B: consecutive threads walk n (contiguous)
        const int64_t gn = n0 + nn, gk = k0 + kk;
        Bs[kk][nn] = (gn < Nn && gk < ke) ? B[gk * Nn + gn] : 0.f;
      }
    }
    __syncthreads();
#pragma unroll
    for (int ks = 0; ks < GK; ks += 8) {
      uint32_t ah[4], al[4];
      split_tf32(As[ks + t][wm * 16 + g], ah[0], al[0]);
      split_tf32(As[ks + t][wm * 16 + g + 8], ah[1], al[1]);
      split_tf32(As[ks + t + 4][wm * 16 + g], ah[2], al[2]);
      split_tf32(As[ks + t + 4][wm * 16 + g + 8], ah[3], al[3]);
#pragma unroll
      for (int nf = 0; nf < 4; ++nf) {
        uint32_t bh[2], bl[2];
        split_tf32(Bs[ks + t][wn * 32 + nf * 8 + g], bh[0], bl[0]);
        split_tf32(Bs[ks + t + 4][wn * 32 + nf * 8 + g], bh[1], bl[1]);
        mma_tf32(acc[nf], al, bh);        // the small terms first
        mma_tf32(acc[nf], ah, bl);
        mma_tf32(acc[nf], ah, bh);
      }
    }
    __syncthreads();
  }
  // C fragment: (g, 2t), (g, 2t + 1), (g + 8, 2t), (g + 8, 2t + 1) of the 16 x 8 piece
  float* o = out + (int64_t)blockIdx.z * M * Nn;
#pragma unroll
  for (int nf = 0; nf < 4; ++nf) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int64_t m = m0 + wm * 16 + g + (e >> 1) * 8;
      const int64_t n = n0 + wn * 32 + nf * 8 + 2 * t + (e & 1);
      if (m < M && n < Nn) o[m * Nn + n] = acc[nf][e];
    }
  }
}

__device__ __forceinline__ float block_sum(float v, float* red) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = 0.f;
  for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
  return t;
}
__device__ __forceinline__ float block_max(float v, float* red) {
  v = warp_max(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = -INFINITY;
  for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t = fmaxf(t, red[w]);
  return t;
}

// One CTA per sample: ||x||, xhat, z = (sum of split-K partials) / (||x|| * temp), loss.
// kPush (reid_cm_forward_push): the CTA also stores the row's target and xhat into slot me * cap + b of EVERY rank's
// receive buffer (peer_base[w]: W * cap int64 targets, then W * cap x D fp32 xhat).  The grid then covers cap rows:
// the CTAs of rows B <= b < cap only store target -1 (the update kernel skips it).
template <bool kPush>
__global__ void __launch_bounds__(256) cm_loss_kernel(const float* __restrict__ inputs,
                                                      const int64_t* __restrict__ targets,
                                                      const float* __restrict__ partial, int splits, int64_t B,
                                                      int64_t C, int64_t D, float temp, float* __restrict__ loss,
                                                      float* __restrict__ xhat, float* __restrict__ inv_norm,
                                                      float* __restrict__ z, int me, int W, int64_t cap,
                                                      const unsigned long long* __restrict__ peer_base) {
  __shared__ float red[8];
  const int64_t b = blockIdx.x;
  const int64_t slot = (int64_t)me * cap + b;
  if (kPush) {
    for (int w = threadIdx.x; w < W; w += blockDim.x)
      reinterpret_cast<int64_t*>(peer_base[w])[slot] = b < B ? targets[b] : -1;
    if (b >= B) {
      __threadfence_system();
      return;
    }
  }
  const float* x = inputs + b * D;
  float ss = 0.f;
  for (int64_t d = threadIdx.x; d < D; d += blockDim.x) ss = fmaf(x[d], x[d], ss);
  ss = block_sum(ss, red);
  const float inv = 1.0f / fmaxf(sqrtf(ss), 1e-12f);  // F.normalize(eps=1e-12), cm.py:125
  for (int64_t d = threadIdx.x; d < D; d += blockDim.x) {
    const float v = x[d] * inv;
    xhat[b * D + d] = v;
    if (kPush)
      for (int w = 0; w < W; ++w)
        reinterpret_cast<float*>(reinterpret_cast<int64_t*>(peer_base[w]) + (int64_t)W * cap)[slot * D + d] = v;
  }
  if (threadIdx.x == 0) inv_norm[b] = inv;
  const float scale = inv / temp;
  float mx = -INFINITY;
  for (int64_t c = threadIdx.x; c < C; c += blockDim.x) {
    float s = 0.f;
    for (int u = 0; u < splits; ++u) s += partial[((int64_t)u * B + b) * C + c];
    s *= scale;
    z[b * C + c] = s;
    mx = fmaxf(mx, s);
  }
  mx = block_max(mx, red);
  float se = 0.f;
  for (int64_t c = threadIdx.x; c < C; c += blockDim.x) se += expf(z[b * C + c] - mx);
  se = block_sum(se, red);
  if (threadIdx.x == 0) {
    // cross_entropy(reduction='none'), :135.  A target outside [0, C) (e.g. a DBSCAN outlier label -1 that was not
    // filtered out) is a device assert in PyTorch; here the sample's loss is NaN and no memory outside z is read.
    const int64_t y = targets[b];
    loss[b] = (y >= 0 && y < C) ? (mx + logf(se)) - z[b * C + y] : __int_as_float(0x7fc00000);
  }
  if (kPush) __threadfence_system();
}

// gz[b][c] = (softmax(z_b)[c] - [c == y_b]) * grad_loss[b] / temp
__global__ void __launch_bounds__(256) cm_gz_kernel(const float* __restrict__ grad_loss, const float* __restrict__ z,
                                                    const int64_t* __restrict__ targets, int64_t C, float temp,
                                                    float* __restrict__ gz) {
  __shared__ float red[8];
  const int64_t b = blockIdx.x;
  const float* zr = z + b * C;
  float mx = -INFINITY;
  for (int64_t c = threadIdx.x; c < C; c += blockDim.x) mx = fmaxf(mx, zr[c]);
  mx = block_max(mx, red);
  float se = 0.f;
  for (int64_t c = threadIdx.x; c < C; c += blockDim.x) se += expf(zr[c] - mx);
  se = block_sum(se, red);
  const float g = grad_loss[b] / temp;
  const int64_t y = targets[b];
  for (int64_t c = threadIdx.x; c < C; c += blockDim.x) {
    float p = expf(zr[c] - mx) / se;
    if (c == y) p -= 1.0f;
    gz[b * C + c] = p * g;
  }
}

// grad_x = (g - xhat * (xhat . g)) * inv_norm   (backward of F.normalize); in place on g
__global__ void __launch_bounds__(256) cm_normalize_bwd_kernel(const float* __restrict__ xhat,
                                                               const float* __restrict__ inv_norm, int64_t D,
                                                               float* __restrict__ g) {
  __shared__ float red[8];
  const int64_t b = blockIdx.x;
  float dot = 0.f;
  for (int64_t d = threadIdx.x; d < D; d += blockDim.x) dot = fmaf(xhat[b * D + d], g[b * D + d], dot);
  dot = block_sum(dot, red);
  const float inv = inv_norm[b];
  for (int64_t d = threadIdx.x; d < D; d += blockDim.x) g[b * D + d] = (g[b * D + d] - xhat[b * D + d] * dot) * inv;
}

// One CTA per batch row; only the first occurrence of a label does work for that label.
constexpr int kUpdMaxPerThread = 16;  // D <= 4096 with 256 threads

__global__ void __launch_bounds__(256) cm_update_kernel(const float* __restrict__ xhat,
                                                        const int64_t* __restrict__ targets,
                                                        float* __restrict__ centroids, int64_t B, int64_t C, int64_t D,
                                                        float momentum, int hard) {
  __shared__ float red[8];
  __shared__ int s_skip, s_best;
  const int64_t b0 = blockIdx.x;
  const int64_t y = targets[b0];
  if (y < 0 || y >= C) return;                         // invalid label: no centroid row to update (loss was NaN)
  if (threadIdx.x == 0) {
    int skip = 0;
    for (int64_t u = 0; u < b0; ++u) skip |= (targets[u] == y);
    s_skip = skip;
  }
  __syncthreads();
  if (s_skip) return;
  float f[kUpdMaxPerThread];
#pragma unroll
  for (int u = 0; u < kUpdMaxPerThread; ++u) {
    const int64_t d = threadIdx.x + (int64_t)u * 256;
    f[u] = d < D ? centroids[y * D + d] : 0.f;
  }
  const float one_m = 1.0f - momentum;
  if (!hard) {
    // cm.py:29-31: for x, y in zip(inputs, targets): f[y] = m f[y] + (1-m) x; f[y] /= ||f[y]||
    for (int64_t b = b0; b < B; ++b) {
      if (targets[b] != y) continue;
      float ss = 0.f;
#pragma unroll
      for (int u = 0; u < kUpdMaxPerThread; ++u) {
        const int64_t d = threadIdx.x + (int64_t)u * 256;
        if (d < D) {
          f[u] = __fadd_rn(__fmul_rn(momentum, f[u]), __fmul_rn(one_m, xhat[b * D + d]));
          ss = fmaf(f[u], f[u], ss);
        }
      }
      ss = block_sum(ss, red);
      const float nrm = sqrtf(ss);
#pragma unroll
      for (int u = 0; u < kUpdMaxPerThread; ++u) f[u] = __fdiv_rn(f[u], nrm);
    }
  } else {
    // cm.py:58-70: hardest positive = first argmin over the label's members of x . f[y]
    float best = INFINITY;
    int best_b = (int)b0;
    for (int64_t b = b0; b < B; ++b) {
      if (targets[b] != y) continue;
      float dot = 0.f;
#pragma unroll
      for (int u = 0; u < kUpdMaxPerThread; ++u) {
        const int64_t d = threadIdx.x + (int64_t)u * 256;
        if (d < D) dot = fmaf(xhat[b * D + d], f[u], dot);
      }
      dot = block_sum(dot, red);
      if (dot < best) {  // strict: np.argmin keeps the first minimum
        best = dot;
        best_b = (int)b;
      }
    }
    if (threadIdx.x == 0) s_best = best_b;
    __syncthreads();
    const int64_t bb = s_best;
    float ss = 0.f;
#pragma unroll
    for (int u = 0; u < kUpdMaxPerThread; ++u) {
      const int64_t d = threadIdx.x + (int64_t)u * 256;
      if (d < D) {
        f[u] = __fadd_rn(__fmul_rn(f[u], momentum), __fmul_rn(one_m, xhat[bb * D + d]));
        ss = fmaf(f[u], f[u], ss);
      }
    }
    ss = block_sum(ss, red);
    const float nrm = sqrtf(ss);
#pragma unroll
    for (int u = 0; u < kUpdMaxPerThread; ++u) f[u] = __fdiv_rn(f[u], nrm);
  }
#pragma unroll
  for (int u = 0; u < kUpdMaxPerThread; ++u) {
    const int64_t d = threadIdx.x + (int64_t)u * 256;
    if (d < D) centroids[y * D + d] = f[u];
  }
}

static int launch_gemm(bool bt, const float* A, const float* Bm, int64_t M, int64_t Nn, int64_t K, int splits,
                       float* out, cudaStream_t st) {
  int64_t kps = (K + splits - 1) / splits;
  kps = (kps + GK - 1) / GK * GK;
  dim3 grid((unsigned)((Nn + GN - 1) / GN), (unsigned)((M + GM - 1) / GM), (unsigned)splits);
  if (bt)
    gemm_f32_kernel<true><<<grid, 256, 0, st>>>(A, Bm, M, Nn, K, kps, out);
  else
    gemm_f32_kernel<false><<<grid, 256, 0, st>>>(A, Bm, M, Nn, K, kps, out);
  REID_LAUNCH_CHECK();
  return REID_OK;
}

static int pick_splits(int64_t M, int64_t Nn, int64_t K) {
  const int64_t tiles = ((M + GM - 1) / GM) * ((Nn + GN - 1) / GN);
  int s = (int)((2 * (int64_t)num_sms() + tiles - 1) / tiles);
  if (s < 1) s = 1;
  if (s > 8) s = 8;
  while (s > 1 && K / s < 64) --s;
  return s;
}

}  // namespace reid

extern "C" {

size_t reid_cm_forward_scratch_bytes(int64_t B, int64_t C, int64_t D) {
  using namespace reid;
  if (B <= 0 || C <= 0 || D <= 0) return 0;
  return sizeof(float) * (size_t)pick_splits(B, C, D) * (size_t)B * (size_t)C;
}

int reid_cm_forward(const float* inputs, const int64_t* targets, const float* centroids, int64_t B, int64_t C,
                    int64_t D, float temp, float* loss, float* xhat, float* inv_norm, float* z, void* scratch,
                    void* stream) {
  using namespace reid;
  REID_CHECK_ARG(inputs && targets && centroids && loss && xhat && inv_norm && z && scratch,
                 "reid_cm_forward: NULL pointer");
  REID_CHECK_ARG(B > 0 && C > 0 && D > 0 && temp > 0.f, "reid_cm_forward: bad shape/temp");
  cudaStream_t st = (cudaStream_t)stream;
  const int splits = pick_splits(B, C, D);
  float* partial = (float*)scratch;
  int rc = launch_gemm(true, inputs, centroids, B, C, D, splits, partial, st);
  if (rc != REID_OK) return rc;
  cm_loss_kernel<false><<<(unsigned)B, 256, 0, st>>>(inputs, targets, partial, splits, B, C, D, temp, loss, xhat,
                                                      inv_norm, z, 0, 1, 0, nullptr);
  REID_LAUNCH_CHECK();
  return REID_OK;
}

int reid_cm_forward_push(const float* inputs, const int64_t* targets, const float* centroids, int64_t B, int64_t C,
                         int64_t D, float temp, int64_t B_split, float* loss, float* xhat, float* inv_norm, float* z,
                         void* scratch, int me, int world, int64_t cap, const uint64_t* peer_base, void* stream) {
  using namespace reid;
  REID_CHECK_ARG(inputs && targets && centroids && loss && xhat && inv_norm && z && scratch && peer_base,
                 "reid_cm_forward_push: NULL pointer");
  REID_CHECK_ARG(B > 0 && C > 0 && D > 0 && temp > 0.f, "reid_cm_forward_push: bad shape/temp");
  REID_CHECK_ARG(world >= 1 && me >= 0 && me < world, "reid_cm_forward_push: bad rank me=%d of world=%d", me, world);
  REID_CHECK_ARG(B <= cap && B <= B_split, "reid_cm_forward_push: B=%lld exceeds cap=%lld or B_split=%lld",
                 (long long)B, (long long)cap, (long long)B_split);
  REID_CHECK_ARG(D <= 256 * kUpdMaxPerThread, "reid_cm_forward_push: D=%lld exceeds %d", (long long)D,
                 256 * kUpdMaxPerThread);
  cudaStream_t st = (cudaStream_t)stream;
  const int splits = pick_splits(B_split, C, D);  // the split-K count of the whole (all-rank) batch
  float* partial = (float*)scratch;
  int rc = launch_gemm(true, inputs, centroids, B, C, D, splits, partial, st);
  if (rc != REID_OK) return rc;
  cm_loss_kernel<true><<<(unsigned)cap, 256, 0, st>>>(inputs, targets, partial, splits, B, C, D, temp, loss, xhat,
                                                      inv_norm, z, me, world, cap,
                                                      (const unsigned long long*)peer_base);
  REID_LAUNCH_CHECK();
  return REID_OK;
}

int reid_cm_backward(const float* grad_loss, const float* z, const int64_t* targets, const float* centroids,
                     const float* xhat, const float* inv_norm, int64_t B, int64_t C, int64_t D, float temp,
                     float* gz_scratch, float* grad_inputs, void* stream) {
  using namespace reid;
  REID_CHECK_ARG(grad_loss && z && targets && centroids && xhat && inv_norm && gz_scratch && grad_inputs,
                 "reid_cm_backward: NULL pointer");
  REID_CHECK_ARG(B > 0 && C > 0 && D > 0 && temp > 0.f, "reid_cm_backward: bad shape/temp");
  cudaStream_t st = (cudaStream_t)stream;
  cm_gz_kernel<<<(unsigned)B, 256, 0, st>>>(grad_loss, z, targets, C, temp, gz_scratch);
  REID_LAUNCH_CHECK();
  int rc = launch_gemm(false, gz_scratch, centroids, B, D, C, 1, grad_inputs, st);
  if (rc != REID_OK) return rc;
  cm_normalize_bwd_kernel<<<(unsigned)B, 256, 0, st>>>(xhat, inv_norm, D, grad_inputs);
  REID_LAUNCH_CHECK();
  return REID_OK;
}

int reid_cm_logits(const float* a, const float* centroids, int64_t B, int64_t C, int64_t D, float* out, void* stream) {
  using namespace reid;
  REID_CHECK_ARG(a && centroids && out && B > 0 && C > 0 && D > 0, "reid_cm_logits: bad arguments");
  return launch_gemm(true, a, centroids, B, C, D, 1, out, (cudaStream_t)stream);
}

int reid_cm_grad_inputs(const float* g, const float* centroids, int64_t B, int64_t C, int64_t D, float* out,
                        void* stream) {
  using namespace reid;
  REID_CHECK_ARG(g && centroids && out && B > 0 && C > 0 && D > 0, "reid_cm_grad_inputs: bad arguments");
  return launch_gemm(false, g, centroids, B, D, C, 1, out, (cudaStream_t)stream);
}

int reid_cm_update(const float* xhat, const int64_t* targets, float* centroids, int64_t B, int64_t C, int64_t D,
                   float momentum, int hard, void* workspace, void* stream) {
  using namespace reid;
  (void)workspace;
  REID_CHECK_ARG(xhat && targets && centroids && B > 0 && C > 0 && D > 0, "reid_cm_update: bad arguments");
  REID_CHECK_ARG(D <= 256 * kUpdMaxPerThread, "reid_cm_update: D=%lld exceeds %d", (long long)D, 256 * kUpdMaxPerThread);
  cm_update_kernel<<<(unsigned)B, 256, 0, (cudaStream_t)stream>>>(xhat, targets, centroids, B, C, D, momentum, hard);
  REID_LAUNCH_CHECK();
  return REID_OK;
}
}
