// a1 (first half), symmetric form -- S = Xh Xh^T is symmetric, so only the tiles (I, J) with I <= J of the
// N x N similarity are put through the tensor cores and every off-diagonal tile feeds the candidate lists
// of BOTH its row block and its column block: half the tcgen05 work and half the L2 -> shared-memory
// operand traffic of simgemm_tc.cu (whose main loop is bound by exactly that traffic).
// (replaces the SGEMM + block-select inside faiss IndexFlatL2 / GpuIndexFlatL2.search,
//  utils/faiss_rerank.py:39-62)
//
// A running top-K cannot be kept for the transposed direction (the rows of a column block are owned by
// other CTAs), so the selection uses a FIXED per-row rejection threshold found beforehand:
//   1. prepass  : simtopk_kernel scores every row against a small quasi-random SAMPLE of the rows
//                 (reid_features_sample) and sample_tau_kernel takes the r-th best sample score as tau_i.
//                 Rank statistics of a sample are distribution free: about r/m * N columns beat tau_i.
//   2. main pass: simsym_kernel appends (score, column) to row i's list whenever score > tau_i -- for the
//                 tile's own rows against tau of the row held in a register, for the transposed direction
//                 against the 256 thresholds of the column block staged in shared memory -- with one
//                 atomicAdd per survivor; there is no list maintenance at all in the epilogue.
// knn_rescore.cu certifies each row exactly as before (every column outside the list scored <= tau_i); a
// threshold that turned out too high or a list that overflowed only un-certifies the row, which is then
// redone by reid_knn_exact, so the result never depends on the sample.
//
// Kernel anatomy = simgemm_tc.cu's CTA-pair flavour: persistent, one CTA per SM, warp 0 TMA producer,
// warp 1 (leader CTA) tcgen05.mma.cta_group::2 issuer, two epilogue warpgroups draining the two TMEM
// accumulators alternately; a work unit is ONE 256 x 256 tile taken from a host-ordered list
// (super-blocks of 8 x 8 tiles so that the ~74 tiles in flight share 16 operand blocks in L2).
#include <stdlib.h>

#include <type_traits>

#include "tc_ptx.cuh"

namespace reid {
namespace tc {

int make_tmap_rows128(CUtensorMap* tmap, const void* base, int64_t n_rows, int64_t D);   // simgemm_tc.cu

// Warps 0..7 are the two epilogue groups, warp 8 the TMA producer, warp 9 the MMA issuer: the warp scheduler
// favours the highest warp id among the eligible ones, and the single-thread MMA / TMA roles are the ones that
// must never wait for an issue slot behind an epilogue warp.
constexpr int kTmaWarp = 8, kMmaWarp = 9;
// NB = column blocks per work unit.  NB = 1: one 256 x 256 tile per unit, the two TMEM accumulators alternate between
// units (drain of one under the MMAs of the next).  NB = 2 ("wide"): a unit is the 256 x 512 strip (I, J0), (I, J1): both
// accumulators are filled from ONE A slice per K step, i.e. 48 KB instead of 64 KB of operands per 2 x 256 x 256 x 64
// MACs.  The main loop runs against the L2 -> shared-memory throughput of the chip (2 MB per tile x 8,256 tiles in
// 1.5 ms = 11.5 TB/s), so the wide strip buys 25 % of it; the price is that the drain is no longer under the MMAs of
// the next unit -- the TMA producer keeps refilling the ring meanwhile, so the operand feed never pauses.
template <int NB>
struct SymCfg {
  static constexpr int kStages = NB == 2 ? 4 : 6;
  static constexpr int kBHalf = 128 * BK * 2;                         // this CTA's half (128 rows) of one B block
  static constexpr int kStage = kATileBytes + NB * kBHalf;            // 32 KB / 48 KB
  static constexpr int kSmem = kStages * kStage + 1024 /*align*/ + 256 /*barriers*/ + 2 * BN * 4 + 8 * 8 * 32 * 8;
};
constexpr int kSymTauBytes = 2 * BN * 4;                  // column thresholds, one buffer per epilogue group
constexpr int kSymHitSlots = 8;                           // staged survivors per lane and tile
constexpr int kSymHitBytes = 8 * kSymHitSlots * 32 * 8;   // 8 epilogue warps x slots x lanes x 8 B = 16 KB

struct SymParams {
  int64_t N;
  int num_k_blocks;                // D / 64
  int n_units;                     // units in the list
  const int32_t* tiles;            // NB = 1: (I, J) pairs, I <= J, in processing order; NB = 2: (I, J0, J1) triples, J1 = -1:
                                   // a single tile
  const float* tau;                // [N] rejection threshold per row (descaled score units)
  float scale2;                    // 2^(2 s): raw accumulator = score * scale2
  float descale;                   // 2^(-2 s)
  int cap;                         // list capacity per row
  unsigned long long* cand;        // [N x cap] (score bits << 32) | column
  int32_t* cand_cnt;               // [N] appended entries (may exceed cap: the list overflowed)
  int dbg;                         // developer switch (REID_TC_DEBUG): 1 = epilogue skips the TMEM reads, 2 = reads but no
                                   // selection, 4 = no TMA (MMA issue only)
};

__device__ __forceinline__ void sym_append(const SymParams& p, int64_t row, int col, float s) {
  const int pos = atomicAdd(p.cand_cnt + row, 1);
  if (pos < p.cap) p.cand[row * p.cap + pos] = ((unsigned long long)__float_as_uint(s) << 32) | (uint32_t)col;
}

template <int NB>
__global__ void __launch_bounds__(kThreads, 1) simsym_kernel(const __grid_constant__ CUtensorMap tmap, const SymParams p) {
  constexpr int kSymStages = SymCfg<NB>::kStages, kSymStage = SymCfg<NB>::kStage, US = NB + 1;
  static_assert(SymCfg<NB>::kSmem <= 227 * 1024, "shared memory");
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* full_bar = (uint64_t*)(smem + kSymStages * kSymStage);
  uint64_t* empty_bar = full_bar + kSymStages;
  uint64_t* tfull_bar = empty_bar + kSymStages;   // [2] accumulator ready
  uint64_t* tempty_bar = tfull_bar + 2;           // [2] accumulator drained (lives in the leader CTA)
  uint32_t* tmem_slot = (uint32_t*)(tempty_bar + 2);
  float* s_tauc = (float*)(smem + kSymStages * kSymStage + 256);     // [2][BN]
  unsigned long long* s_hits = (unsigned long long*)(smem + kSymStages * kSymStage + 256 + kSymTauBytes);  // [8][slots][32]

  const int warp = threadIdx.x >> 5, lane = lane_id();
  const uint32_t cta_rank = cluster_ctarank();
  const bool leader = cta_rank == 0;

  if (warp == kTmaWarp && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap) : "memory");
    for (int s = 0; s < kSymStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull_bar[a], 1);
      mbar_init(&tempty_bar[a], 8);     // the 4 warps of the owning epilogue group, in both CTAs of the pair
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kMmaWarp) {  // TMEM: all 512 columns = two 128 x 256 fp32 accumulators (per CTA)
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
  }
  tcgen05_fence_before();
  cluster_sync_all();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int unit0 = blockIdx.x >> 1, unit_step = gridDim.x >> 1;

  if (warp == kTmaWarp) {
    // ------------------------------ TMA producer ------------------------------
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int u = unit0; u < p.n_units; u += unit_step) {
        const int ti = p.tiles[US * u], tj = p.tiles[US * u + 1];
        const int tj1 = NB == 2 ? p.tiles[US * u + 2] : -1;
        const int a_row = ti * BN + (int)cta_rank * BM;
        const int b_row = tj * BN + (int)cta_rank * 128;
        const int b1_row = tj1 * BN + (int)cta_rank * 128;
        const uint32_t tx = 2 * (kATileBytes + (tj1 >= 0 ? 2 : 1) * SymCfg<NB>::kBHalf);
        for (int kb = 0; kb < p.num_k_blocks; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* a_dst = smem + stage * kSymStage;
          uint8_t* b_dst = a_dst + kATileBytes;
          if (REID_DBG(p) & 4) {
            if (leader) mbar_arrive(&full_bar[stage]);
          } else {
            if (leader) mbar_expect_tx(&full_bar[stage], tx);   // the pair's bytes land on the leader's barrier
            const uint32_t lbar = mapa_u32(smem_u32(&full_bar[stage]), 0);
            tma_load_2d_pair(a_dst, &tmap, lbar, kb * BK, a_row);
            tma_load_2d_pair(b_dst, &tmap, lbar, kb * BK, b_row);
            if (NB == 2 && tj1 >= 0) tma_load_2d_pair(b_dst + SymCfg<NB>::kBHalf, &tmap, lbar, kb * BK, b1_row);
          }
          if (++stage == kSymStages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == kMmaWarp) {
    // ------------------------------ MMA issuer (leader CTA only) ----------------
    if (lane == 0 && leader) {
      constexpr uint32_t idesc = make_idesc(BM * 2, BN);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int u = unit0; u < p.n_units; u += unit_step) {
        bool two = false;
        if (NB == 2) {                                // the strip takes both accumulators
          two = p.tiles[US * u + 2] >= 0;
          mbar_wait(&tempty_bar[0], acc_phase ^ 1);
          mbar_wait(&tempty_bar[1], acc_phase ^ 1);
        } else {
          mbar_wait(&tempty_bar[acc], acc_phase ^ 1);   // every epilogue warp of the pair has drained this accumulator
        }
        tcgen05_fence_after();
        const uint32_t tmem_c = tmem_base + (uint32_t)(acc * BN);
        for (int kb = 0; kb < p.num_k_blocks; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tcgen05_fence_after();
          const uint32_t a_addr = smem_u32(smem + stage * kSymStage);
          const uint32_t b_addr = a_addr + kATileBytes;
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) {
            const uint64_t da = make_smem_desc(a_addr + k * UMMA_K * 2);
            const uint64_t db = make_smem_desc(b_addr + k * UMMA_K * 2);
            umma_f16_pair(tmem_c, da, db, idesc, (kb | k) != 0);
          }
          if (NB == 2 && two) {
#pragma unroll
            for (int k = 0; k < BK / UMMA_K; ++k) {
              const uint64_t da = make_smem_desc(a_addr + k * UMMA_K * 2);
              const uint64_t db = make_smem_desc(b_addr + SymCfg<NB>::kBHalf + k * UMMA_K * 2);
              umma_f16_pair(tmem_c + BN, da, db, idesc, (kb | k) != 0);
            }
          }
          umma_commit_pair(&empty_bar[stage]);
          if (++stage == kSymStages) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (NB == 2) {
          umma_commit_pair(&tfull_bar[0]);
          umma_commit_pair(&tfull_bar[1]);
          acc_phase ^= 1;
        } else {
          umma_commit_pair(&tfull_bar[acc]);
          if (++acc == 2) {
            acc = 0;
            acc_phase ^= 1;
          }
        }
      }
    }
  } else {
    // ------------------------------ epilogue: fixed-threshold selection, both directions -------------
    const int wg = warp >> 2;                           // group g drains accumulator g: every other tile (NB = 1) / block J_g
    const int quarter = warp & 3;                       // TMEM lanes this warp may read
    const int r_in_tile = (int)cta_rank * BM + quarter * 32 + lane;
    const int gt = (warp - wg * 4) * 32 + lane;         // 0..127 inside the group
    const uint32_t tempty_remote = mapa_u32(smem_u32(&tempty_bar[wg]), 0);
    float* tauc = s_tauc + wg * BN;
    unsigned long long* hits = s_hits + (size_t)warp * kSymHitSlots * 32;
    uint32_t acc_phase = 0;
    int tile_ctr = 0;
    for (int u = unit0; u < p.n_units; u += unit_step, ++tile_ctr) {
      if (NB == 1 && (tile_ctr & 1) != wg) continue;
      const int ti = p.tiles[US * u], tj = p.tiles[US * u + 1 + (NB == 2 ? wg : 0)];
      if (NB == 2 && tj < 0) {                            // single tile: nothing in this group's accumulator
        mbar_wait(&tfull_bar[wg], acc_phase);
        acc_phase ^= 1;
        __syncwarp();
        if (lane == 0) {
          if (leader) mbar_arrive(&tempty_bar[wg]);
          else mbar_arrive_cluster(tempty_remote);
        }
        continue;
      }
      const int64_t row = (int64_t)ti * BN + r_in_tile;
      const bool row_ok = row < p.N;
      const float tr = row_ok ? p.tau[row] * p.scale2 : INFINITY;          // compare raw accumulators
      // thresholds of the column block (transposed direction); none on the diagonal, where the tile holds
      // both (i, j) and (j, i) already
      __syncwarp();
      asm volatile("bar.sync %0, 128;" ::"r"(1 + wg) : "memory");          // the previous tile's readers are done
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int c = gt + h * 128;
        const int64_t col = (int64_t)tj * BN + c;
        tauc[c] = (ti != tj && col < p.N) ? p.tau[col] * p.scale2 : INFINITY;
      }
      asm volatile("bar.sync %0, 128;" ::"r"(1 + wg) : "memory");
      mbar_wait(&tfull_bar[wg], acc_phase);
      acc_phase ^= 1;
      tcgen05_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(wg * BN);
      int n_hit = 0;
#pragma unroll 1
      for (int ch = 0; ch < BN / 32; ++ch) {
        if (REID_DBG(p) & 1) break;
        uint32_t v[32];
        tmem_ld_32x32b_x32(taddr + ch * 32, v);
        const int col0 = tj * BN + ch * 32;
        if (REID_DBG(p) & 2) {
          float mx = 0.f;
#pragma unroll
          for (int c = 0; c < 32; ++c) mx = fmaxf(mx, __uint_as_float(v[c]));
          if (mx == 123.456f) sym_append(p, 0, 0, mx);
          continue;
        }
        const float4* tc4 = reinterpret_cast<const float4*>(tauc + ch * 32);
        unsigned hit = 0;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const float4 t4 = tc4[q];
          const float a0 = __uint_as_float(v[4 * q]), a1 = __uint_as_float(v[4 * q + 1]);
          const float a2 = __uint_as_float(v[4 * q + 2]), a3 = __uint_as_float(v[4 * q + 3]);
          hit |= (unsigned)((a0 > tr) | (a0 > t4.x)) << (4 * q);
          hit |= (unsigned)((a1 > tr) | (a1 > t4.y)) << (4 * q + 1);
          hit |= (unsigned)((a2 > tr) | (a2 > t4.z)) << (4 * q + 2);
          hit |= (unsigned)((a3 > tr) | (a3 > t4.w)) << (4 * q + 3);
        }
        while (hit) {                                    // rare: about r/m of the scores get here
          const int c = __ffs(hit) - 1;
          hit &= hit - 1;
          float a = 0.f;
#pragma unroll
          for (int e = 0; e < 32; ++e) a = e == c ? __uint_as_float(v[e]) : a;   // v[] stays in registers
          const int cl = ch * 32 + c;                    // column inside the tile
          const bool d_hit = a > tr && col0 + c < p.N;
          const bool t_hit = row_ok && a > tauc[cl];
          // Survivors are parked in shared memory (lane-private slots) and appended to the global lists only
          // after the accumulator has gone back to the MMA warp: an atomicAdd round trip per survivor inside the
          // drain would outlast the tile period.  entry = score | column-in-tile | both-directions flags.
          if (d_hit | t_hit) {
            const unsigned long long e8 = ((unsigned long long)__float_as_uint(a * p.descale) << 32) |
                                          ((unsigned long long)cl << 2) | (d_hit ? 1ull : 0ull) | (t_hit ? 2ull : 0ull);
            if (n_hit < kSymHitSlots) {
              hits[n_hit * 32 + lane] = e8;
              ++n_hit;
            } else {                                     // lane out of slots: append right away
              const float sc = a * p.descale;
              if (d_hit) sym_append(p, row, col0 + c, sc);
              if (t_hit) sym_append(p, col0 + c, (int)row, sc);
            }
          }
        }
      }
      // the accumulator is drained: hand it back to the MMA warp
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (leader) mbar_arrive(&tempty_bar[wg]);
        else mbar_arrive_cluster(tempty_remote);
      }
      // flush the parked survivors (every lane its own; the atomics of the 32 lanes overlap)
      const int max_hit = __reduce_max_sync(kFull, n_hit);
      for (int h = 0; h < max_hit; ++h) {
        if (h < n_hit) {
          const unsigned long long e8 = hits[h * 32 + lane];
          const float sc = __uint_as_float((uint32_t)(e8 >> 32));
          const int col = tj * BN + (int)((e8 >> 2) & 0xffu);
          if (e8 & 1ull) sym_append(p, row, col, sc);
          if (e8 & 2ull) sym_append(p, col, (int)row, sc);
        }
      }
    }
  }

  tcgen05_fence_before();
  cluster_sync_all();
  if (warp == kMmaWarp) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
}

// xs[m] = xh[(m * stride) mod N]: a low-discrepancy sample of the rows (stride ~ N / golden ratio, coprime
// with N), independent of how the caller ordered them.
__global__ void __launch_bounds__(256) sample_rows_kernel(const uint4* __restrict__ xh, int64_t N, int64_t row_u4,
                                                          int64_t n_sample, int64_t stride, uint4* __restrict__ xs) {
  const int64_t m = blockIdx.x;
  const int64_t src = (int64_t)(((unsigned long long)m * (unsigned long long)stride) % (unsigned long long)N);
  for (int64_t t = threadIdx.x; t < row_u4; t += blockDim.x) xs[m * row_u4 + t] = xh[src * row_u4 + t];
}

// tau[row] = r-th largest sample score of the row (over all of its prepass lists); -inf when the lists hold
// fewer than r entries.  One warp per row.  The prepass already published a threshold row_tau with at least
// keep >= r listed scores at or above it, so only those entries can matter: they are collected into shared
// memory (<= 512) and the r-th largest is found by a bitwise binary search on the order-preserving image
// (16 bits deep).
constexpr int kTauMax = 512;
constexpr int kTauWarps = 8;
__global__ void __launch_bounds__(kTauWarps * 32) sample_tau_kernel(const unsigned long long* __restrict__ cand,
                                                                   const int32_t* __restrict__ cand_cnt,
                                                                   const uint32_t* __restrict__ row_tau, int n_lists,
                                                                   int64_t n_rows, int r, float* __restrict__ tau,
                                                                   uint32_t* __restrict__ tau_ord,
                                                                   unsigned long long* __restrict__ cand2,
                                                                   int32_t* __restrict__ cand2_cnt, int cap2, int64_t row0) {
  // cand2 != nullptr (sample-first symmetric search): the columns of the prepass ARE rows of the matrix, so the listed
  // scores above tau are this row's candidates among them -- they go straight to the row's main list (row0 + row),
  // and the symmetric pass skips the sample blocks.
  __shared__ uint32_t s_o[kTauWarps][kTauMax];
  __shared__ uint32_t s_c[kTauWarps][kTauMax];          // columns of the collected scores (emit mode)
  const int w = threadIdx.x >> 5, lane = lane_id();
  const int64_t row = (int64_t)blockIdx.x * kTauWarps + w;
  if (row >= n_rows) return;
  const uint32_t floor_ord = row_tau[row];              // 0 = nothing published: keep everything
  int n = 0;
  for (int q = 0; q < n_lists; ++q) {
    const int c = min(cand_cnt[row * n_lists + q], kCap);
    const unsigned long long* src = cand + (row * n_lists + q) * (int64_t)kCap;
    for (int base = 0; base < c; base += 32) {
      const int t = base + lane;
      uint32_t o = 0;
      unsigned long long e = 0ull;
      if (t < c) {
        e = src[t];
        o = float_ord(__uint_as_float((uint32_t)(e >> 32)));
      }
      const bool in = t < c && o >= floor_ord;
      const unsigned b = __ballot_sync(kFull, in);
      const int pos = n + __popc(b & ((1u << lane) - 1u));
      if (in && pos < kTauMax) {
        s_o[w][pos] = o;
        if (cand2) s_c[w][pos] = (uint32_t)e;
      }
      n += __popc(b);
    }
  }
  __syncwarp();
  const int m = min(n, kTauMax);                        // a truncated set can only lower the result: still valid
  // the top 16 bits of the image are plenty: a threshold rounded DOWN only lets a few more columns through.  Only as
  // many registers as m needs take part (with the published floors of the emit mode a row collects a few dozen scores).
  auto search = [&](auto per_tag) {
    constexpr int kPer = decltype(per_tag)::value;
    uint32_t o[kPer];
#pragma unroll
    for (int u = 0; u < kPer; ++u) {
      const int t = u * 32 + lane;
      o[u] = t < m ? s_o[w][t] : 0u;
    }
    uint32_t T_ = 0;
#pragma unroll 1
    for (int bit = 31; bit >= 16; --bit) {
      const uint32_t c2 = T_ | (1u << bit);
      int c = 0;
#pragma unroll
      for (int u = 0; u < kPer; ++u) c += o[u] >= c2;
      c = __reduce_add_sync(kFull, c);
      if (c >= r) T_ = c2;
    }
    return T_;
  };
  uint32_t T = m <= 64    ? search(std::integral_constant<int, 2>{})
               : m <= 192 ? search(std::integral_constant<int, 6>{})
                          : search(std::integral_constant<int, kTauMax / 32>{});
  bool ok = m >= r;
  if (cand2) {
    // The lists are complete only above the published floor (= the largest threshold any list of the row rejected with,
    // reid_knn_candidates_tc_abt publish_final), and the 16-bit search rounds T down -- possibly below the floor.
    // max(T, floor) keeps every score above it in the lists (also when the collection above was truncated): they are
    // swept once more and everything above the threshold goes to the main list.  (A floor that came from a lucky seed
    // can exceed the true r-th best: the row then gets fewer candidates than planned, never wrong ones.)
    T = (ok && T > floor_ord) ? T : floor_ord;
    ok = ok || floor_ord != 0u;          // fewer than r scores above the floor: the floor itself is the threshold
    // Nobody else appends to this row's main list while this kernel runs (the transposed appends of the prepass go to
    // SAMPLE rows and are launched after the sample rows' thresholds; the symmetric pass comes later), so the warp
    // owns the counter: positions from ballots, one plain update at the end.
    if (ok && n <= kTauMax) {            // the usual case: everything at or above the floor sits in shared memory
      const int base0 = cand2_cnt[row0 + row];
      int n_e = 0;
      for (int b0 = 0; b0 < m; b0 += 32) {
        const int t = b0 + lane;
        const bool hit = t < m && s_o[w][t] > T;
        const unsigned bal = __ballot_sync(kFull, hit);
        const int pos = base0 + n_e + __popc(bal & ((1u << lane) - 1u));
        if (hit && pos < cap2)
          cand2[(row0 + row) * cap2 + pos] =
              ((unsigned long long)__float_as_uint(ord_float(s_o[w][t])) << 32) | (unsigned long long)s_c[w][t];
        n_e += __popc(bal);
      }
      if (lane == 0) cand2_cnt[row0 + row] = base0 + n_e;
    } else if (ok) {
      const int base0 = cand2_cnt[row0 + row];
      int n_e = 0;
      for (int q = 0; q < n_lists; ++q) {
        const int c = min(cand_cnt[row * n_lists + q], kCap);
        const unsigned long long* src = cand + (row * n_lists + q) * (int64_t)kCap;
        for (int b0 = 0; b0 < c; b0 += 32) {
          const int t = b0 + lane;
          const unsigned long long e = t < c ? src[t] : 0ull;
          const bool hit = t < c && float_ord(__uint_as_float((uint32_t)(e >> 32))) > T;
          const unsigned bal = __ballot_sync(kFull, hit);
          const int pos = base0 + n_e + __popc(bal & ((1u << lane) - 1u));
          if (hit && pos < cap2) cand2[(row0 + row) * cap2 + pos] = e;
          n_e += __popc(bal);
        }
      }
      if (lane == 0) cand2_cnt[row0 + row] = base0 + n_e;
    }
  }
  if (lane == 0) {
    tau[row] = ok ? ord_float(T) : -INFINITY;
    tau_ord[row] = ok ? T : 0u;
  }
}

// Provisional threshold of the non-sample rows in the sample-first layout: tau' = the smallest of the sample rows'
// thresholds tau_ord[0, m) (a row that scores like the weakest sample row still finds r sample scores above it),
// written to tau[m, N) and tau_ord[m, N).  Every block finds the minimum and writes its grid-stride share.
constexpr int kFloorThreads = 1024;
__global__ void __launch_bounds__(kFloorThreads) tau_floor_kernel(float* __restrict__ tau, uint32_t* __restrict__ tau_ord,
                                                                  int64_t m, int64_t N) {
  __shared__ uint32_t s_min;
  if (threadIdx.x == 0) s_min = 0xffffffffu;
  uint32_t v = 0xffffffffu;
  for (int64_t i = threadIdx.x; i < m; i += kFloorThreads) v = min(v, tau_ord[i]);
  v = __reduce_min_sync(kFull, v);
  __syncthreads();
  if (lane_id() == 0) atomicMin(&s_min, v);
  __syncthreads();
  const uint32_t T = s_min;
  const float t = T ? ord_float(T) : -INFINITY;
  for (int64_t i = m + (int64_t)blockIdx.x * kFloorThreads + threadIdx.x; i < N; i += (int64_t)gridDim.x * kFloorThreads) {
    tau[i] = t;
    tau_ord[i] = T;
  }
}

// Threshold of a non-sample row in the sample-first layout, after the symmetric kernel has run the sample block column
// with tau[row] = tau' (tau_floor_kernel): the row's list then holds exactly its sample scores above tau', and
//   tau[row] = max(tau', r-th best of them)   when at least r are listed,   tau' otherwise.
// Sound either way: an unlisted sample column scored <= tau' <= tau[row].  One warp per row; as in sample_tau_kernel the
// search resolves the top 16 bits of the image (rounded down: a few more columns get through).  Only the first
// min(count, kListTauMax) entries are read: a subset can only lower the r-th best (an overflowed list un-certifies the
// row in any case).
constexpr int kListTauMax = 1024;
__global__ void __launch_bounds__(kTauWarps * 32) list_tau_kernel(const unsigned long long* __restrict__ cand,
                                                                 const int32_t* __restrict__ cand_cnt, int cap, int64_t row0,
                                                                 int64_t n_rows, int r, float* __restrict__ tau,
                                                                 uint32_t* __restrict__ tau_ord) {
  const int w = threadIdx.x >> 5, lane = lane_id();
  const int64_t row = row0 + (int64_t)blockIdx.x * kTauWarps + w;
  if (row >= row0 + n_rows) return;
  const uint32_t floor_ord = tau_ord[row];
  const int n = min(min(cand_cnt[row], cap), kListTauMax);
  if (n < r) return;                                  // tau' stays
  const unsigned long long* src = cand + row * (int64_t)cap;
  auto search = [&](auto per_tag) {
    constexpr int kPer = decltype(per_tag)::value;
    uint32_t o[kPer];
#pragma unroll
    for (int u = 0; u < kPer; ++u) {
      const int t = u * 32 + lane;
      o[u] = t < n ? float_ord(__uint_as_float((uint32_t)(src[t] >> 32))) : 0u;
    }
    uint32_t T_ = 0;
#pragma unroll 1
    for (int bit = 31; bit >= 16; --bit) {
      const uint32_t c2 = T_ | (1u << bit);
      int c = 0;
#pragma unroll
      for (int u = 0; u < kPer; ++u) c += o[u] >= c2;
      c = __reduce_add_sync(kFull, c);
      if (c >= r) T_ = c2;
    }
    return T_;
  };
  const uint32_t T = n <= 64 ? search(std::integral_constant<int, 2>{})
                     : n <= 256 ? search(std::integral_constant<int, 8>{})
                                : search(std::integral_constant<int, kListTauMax / 32>{});
  if (lane == 0 && T > floor_ord) {
    tau[row] = ord_float(T);
    tau_ord[row] = T;
  }
}

}  // namespace tc
}  // namespace reid

extern "C" {

int reid_features_sample(const void* xh, int64_t N, int64_t D, int64_t n_sample, int64_t stride, void* xs, void* stream) {
  using namespace reid;
  REID_CHECK_ARG(xh && xs && N > 0 && D > 0 && D % 8 == 0 && n_sample > 0 && stride > 0, "reid_features_sample: bad arguments");
  REID_CHECK_ARG((((uintptr_t)xh | (uintptr_t)xs) & 15) == 0, "reid_features_sample: operands must be 16-byte aligned");
  tc::sample_rows_kernel<<<(unsigned)n_sample, 256, 0, (cudaStream_t)stream>>>((const uint4*)xh, N, D / 8, n_sample, stride,
                                                                             (uint4*)xs);
  REID_LAUNCH_CHECK();
  return REID_OK;
}

int reid_knn_sample_tau(const uint64_t* cand, const int32_t* cand_cnt, const uint32_t* row_tau, int n_lists, int64_t n_rows,
                        int r, float* tau, uint32_t* tau_ord, void* stream) {
  return reid_knn_sample_tau_emit(cand, cand_cnt, row_tau, n_lists, n_rows, r, tau, tau_ord, nullptr, nullptr, 0, 0, stream);
}

int reid_knn_sample_tau_emit(const uint64_t* cand, const int32_t* cand_cnt, const uint32_t* row_tau, int n_lists, int64_t n_rows,
                             int r, float* tau, uint32_t* tau_ord, uint64_t* cand_main, int32_t* cand_main_cnt, int cap_main,
                             int64_t row0, void* stream) {
  using namespace reid;
  REID_CHECK_ARG(!cand_main || (cand_main_cnt && cap_main >= 1 && row0 >= 0), "reid_knn_sample_tau_emit: bad main lists");
  REID_CHECK_ARG(cand && cand_cnt && row_tau && tau && tau_ord && n_lists >= 1 && n_rows >= 0 && r >= 1,
                 "reid_knn_sample_tau: bad arguments");
  if (n_rows == 0) return REID_OK;
  tc::sample_tau_kernel<<<(unsigned)((n_rows + tc::kTauWarps - 1) / tc::kTauWarps), tc::kTauWarps * 32, 0, (cudaStream_t)stream>>>(
      (const unsigned long long*)cand, cand_cnt, row_tau, n_lists, n_rows, r, tau, tau_ord, (unsigned long long*)cand_main,
      cand_main_cnt, cap_main, row0);
  REID_LAUNCH_CHECK();
  return REID_OK;
}

int reid_upload_rows_strided(void* dst, const void* src_host, size_t row_bytes, size_t src_pitch_bytes, int64_t n_rows,
                             void* stream) {
  using namespace reid;
  REID_CHECK_ARG(dst && src_host && row_bytes > 0 && src_pitch_bytes >= row_bytes && n_rows >= 0,
                 "reid_upload_rows_strided: bad arguments");
  if (n_rows == 0) return REID_OK;
  REID_CUDA(cudaMemcpy2DAsync(dst, row_bytes, src_host, src_pitch_bytes, row_bytes, (size_t)n_rows, cudaMemcpyHostToDevice,
                              (cudaStream_t)stream));
  return REID_OK;
}

static int launch_sym(int nb, const void* xh, int64_t N, int64_t D, int scale_log2, const float* tau, const int32_t* units,
                      int64_t n_units, int cap, uint64_t* cand, int32_t* cand_cnt, int reset_counts, void* stream) {
  using namespace reid;
  REID_CHECK_ARG(xh && tau && units && cand && cand_cnt, "reid_knn_candidates_sym: NULL pointer");
  REID_CHECK_ARG(N > 0 && N < (1ll << 31) && D > 0 && D % tc::BK == 0, "reid_knn_candidates_sym: need D %% 64 == 0 (D=%lld)",
                 (long long)D);
  REID_CHECK_ARG(((uintptr_t)xh & 15) == 0, "reid_knn_candidates_sym: xh must be 16-byte aligned");
  REID_CHECK_ARG(n_units > 0 && n_units < (1ll << 30) && cap >= 1, "reid_knn_candidates_sym: bad tile list / capacity");
  REID_CHECK_ARG(num_sms() >= 2, "reid_knn_candidates_sym: needs CTA pairs");
  cudaStream_t st = (cudaStream_t)stream;
  CUtensorMap tmap;
  int rc = tc::make_tmap_rows128(&tmap, xh, N, D);
  if (rc != REID_OK) return rc;
  tc::SymParams p;
  p.N = N;
  p.num_k_blocks = (int)(D / tc::BK);
  p.n_units = (int)n_units;
  p.tiles = units;
  p.tau = tau;
  p.scale2 = ldexpf(1.0f, 2 * scale_log2);
  p.descale = ldexpf(1.0f, -2 * scale_log2);
  p.cap = cap;
  p.cand = (unsigned long long*)cand;
  p.cand_cnt = cand_cnt;
  p.dbg = dev_env("REID_TC_DEBUG", 0);
  if (reset_counts) REID_CUDA(cudaMemsetAsync(cand_cnt, 0, sizeof(int32_t) * (size_t)N, st));
  const int slots = num_sms() / 2;
  const int grid = (int)(n_units < slots ? n_units : slots) * 2;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(tc::kThreads);
  cfg.stream = st;
  cfg.dynamicSmemBytes = nb == 2 ? tc::SymCfg<2>::kSmem : tc::SymCfg<1>::kSmem;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (nb == 2) {
    REID_CUDA(cudaFuncSetAttribute(tc::simsym_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::SymCfg<2>::kSmem));
    REID_CUDA(cudaLaunchKernelEx(&cfg, tc::simsym_kernel<2>, tmap, p));
  } else {
    REID_CUDA(cudaFuncSetAttribute(tc::simsym_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::SymCfg<1>::kSmem));
    REID_CUDA(cudaLaunchKernelEx(&cfg, tc::simsym_kernel<1>, tmap, p));
  }
  REID_LAUNCH_CHECK();
  return REID_OK;
}

int reid_knn_candidates_sym(const void* xh, int64_t N, int64_t D, int scale_log2, const float* tau, const int32_t* tiles,
                            int64_t n_tiles, int cap, uint64_t* cand, int32_t* cand_cnt, int reset_counts, void* stream) {
  return launch_sym(1, xh, N, D, scale_log2, tau, tiles, n_tiles, cap, cand, cand_cnt, reset_counts, stream);
}

int reid_knn_candidates_sym_wide(const void* xh, int64_t N, int64_t D, int scale_log2, const float* tau, const int32_t* units,
                                 int64_t n_units, int cap, uint64_t* cand, int32_t* cand_cnt, int reset_counts, void* stream) {
  return launch_sym(2, xh, N, D, scale_log2, tau, units, n_units, cap, cand, cand_cnt, reset_counts, stream);
}

int reid_knn_candidates_sym_tiles(const void* xh, int64_t N, int64_t D, int scale_log2, const float* tau, const int32_t* tiles,
                                  int64_t n_tiles, int cap, uint64_t* cand, int32_t* cand_cnt, int reset_counts, void* stream) {
  return launch_sym(1, xh, N, D, scale_log2, tau, tiles, n_tiles, cap, cand, cand_cnt, reset_counts, stream);
}

int reid_knn_tau_floor(float* tau, uint32_t* tau_ord, int64_t m, int64_t N, void* stream) {
  using namespace reid;
  REID_CHECK_ARG(tau && tau_ord, "reid_knn_tau_floor: NULL pointer");
  REID_CHECK_ARG(m >= 1 && m <= N, "reid_knn_tau_floor: need 1 <= m <= N (m=%lld N=%lld)", (long long)m, (long long)N);
  if (m == N) return REID_OK;
  const int64_t blocks = (N - m + 4 * tc::kFloorThreads - 1) / (4 * tc::kFloorThreads);
  tc::tau_floor_kernel<<<(unsigned)(blocks < 148 ? blocks : 148), tc::kFloorThreads, 0, (cudaStream_t)stream>>>(tau, tau_ord, m,
                                                                                                             N);
  REID_LAUNCH_CHECK();
  return REID_OK;
}

int reid_knn_list_tau(const uint64_t* cand, const int32_t* cand_cnt, int cap, int64_t row0, int64_t n_rows, int r, float* tau,
                      uint32_t* tau_ord, void* stream) {
  using namespace reid;
  REID_CHECK_ARG(cand && cand_cnt && tau && tau_ord, "reid_knn_list_tau: NULL pointer");
  REID_CHECK_ARG(cap >= 1 && row0 >= 0 && n_rows >= 0 && r >= 1, "reid_knn_list_tau: bad arguments (cap=%d row0=%lld n_rows=%lld r=%d)",
                 cap, (long long)row0, (long long)n_rows, r);
  if (n_rows == 0) return REID_OK;
  tc::list_tau_kernel<<<(unsigned)((n_rows + tc::kTauWarps - 1) / tc::kTauWarps), tc::kTauWarps * 32, 0, (cudaStream_t)stream>>>(
      (const unsigned long long*)cand, cand_cnt, cap, row0, n_rows, r, tau, tau_ord);
  REID_LAUNCH_CHECK();
  return REID_OK;
}
}
