// a1 (first half) -- the N x N similarity contraction on the 5th-generation tensor cores, fused
// with a per-row running top-K selection (replaces the SGEMM + block-select inside faiss
// IndexFlatL2 / GpuIndexFlatL2.search, utils/faiss_rerank.py:39-62).
//
//   S = Xh . Xh^T,  Xh = fp16(2^s X)  (N x D, K-major for both operands)
//
// One persistent CTA per SM (kCtas = 2: CTA pairs, tcgen05 cta_group::2), warp-specialised:
//   warp 0      TMA producer : cp.async.bulk.tensor 128B-swizzled 64-wide K slices of the CTA's 128 query rows
//                              (A) and of its share of the 256-row column tile (B) into a 4 / 6-stage
//                              shared-memory ring
//   warp 1      MMA issuer   : one elected lane (leader CTA) issues tcgen05.mma (M = 128 * kCtas, N = 256, K = 16,
//                              fp16 -> fp32) into one of two 256-column TMEM accumulators; tcgen05.commit frees
//                              the ring slot / publishes the accumulator
//   warps 2..9  epilogue     : two groups of four warps, group g drains accumulator g (every other column tile):
//                              tcgen05.ld 32 columns at a time; thread <-> query row; every score is compared
//                              with the row's running threshold tau and survivors are appended to the row's
//                              candidate list (global scratch).  The accumulator is handed back first; lists
//                              that could overflow during the next tile are then compacted warp-cooperatively
//                              to the best K (bitwise binary search, ballot prefix sums) and tau is raised and
//                              published per row, so after warm-up almost every score dies on a single compare.
// A work unit is (128 * kCtas-row query tile) x (one of n_splits column ranges); units are dealt round-robin,
// column-range major so that concurrently running CTAs stream the same B tiles out of L2.
// The scores are only candidates: knn_rescore.cu re-scores them exactly and certifies the result.
// Since the symmetric search (simgemm_sym.cu) this kernel serves N < 8192, k > 32, the row shards of the "rows"
// multi-GPU plan, and -- with a negative `keep` -- the sampling prepass that finds the symmetric search's thresholds.
#include <stdlib.h>

#include "tc_ptx.cuh"

namespace reid {
namespace tc {

// Cooperative compaction of one row's candidate list (n entries at `list`, n <= kCap) to (at least) its
// best `keep` entries.  Entry = (score bits << 32) | column.  The threshold is found by a bitwise binary
// search on the order-preserving integer image of the scores.  kBits = 32 resolves it exactly (exactly
// `keep` survivors, ties by list position); kBits = 16 stops at the top 16 bits, which can only LOWER the
// threshold: a few more than `keep` survive, never fewer -- half the dependent REDUX chain, used for the
// in-flight compactions where only the trend of tau matters.  Returns the new tau and the survivor count.
template <int kBits>
__device__ __forceinline__ float warp_compact(unsigned long long* list, int n, int keep, int& n_out) {
  const int lane = lane_id();
  constexpr int kPer = kCap / 32;
  unsigned long long e[kPer];
  uint32_t o[kPer];
  __syncwarp();  // the owner lane's appends must be visible to the whole warp
#pragma unroll
  for (int j = 0; j < kPer; ++j) {
    const int i = j * 32 + lane;
    e[j] = i < n ? list[i] : 0ull;
    o[j] = i < n ? float_ord(__uint_as_float((uint32_t)(e[j] >> 32))) : 0u;  // 0 sorts below every real score
  }
  __syncwarp();
  // largest T (on the searched bits) with #{o >= T} >= keep
  uint32_t T = 0;
#pragma unroll 1
  for (int bit = 31; bit >= 32 - kBits; --bit) {
    const uint32_t cand = T | (1u << bit);
    int c = 0;
#pragma unroll
    for (int j = 0; j < kPer; ++j) c += o[j] >= cand;
    c = __reduce_add_sync(kFull, c);
    if (c >= keep) T = cand;
  }
  int n_gt = 0;
#pragma unroll
  for (int j = 0; j < kPer; ++j) n_gt += o[j] > T;
  n_gt = __reduce_add_sync(kFull, n_gt);
  // exact search: n_gt < keep and the ties at T fill the quota; coarse search: everything >= T stays
  const int quota = kBits == 32 ? keep - n_gt : 0x7fffffff;
  int eq_seen = 0, kept_seen = 0;
  const unsigned lt = (1u << lane) - 1u;
#pragma unroll
  for (int j = 0; j < kPer; ++j) {
    const bool gt = o[j] > T, eq = o[j] == T && (j * 32 + lane) < n;
    const unsigned beq = __ballot_sync(kFull, eq);
    const bool keep_me = gt || (eq && eq_seen + __popc(beq & lt) < quota);
    const unsigned bk = __ballot_sync(kFull, keep_me);
    if (keep_me) list[kept_seen + __popc(bk & lt)] = e[j];
    eq_seen += __popc(beq);
    kept_seen += __popc(bk);
  }
  __syncwarp();
  n_out = kept_seen;
  return ord_float(T);
}

struct Params {
  int64_t N;
  int64_t row_begin, row_end;
  int num_k_blocks;     // D / 64
  int n_mblk;           // query tiles in the shard
  int n_splits;
  int n_tiles;          // ceil(N / 256) column tiles
  int keep;             // K: entries kept per (row, split)
  float descale;        // 2^(-2 s)
  unsigned long long* cand;   // [(rows) x n_splits x kCap]
  int32_t* cand_cnt;          // [(rows) x n_splits]
  uint32_t* row_tau;          // [rows] shared rejection threshold per query row (order-preserving image), 0 = none
  // transposed direction (sample-first symmetric search, knn_tc._candidates_sym_sf): the columns are the SAMPLE rows,
  // whose own thresholds are known already; every score above its column's threshold is appended to that sample row's
  // main list (entry column = this query row) -- the tiles (sample block, other block) of the symmetric pass are then
  // covered by this prepass and skipped there.  tau_col == nullptr: off.
  const float* tau_col;       // [N] threshold per column (descaled score units)
  unsigned long long* cand2;  // [N x cap2] main lists of the column rows
  int32_t* cand2_cnt;         // [N]
  int cap2;
  int publish_final;          // every list publishes its FINAL rejection threshold (boot seeds included) in row_tau, so that
                              // row_tau ends up >= every threshold any list of the row ever rejected with: what
                              // reid_knn_sample_tau_emit needs to hand the listed scores on as complete candidate sets
  int boot;                   // sampling prepass: seed tau from the first 32 scores of a unit (see the epilogue)
  int dbg;                    // developer switch (REID_TC_DEBUG): 1 = epilogue skips TMEM reads, 2 = reads but no selection, 4 = no TMA
};

template <int kCtas>
struct Cfg {
  // per-CTA bytes of one pipeline stage: its 128 query rows of A + its share of the 256-row B tile
  static constexpr int kBRows = BN / kCtas;
  static constexpr int kBBytes = kBRows * BK * 2;
  static constexpr int kStage = kATileBytes + kBBytes;      // 48 KB (1 CTA) / 32 KB (pair)
  static constexpr int kNumStages = kCtas == 1 ? 4 : 6;
  static constexpr int kTauColBytes = 2 * BN * 4;            // column thresholds, one buffer per epilogue group
  static constexpr int kHitSlots = 8;                        // parked transposed survivors per lane and tile
  static constexpr int kHitBytes = 8 * kHitSlots * 32 * 8;   // 8 epilogue warps x slots x lanes x 8 B
  static constexpr int kSmem = kNumStages * kStage + 1024 /*align*/ + 256 /*barriers*/ + kTauColBytes + kHitBytes;
};

// kCtas = 1: one CTA per 128-row tile (tcgen05.mma.cta_group::1, M = 128).
// kCtas = 2: a CTA pair per 256-row tile (cta_group::2, M = 256): each CTA stages its own 128 query rows
//            and HALF of the column tile, so the B operand is fetched from L2 once per pair; the leader
//            CTA issues the MMAs, both CTAs run a TMA producer and the top-K epilogue on their own
//            128 accumulator lanes.
template <int kCtas>
__global__ void __launch_bounds__(kThreads, 1) simtopk_kernel(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ CUtensorMap tmap_b,
                                                                  const Params p) {
  using C = Cfg<kCtas>;
  constexpr int kNumStages = C::kNumStages;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* full_bar = (uint64_t*)(smem + kNumStages * C::kStage);
  uint64_t* empty_bar = full_bar + kNumStages;
  uint64_t* tfull_bar = empty_bar + kNumStages;   // [2] accumulator ready
  uint64_t* tempty_bar = tfull_bar + 2;           // [2] accumulator drained (lives in the leader CTA)
  uint32_t* tmem_slot = (uint32_t*)(tempty_bar + 2);
  float* s_tauc = (float*)(smem + kNumStages * C::kStage + 256);                                                  // [2][BN]
  unsigned long long* s_hits = (unsigned long long*)(smem + kNumStages * C::kStage + 256 + C::kTauColBytes);     // [8][slots][32]

  const int warp = threadIdx.x >> 5, lane = lane_id();
  const uint32_t cta_rank = kCtas == 2 ? cluster_ctarank() : 0u;
  const bool leader = cta_rank == 0;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_b) : "memory");
    for (int s = 0; s < kNumStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull_bar[a], 1);
      mbar_init(&tempty_bar[a], 4 * kCtas);   // the 4 warps of the owning epilogue group, in every CTA of the pair
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {  // TMEM: all 512 columns = two 128 x 256 fp32 accumulators (per CTA)
    if (kCtas == 1) {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    } else {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
    }
  }
  tcgen05_fence_before();
  if (kCtas == 2) cluster_sync_all(); else __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int n_units = p.n_mblk * p.n_splits;         // n_mblk counts (128 * kCtas)-row tiles
  const int unit0 = blockIdx.x / kCtas, unit_step = gridDim.x / kCtas;

  if (warp == 0) {
    // ------------------------------ TMA producer ------------------------------
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int u = unit0; u < n_units; u += unit_step) {
        const int split = u / p.n_mblk, mblk = u % p.n_mblk;
        const int t0 = (int)((int64_t)p.n_tiles * split / p.n_splits), t1 = (int)((int64_t)p.n_tiles * (split + 1) / p.n_splits);
        const int m_row = (int)p.row_begin + mblk * (BM * kCtas) + (int)cta_rank * BM;
        for (int t = t0; t < t1; ++t) {
          for (int kb = 0; kb < p.num_k_blocks; ++kb) {
            mbar_wait(&empty_bar[stage], phase ^ 1);
            uint8_t* a_dst = smem + stage * C::kStage;
            uint8_t* b_dst = a_dst + kATileBytes;
            if (REID_DBG(p) & 4) {
              if (kCtas == 1 || leader) mbar_arrive(&full_bar[stage]);
            } else if (kCtas == 1) {
              mbar_expect_tx(&full_bar[stage], C::kStage);
              tma_load_2d(a_dst, &tmap, &full_bar[stage], kb * BK, m_row);
              tma_load_2d(b_dst, &tmap_b, &full_bar[stage], kb * BK, t * BN);
              tma_load_2d(b_dst + kATileBytes, &tmap_b, &full_bar[stage], kb * BK, t * BN + 128);
            } else {
              // all bytes of the pair are accounted on the leader's barrier
              if (leader) mbar_expect_tx(&full_bar[stage], 2 * C::kStage);
              const uint32_t lbar = mapa_u32(smem_u32(&full_bar[stage]), 0);
              tma_load_2d_pair(a_dst, &tmap, lbar, kb * BK, m_row);
              tma_load_2d_pair(b_dst, &tmap_b, lbar, kb * BK, t * BN + (int)cta_rank * 128);
            }
            if (++stage == kNumStages) {
              stage = 0;
              phase ^= 1;
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------ MMA issuer (leader CTA only) ----------------
    if (lane == 0 && leader) {
      constexpr uint32_t idesc = make_idesc(BM * kCtas, BN);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int u = unit0; u < n_units; u += unit_step) {
        const int split = u / p.n_mblk;
        const int t0 = (int)((int64_t)p.n_tiles * split / p.n_splits), t1 = (int)((int64_t)p.n_tiles * (split + 1) / p.n_splits);
        for (int t = t0; t < t1; ++t) {
          mbar_wait(&tempty_bar[acc], acc_phase ^ 1);   // every epilogue warp of the pair has drained this accumulator
          tcgen05_fence_after();
          const uint32_t tmem_c = tmem_base + (uint32_t)(acc * BN);
          for (int kb = 0; kb < p.num_k_blocks; ++kb) {
            mbar_wait(&full_bar[stage], phase);
            tcgen05_fence_after();
            const uint32_t a_addr = smem_u32(smem + stage * C::kStage);
            const uint32_t b_addr = a_addr + kATileBytes;
#pragma unroll
            for (int k = 0; k < BK / UMMA_K; ++k) {
              const uint64_t da = make_smem_desc(a_addr + k * UMMA_K * 2);
              const uint64_t db = make_smem_desc(b_addr + k * UMMA_K * 2);
              if (kCtas == 1) umma_f16(tmem_c, da, db, idesc, (kb | k) != 0);
              else umma_f16_pair(tmem_c, da, db, idesc, (kb | k) != 0);
            }
            if (kCtas == 1) umma_commit(&empty_bar[stage]); else umma_commit_pair(&empty_bar[stage]);
            if (++stage == kNumStages) {
              stage = 0;
              phase ^= 1;
            }
          }
          if (kCtas == 1) umma_commit(&tfull_bar[acc]); else umma_commit_pair(&tfull_bar[acc]);
          if (++acc == 2) {
            acc = 0;
            acc_phase ^= 1;
          }
        }
      }
    }
  } else {
    // ------------------------------ epilogue: fused running top-K ----------------
    // Two epilogue warpgroups: group g drains accumulator g (every other column tile), so each has two
    // MMA tile periods for its drain + list maintenance.  Every (row, column range, group) owns a list.
    const int wg = (warp - 2) >> 2;
    const int quarter = warp & 3;                       // TMEM lanes this warp may read
    const int r_in_tile = (int)cta_rank * BM + quarter * 32 + lane;
    const uint32_t tempty_remote = kCtas == 2 ? mapa_u32(smem_u32(&tempty_bar[wg]), 0) : 0u;
    const int n_lists = p.n_splits * 2;
    uint32_t acc_phase = 0;
    int tile_ctr = 0;                                   // running tile count of this CTA == the MMA warp's
    for (int u = unit0; u < n_units; u += unit_step) {
      const int split = u / p.n_mblk, mblk = u % p.n_mblk;
      const int t0 = (int)((int64_t)p.n_tiles * split / p.n_splits), t1 = (int)((int64_t)p.n_tiles * (split + 1) / p.n_splits);
      const int64_t lrow = (int64_t)mblk * (BM * kCtas) + r_in_tile;     // local row in the shard
      const bool row_ok = p.row_begin + lrow < p.row_end;
      const int64_t list_id = (row_ok ? lrow : 0) * n_lists + split * 2 + wg;
      unsigned long long* list = p.cand + list_id * (int64_t)kCap;
      float tau = row_ok ? -INFINITY : INFINITY;
      int cnt = 0;
      volatile uint32_t* my_tau = p.row_tau + (row_ok ? lrow : 0);
      for (int t = t0; t < t1; ++t, ++tile_ctr) {
        if ((tile_ctr & 1) != wg) continue;
        // Any threshold published for this row -- by the other epilogue group, or by a CTA that already
        // swept another column range -- is a valid rejection threshold here too: `keep` columns with a
        // higher score are known to exist somewhere.  Picking it up removes most of the warm-up.
        {
          const uint32_t g = *my_tau;
          if (g && row_ok) tau = fmaxf(tau, ord_float(g));
        }
        float* tauc = s_tauc + wg * BN;
        unsigned long long* hits = s_hits + (size_t)(warp - 2) * C::kHitSlots * 32;
        int n_hit = 0;
        if (p.tau_col) {                                  // thresholds of this tile's columns (uniform branch)
          __syncwarp();
          asm volatile("bar.sync %0, 128;" ::"r"(1 + wg) : "memory");        // the previous tile's readers are done
          const int gt = ((warp - 2) & 3) * 32 + lane;
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const int c = gt + h * 128;
            const int64_t col = (int64_t)t * BN + c;
            tauc[c] = col < p.N ? p.tau_col[col] : INFINITY;
          }
          asm volatile("bar.sync %0, 128;" ::"r"(1 + wg) : "memory");
        }
        mbar_wait(&tfull_bar[wg], acc_phase);
        acc_phase ^= 1;
        tcgen05_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(wg * BN);
#pragma unroll 1
        for (int ch = 0; ch < BN / 32; ++ch) {
          if (REID_DBG(p) & 1) break;
          uint32_t v[32];
          tmem_ld_32x32b_x32(taddr + ch * 32, v);
          const int col0 = t * BN + ch * 32;
          if (p.tau_col && row_ok) {                      // transposed direction: score against the column's threshold
            const float4* tc4 = reinterpret_cast<const float4*>(tauc + ch * 32);
            unsigned hit = 0;
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              const float4 t4 = tc4[q];
              hit |= (unsigned)(__uint_as_float(v[4 * q]) * p.descale > t4.x) << (4 * q);
              hit |= (unsigned)(__uint_as_float(v[4 * q + 1]) * p.descale > t4.y) << (4 * q + 1);
              hit |= (unsigned)(__uint_as_float(v[4 * q + 2]) * p.descale > t4.z) << (4 * q + 2);
              hit |= (unsigned)(__uint_as_float(v[4 * q + 3]) * p.descale > t4.w) << (4 * q + 3);
            }
            while (hit) {                                 // rare: about r / m of the scores
              const int c = __ffs(hit) - 1;
              hit &= hit - 1;
              float a = 0.f;
#pragma unroll
              for (int e = 0; e < 32; ++e) a = e == c ? __uint_as_float(v[e]) : a;
              const float sc = a * p.descale;
              const int64_t col = col0 + c;               // < N: columns beyond N carry an infinite threshold
              if (n_hit < C::kHitSlots) {                 // parked; appended after the accumulator has been handed back
                hits[n_hit * 32 + lane] = ((unsigned long long)__float_as_uint(sc) << 32) | (unsigned long long)(ch * 32 + c);
                ++n_hit;
              } else {
                const int pos = atomicAdd(p.cand2_cnt + col, 1);
                if (pos < p.cap2)
                  p.cand2[col * p.cap2 + pos] = ((unsigned long long)__float_as_uint(sc) << 32) | (uint32_t)(p.row_begin + lrow);
              }
            }
          }
          if (p.boot && cnt == 0 && tau == -INFINITY) {
            // Sampling prepass (reid_knn_sample_tau wants the r-th best of a few thousand scores, r ~ 16): instead
            // of appending the first tiles unfiltered -- uncoalesced 8-byte stores that outlast the MMA -- seed the
            // threshold with the 5th largest of the first 32 scores, a value about 5/32 of all scores beat (the chance
            // that fewer than r of a list's ~1000 scores beat it is ~1e-5).  A seed
            // that lands too high only makes the final threshold lower (more candidates), never wrong.
            float m1 = -INFINITY, m2 = -INFINITY, m3 = -INFINITY, m4 = -INFINITY, m5 = -INFINITY;
#pragma unroll
            for (int c = 0; c < 32; ++c) {
              float s = __uint_as_float(v[c]) * p.descale, lo;
              lo = fminf(m1, s), m1 = fmaxf(m1, s), s = lo;
              lo = fminf(m2, s), m2 = fmaxf(m2, s), s = lo;
              lo = fminf(m3, s), m3 = fmaxf(m3, s), s = lo;
              lo = fminf(m4, s), m4 = fmaxf(m4, s), s = lo;
              m5 = fmaxf(m5, s);
            }
            tau = m5;
          }
          if (REID_DBG(p) & 2) {
            float m = 0.f;
#pragma unroll
            for (int c = 0; c < 32; ++c) m = fmaxf(m, __uint_as_float(v[c]));
            if (m == 123.456f) list[cnt++] = 1ull;
          } else if (col0 + 32 <= p.N) {
#pragma unroll
            for (int c = 0; c < 32; ++c) {
              const float s = __uint_as_float(v[c]) * p.descale;
              if (s > tau) list[cnt++] = ((unsigned long long)__float_as_uint(s) << 32) | (uint32_t)(col0 + c);
            }
          } else {
#pragma unroll
            for (int c = 0; c < 32; ++c) {
              const float s = __uint_as_float(v[c]) * p.descale;
              if (s > tau && col0 + c < p.N) list[cnt++] = ((unsigned long long)__float_as_uint(s) << 32) | (uint32_t)(col0 + c);
            }
          }
        }
        // the accumulator is drained: hand it back to the MMA warp before doing any list maintenance
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (kCtas == 1 || leader) mbar_arrive(&tempty_bar[wg]);
          else mbar_arrive_cluster(tempty_remote);
        }
        if (p.tau_col) {                                  // flush the parked transposed survivors
          const int max_hit = __reduce_max_sync(kFull, n_hit);
          for (int h = 0; h < max_hit; ++h) {
            if (h < n_hit) {
              const unsigned long long e8 = hits[h * 32 + lane];
              const int64_t col = (int64_t)t * BN + (int)(e8 & 0xffu);
              const int pos = atomicAdd(p.cand2_cnt + col, 1);
              if (pos < p.cap2)
                p.cand2[col * p.cap2 + pos] = (e8 & 0xffffffff00000000ull) | (uint32_t)(p.row_begin + lrow);
            }
          }
        }
        // a tile appends at most BN entries: lists that could overflow during the next tile are compacted
        // now (coarse threshold), one row at a time, while the tensor core works on the other accumulator
        unsigned need = __ballot_sync(kFull, cnt > kCap - BN);
        while (need) {
          const int src = __ffs(need) - 1;
          need &= need - 1;
          unsigned long long* l = (unsigned long long*)__shfl_sync(kFull, (unsigned long long)list, src);
          const int n = __shfl_sync(kFull, cnt, src);
          int kept;
          float nt = warp_compact<16>(l, n, p.keep, kept);
          if (kept > kCap - BN) nt = warp_compact<32>(l, kept, p.keep, kept);  // a flood of near-ties: resolve exactly
          if (lane == src) {
            tau = fmaxf(tau, nt);
            cnt = kept;
            atomicMax(p.row_tau + lrow, float_ord(tau));
          }
        }
      }
      // unit done: publish the count; the list is left untrimmed (<= kCap entries) -- knn_rescore.cu only
      // looks at entries above the row's final threshold
      if (row_ok) {
        p.cand_cnt[list_id] = cnt;
        if (p.publish_final && tau > -INFINITY) atomicMax(p.row_tau + lrow, float_ord(tau));
      }
    }
  }

  tcgen05_fence_before();
  if (kCtas == 2) cluster_sync_all(); else __syncthreads();
  if (warp == 1) {
    if (kCtas == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
    else asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
  }
}

__global__ void __launch_bounds__(256) to_half_kernel(const float* __restrict__ x, int64_t n_rows, int64_t D, float scale,
                                                      __half* __restrict__ xh, float* __restrict__ max_sqnorm,
                                                      const int32_t* __restrict__ src_row) {
  // warp per row, grid-stride: the launch is sized to the machine (no partial last wave of 8-row CTAs)
  for (int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); row < n_rows;
       row += (int64_t)gridDim.x * (blockDim.x >> 5)) {
  float ss = 0.f;
  float amax = 0.f;                                      // largest |x| of the row: an fp16 overflow check
  if ((D & 3) == 0 && ((((uintptr_t)x) | ((uintptr_t)xh)) & 15) == 0) {
    // 16-byte loads, 8-byte stores: the stage is a pure stream (4ND bytes in, 2ND out)
    const int64_t srow = src_row ? (int64_t)src_row[row] : row;      // sample-first layout of the symmetric search
    const float4* src = reinterpret_cast<const float4*>(x + srow * D);
    uint2* dst = reinterpret_cast<uint2*>(xh + row * D);
    // eight independent 16-byte loads per lane in flight (4 KB per warp) before the first use: the stream is bound by
    // bytes in flight, not by the conversions.  ss is accumulated in ascending element order, batch or not.
    const int64_t n4 = D >> 2;
    constexpr int kBatch = 8;
    for (int64_t base = 0; base < n4; base += 32 * kBatch) {
      float4 v[kBatch];
#pragma unroll
      for (int u = 0; u < kBatch; ++u) {
        const int64_t d4 = base + u * 32 + lane_id();
        v[u] = d4 < n4 ? __ldcs(src + d4) : make_float4(0.f, 0.f, 0.f, 0.f);   // streamed once: keep it out of L2's way
      }
#pragma unroll
      for (int u = 0; u < kBatch; ++u) {
        const int64_t d4 = base + u * 32 + lane_id();
        if (d4 < n4) {
          ss = fmaf(v[u].x, v[u].x, ss);
          ss = fmaf(v[u].y, v[u].y, ss);
          ss = fmaf(v[u].z, v[u].z, ss);
          ss = fmaf(v[u].w, v[u].w, ss);
          amax = fmaxf(amax, fmaxf(fmaxf(fabsf(v[u].x), fabsf(v[u].y)), fmaxf(fabsf(v[u].z), fabsf(v[u].w))));
          const __half2 lo = __floats2half2_rn(v[u].x * scale, v[u].y * scale);
          const __half2 hi = __floats2half2_rn(v[u].z * scale, v[u].w * scale);
          uint2 o;
          o.x = *reinterpret_cast<const uint32_t*>(&lo);
          o.y = *reinterpret_cast<const uint32_t*>(&hi);
          dst[d4] = o;
        }
      }
    }
  } else {
    for (int64_t d = lane_id(); d < D; d += 32) {
      const float v = x[(src_row ? (int64_t)src_row[row] : row) * D + d];
      ss = fmaf(v, v, ss);
      amax = fmaxf(amax, fabsf(v));
      xh[row * D + d] = __float2half_rn(v * scale);
    }
  }
  ss = warp_sum(ss);
  // |x| * 2^s >= 65520 rounds to +-inf in fp16: the row's scores can be inf or NaN (inf - inf) whatever the exact dot,
  // outside every error bound.  The maximum is then reported as +inf, so eps = inf and no row can be certified.
  const bool overflow = __any_sync(kFull, !(amax * scale < 65520.f));
  if (lane_id() == 0 && max_sqnorm) {                    // sqnorm_range[0] = max, [1] = min (non-negative floats order like
    atomicMax((unsigned*)max_sqnorm, __float_as_uint(overflow ? INFINITY : ss));   // their bit patterns)
    atomicMin((unsigned*)max_sqnorm + 1, __float_as_uint(ss));
  }
  }
}

static unsigned to_half_grid(int64_t n_rows) {
  static int per_sm = 0;                                    // resident CTAs per SM (registers decide), asked once
  if (per_sm == 0) {
    int b = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, to_half_kernel, 256, 0) != cudaSuccess || b < 1) b = 4;
    per_sm = b;
  }
  const int64_t want = (n_rows + 7) / 8, cap = (int64_t)reid::num_sms() * per_sm;
  return (unsigned)(want < cap ? want : cap);
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}

// fp16 row-major (n_rows x D) matrix -> tensor map with a (64 x 128-row) box, 128-byte swizzle
int make_tmap_rows128(CUtensorMap* tmap, const void* base, int64_t n_rows, int64_t D) {
  EncodeTiledFn encode = get_encode_fn();
  if (!encode) {
    set_error("cuTensorMapEncodeTiled is not available from the driver");
    return REID_ERR_CUDA;
  }
  const cuuint64_t gdim[2] = {(cuuint64_t)D, (cuuint64_t)n_rows};
  const cuuint64_t gstride[1] = {(cuuint64_t)D * 2};
  const cuuint32_t box[2] = {(cuuint32_t)BK, 128u};
  const cuuint32_t estr[2] = {1u, 1u};
  CUresult cr = encode(tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), gdim, gstride, box, estr,
                       CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                       CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (cr != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d)", (int)cr);
    return REID_ERR_CUDA;
  }
  return REID_OK;
}

}  // namespace tc
}  // namespace reid

extern "C" {

int reid_knn_tc_plan(int64_t N, int64_t n_rows, int cta_group, int* n_splits_out) {
  using namespace reid;
  REID_CHECK_ARG(N > 0 && n_rows > 0 && n_splits_out && (cta_group == 1 || cta_group == 2),
                 "reid_knn_tc_plan: bad arguments");
  const int slots = num_sms() / cta_group;             // concurrently running work units
  const int64_t n_mblk = (n_rows + tc::BM * cta_group - 1) / (tc::BM * cta_group);
  const int64_t n_tiles = (N + tc::BN - 1) / tc::BN;
  int best = 1;
  double best_eff = -1.0;
  for (int s = 1; s <= REID_TC_MAX_SPLITS; ++s) {
    if (s > n_tiles) break;
    const int64_t units = n_mblk * s;
    const int64_t waves = (units + slots - 1) / slots;
    const double eff = (double)units / (double)(waves * slots);
    if (eff > best_eff + 0.02) {  // prefer fewer splits unless the gain is real
      best_eff = eff;
      best = s;
    }
  }
  *n_splits_out = best;
  return REID_OK;
}

int reid_features_to_half_acc(const float* x, int64_t n_rows, int64_t D, int scale_log2, void* xh, float* max_sqnorm_inout,
                              void* stream) {
  using namespace reid;
  REID_CHECK_ARG(x && xh && n_rows >= 0 && D > 0, "reid_features_to_half_acc: bad arguments");
  REID_CHECK_ARG(scale_log2 >= -8 && scale_log2 <= 12, "reid_features_to_half_acc: scale_log2=%d out of range", scale_log2);
  if (n_rows == 0) return REID_OK;
  tc::to_half_kernel<<<tc::to_half_grid(n_rows), 256, 0, (cudaStream_t)stream>>>(x, n_rows, D, ldexpf(1.0f, scale_log2),
                                                                                     (__half*)xh, max_sqnorm_inout, nullptr);
  REID_LAUNCH_CHECK();
  return REID_OK;
}

int reid_sqnorm_range_reset(float* sqnorm_range, void* stream) {
  using namespace reid;
  REID_CHECK_ARG(sqnorm_range, "reid_sqnorm_range_reset: NULL pointer");
  REID_CUDA(cudaMemsetAsync(sqnorm_range, 0, sizeof(float), (cudaStream_t)stream));
  REID_CUDA(cudaMemsetAsync(sqnorm_range + 1, 0x7f, sizeof(float), (cudaStream_t)stream));
  return REID_OK;
}

int reid_features_to_half_gather(const float* x, const int32_t* src_row, int64_t n_rows, int64_t D, int scale_log2, void* xh,
                                 float* max_sqnorm_inout, void* stream) {
  using namespace reid;
  REID_CHECK_ARG(x && src_row && xh && n_rows >= 0 && D > 0, "reid_features_to_half_gather: bad arguments");
  REID_CHECK_ARG(scale_log2 >= -8 && scale_log2 <= 12, "reid_features_to_half_gather: scale_log2=%d out of range", scale_log2);
  if (n_rows == 0) return REID_OK;
  tc::to_half_kernel<<<tc::to_half_grid(n_rows), 256, 0, (cudaStream_t)stream>>>(x, n_rows, D, ldexpf(1.0f, scale_log2),
                                                                                     (__half*)xh, max_sqnorm_inout, src_row);
  REID_LAUNCH_CHECK();
  return REID_OK;
}

int reid_features_to_half(const float* x, int64_t n_rows, int64_t D, int scale_log2, void* xh, float* max_sqnorm_out,
                          void* stream) {
  using namespace reid;
  REID_CHECK_ARG(x && xh && n_rows >= 0 && D > 0, "reid_features_to_half: bad arguments");
  REID_CHECK_ARG(scale_log2 >= -8 && scale_log2 <= 12, "reid_features_to_half: scale_log2=%d out of range", scale_log2);
  cudaStream_t st = (cudaStream_t)stream;
  if (max_sqnorm_out) {                                  // [0] = 0, [1] = 0x7f7f7f7f (3.4e38): identities of max / min
    REID_CUDA(cudaMemsetAsync(max_sqnorm_out, 0, sizeof(float), st));
    REID_CUDA(cudaMemsetAsync(max_sqnorm_out + 1, 0x7f, sizeof(float), st));
  }
  if (n_rows == 0) return REID_OK;
  tc::to_half_kernel<<<tc::to_half_grid(n_rows), 256, 0, st>>>(x, n_rows, D, ldexpf(1.0f, scale_log2), (__half*)xh,
                                                                  max_sqnorm_out, nullptr);
  REID_LAUNCH_CHECK();
  return REID_OK;
}

int reid_knn_candidates_tc(const void* xh, int64_t N, int64_t D, int scale_log2, int64_t row_begin, int64_t row_end,
                           int keep, int n_splits, int cta_group, uint64_t* cand, int32_t* cand_cnt, uint32_t* row_tau,
                           void* stream) {
  return reid_knn_candidates_tc_ab(xh, N, xh, N, D, scale_log2, row_begin, row_end, keep, n_splits, cta_group, cand,
                                   cand_cnt, row_tau, stream);
}

int reid_knn_candidates_tc_ab(const void* xa, int64_t Na, const void* xh, int64_t N, int64_t D, int scale_log2,
                              int64_t row_begin, int64_t row_end, int keep, int n_splits, int cta_group, uint64_t* cand,
                              int32_t* cand_cnt, uint32_t* row_tau, void* stream) {
  return reid_knn_candidates_tc_abt(xa, Na, xh, N, D, scale_log2, row_begin, row_end, keep, n_splits, cta_group, cand, cand_cnt,
                                    row_tau, 0, nullptr, nullptr, nullptr, 0, stream);
}

int reid_knn_candidates_tc_abt(const void* xa, int64_t Na, const void* xh, int64_t N, int64_t D, int scale_log2,
                               int64_t row_begin, int64_t row_end, int keep, int n_splits, int cta_group, uint64_t* cand,
                               int32_t* cand_cnt, uint32_t* row_tau, int publish_final, const float* tau_col,
                               uint64_t* cand_col, int32_t* cand_col_cnt, int cap_col, void* stream) {
  using namespace reid;
  REID_CHECK_ARG(!tau_col || (cand_col && cand_col_cnt && cap_col >= 1), "reid_knn_candidates_tc_abt: tau_col needs the column lists");
  const int boot = keep < 0;          // keep < 0: sampling prepass, |keep| kept, threshold seeded from the first scores
  if (boot) keep = -keep;
  REID_CHECK_ARG(xa && xh && cand && cand_cnt && row_tau, "reid_knn_candidates_tc: NULL pointer");
  REID_CHECK_ARG(N > 0 && N < (1ll << 31) && Na > 0 && Na < (1ll << 31) && D > 0 && D % tc::BK == 0,
                 "reid_knn_candidates_tc: need D %% 64 == 0 (D=%lld)", (long long)D);
  REID_CHECK_ARG(((uintptr_t)xh & 15) == 0 && ((uintptr_t)xa & 15) == 0, "reid_knn_candidates_tc: operands must be 16-byte aligned");
  REID_CHECK_ARG(0 <= row_begin && row_begin < row_end && row_end <= Na, "reid_knn_candidates_tc: bad row range");
  REID_CHECK_ARG(keep >= 1 && keep <= REID_TC_KEEP_MAX, "reid_knn_candidates_tc: keep=%d not in 1..%d", keep,
                 REID_TC_KEEP_MAX);
  REID_CHECK_ARG(cta_group == 1 || cta_group == 2, "reid_knn_candidates_tc: cta_group=%d must be 1 or 2", cta_group);
  const int64_t n_tiles = (N + tc::BN - 1) / tc::BN;
  // the prepass mode may cut its few column tiles finer: its lists are only read by reid_knn_sample_tau
  REID_CHECK_ARG(n_splits >= 1 && n_splits <= (boot ? 2 * REID_TC_MAX_SPLITS : REID_TC_MAX_SPLITS) && n_splits <= n_tiles,
                 "reid_knn_candidates_tc: n_splits=%d", n_splits);
  CUtensorMap tmap, tmap_b;
  int rc = tc::make_tmap_rows128(&tmap, xa, Na, D);
  if (rc != REID_OK) return rc;
  rc = tc::make_tmap_rows128(&tmap_b, xh, N, D);
  if (rc != REID_OK) return rc;
  tc::Params p;
  p.N = N;
  p.row_begin = row_begin;
  p.row_end = row_end;
  p.num_k_blocks = (int)(D / tc::BK);
  p.n_mblk = (int)((row_end - row_begin + tc::BM * cta_group - 1) / (tc::BM * cta_group));
  p.n_splits = n_splits;
  p.n_tiles = (int)n_tiles;
  p.keep = keep;
  p.boot = boot;
  p.descale = ldexpf(1.0f, -2 * scale_log2);
  p.cand = (unsigned long long*)cand;
  p.cand_cnt = cand_cnt;
  p.row_tau = row_tau;
  p.tau_col = tau_col;
  p.cand2 = (unsigned long long*)cand_col;
  p.cand2_cnt = cand_col_cnt;
  p.cap2 = cap_col;
  p.publish_final = publish_final;
  REID_CUDA(cudaMemsetAsync(row_tau, 0, sizeof(uint32_t) * (size_t)(row_end - row_begin), (cudaStream_t)stream));
  p.dbg = dev_env("REID_TC_DEBUG", 0);
  const int units = p.n_mblk * n_splits;
  const int slots = num_sms() / cta_group;
  const int grid = (units < slots ? units : slots) * cta_group;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(tc::kThreads);
  cfg.stream = (cudaStream_t)stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)cta_group;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (cta_group == 1) {
    cfg.dynamicSmemBytes = tc::Cfg<1>::kSmem;
    REID_CUDA(cudaFuncSetAttribute(tc::simtopk_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::Cfg<1>::kSmem));
    REID_CUDA(cudaLaunchKernelEx(&cfg, tc::simtopk_kernel<1>, tmap, tmap_b, p));
  } else {
    cfg.dynamicSmemBytes = tc::Cfg<2>::kSmem;
    REID_CUDA(cudaFuncSetAttribute(tc::simtopk_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::Cfg<2>::kSmem));
    REID_CUDA(cudaLaunchKernelEx(&cfg, tc::simtopk_kernel<2>, tmap, tmap_b, p));
  }
  REID_LAUNCH_CHECK();
  return REID_OK;
}
}
