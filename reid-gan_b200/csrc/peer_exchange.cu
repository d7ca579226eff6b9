// Exchange steps of the row-sharded pass over NVLink peer memory (SURVEY.md 8e) -- plain stores from this GPU's kernels
// into buffers that live on the other GPUs of the box (mapped into this process by the host layer:
// torch.distributed._symmetric_memory hands out one base pointer per rank).  No NCCL call, no padding on the wire:
// only the valid entries of a list travel.
//
// reid_peer_push_lists: the hand-over of the tile-sharded search.  Rank `me` has appended the survivors of ITS tiles
// to partial lists of ALL rows (slot == row, W blocks of B rows, `cap` entries each).  The rows of block w belong
// to rank w, which keeps W partial lists per own row: list q of local row r at (q * B + r).  So block w of this
// rank's lists goes to list `me` of rank w -- the all-to-all of sharded.knn_search_tiles, minus the unused tail
// of every list (the lists are sized for 4x their expected length).
#include "common.cuh"

namespace reid {

__global__ void __launch_bounds__(256) peer_push_lists_kernel(const unsigned long long* __restrict__ part,
                                                              const int32_t* __restrict__ part_cnt, int W, int64_t B,
                                                              int cap, int me, const unsigned long long* __restrict__ peer_base,
                                                              int64_t cnt_offset_bytes) {
  const int64_t slot = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);      // w * B + r
  if (slot >= (int64_t)W * B) return;
  const int w = (int)(slot / B);
  const int64_t r = slot - (int64_t)w * B;
  const int lane = lane_id();
  const int c_true = part_cnt[slot];
  const int c = c_true < cap ? c_true : cap;
  unsigned char* base = reinterpret_cast<unsigned char*>(peer_base[w]);
  unsigned long long* dst = reinterpret_cast<unsigned long long*>(base) + ((int64_t)me * B + r) * cap;
  const unsigned long long* src = part + slot * cap;
  for (int t = lane; t < c; t += 32) dst[t] = src[t];
  // the TRUE count travels (a list that overflowed must be recognised by the owner's certificate)
  if (lane == 0) reinterpret_cast<int32_t*>(base + cnt_offset_bytes)[(int64_t)me * B + r] = c_true;
  __threadfence_system();
}

// reid_peer_push_records: the ragged all-gathers of the row-sharded sparse stages (V rows, V_qe rows, eps-neighbour
// lists).  Same record format as rows_pack_kernel (rerank_sparse.cu) -- rec = { count, idx[stride], (val bits[stride]) }
// -- but instead of packing into a staging buffer that NCCL then replicates, every warp writes its row's record
// straight into the receive buffer of EVERY rank (record (me * max_rows + row) there): one read of the row, `world`
// coalesced stores of its valid entries, nothing else on the wire.
__global__ void __launch_bounds__(256) peer_push_records_kernel(const int32_t* __restrict__ cnt, const int64_t* __restrict__ ptr,
                                                                const int32_t* __restrict__ idx, const float* __restrict__ val,
                                                                int64_t n_rows, int64_t max_rows, int stride, int words, int me,
                                                                int W, const unsigned long long* __restrict__ peer_base,
                                                                int64_t rec_offset_bytes) {
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= max_rows) return;
  const int lane = lane_id();
  const int c = row < n_rows ? cnt[row] : 0;                 // padding rows of the last block: count 0
  const int m = c < stride ? c : stride;
  const int64_t a = row < n_rows ? ptr[row] : 0;
  const int64_t rec_index = ((int64_t)me * max_rows + row) * words;
  for (int t0 = 0; t0 < m || t0 == 0; t0 += 32) {
    const int t = t0 + lane;
    int32_t iv = 0, vv = 0;
    if (t < m) {
      iv = idx[a + t];
      if (val) vv = __float_as_int(val[a + t]);
    }
    for (int w = 0; w < W; ++w) {
      int32_t* r = reinterpret_cast<int32_t*>(reinterpret_cast<unsigned char*>(peer_base[w]) + rec_offset_bytes) + rec_index;
      if (t0 == 0 && lane == 0) r[0] = c;                    // the true count (a row longer than the stride is noticed)
      if (t < m) {
        r[1 + t] = iv;
        if (val) r[1 + stride + t] = vv;
      }
    }
  }
  __threadfence_system();
}

// reid_peer_allgather: fixed-size blocks (thresholds, neighbour lists): my block goes to slot `me` of every rank.
__global__ void __launch_bounds__(256) peer_allgather_kernel(const uint32_t* __restrict__ src, int64_t n4, int me, int W,
                                                             const unsigned long long* __restrict__ peer_base,
                                                             int64_t dst_offset_bytes) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t v = src[i];
    for (int w = 0; w < W; ++w)
      reinterpret_cast<uint32_t*>(reinterpret_cast<unsigned char*>(peer_base[w]) + dst_offset_bytes)[(int64_t)me * n4 + i] = v;
  }
  __threadfence_system();
}

// reid_peer_scatter_rows: the feature all-gather of distributed evaluation.  Local row r goes to rows dst[2r] and
// dst[2r + 1] of the (M, D) matrix [query; gallery] of every rank (-1: not in that list).  One warp per row: each
// float4 of the row is loaded once and stored 2 x W times.  A destination >= M is counted and never written.
__global__ void __launch_bounds__(256) peer_scatter_rows_kernel(const float4* __restrict__ src, int64_t n_rows, int64_t D4,
                                                                const int32_t* __restrict__ dst_rows, int64_t M, int W,
                                                                const unsigned long long* __restrict__ peer_base,
                                                                int64_t dst_offset_bytes,
                                                                unsigned long long* __restrict__ bad_count) {
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= n_rows) return;
  const int lane = lane_id();
  int64_t d0 = dst_rows[2 * row], d1 = dst_rows[2 * row + 1];
  if (d0 >= M || d1 >= M) {
    if (lane == 0 && bad_count) atomicAdd(bad_count, (unsigned long long)((d0 >= M) + (d1 >= M)));
    if (d0 >= M) d0 = -1;
    if (d1 >= M) d1 = -1;
  }
  if (d0 < 0 && d1 < 0) return;
  const float4* s = src + row * D4;
  for (int64_t c = lane; c < D4; c += 32) {
    const float4 v = s[c];
    for (int w = 0; w < W; ++w) {
      float4* x = reinterpret_cast<float4*>(reinterpret_cast<unsigned char*>(peer_base[w]) + dst_offset_bytes);
      if (d0 >= 0) x[d0 * D4 + c] = v;
      if (d1 >= 0) x[d1 * D4 + c] = v;
    }
  }
  __threadfence_system();
}

}  // namespace reid

extern "C" {

int reid_peer_push_lists(const uint64_t* part, const int32_t* part_cnt, int world, int64_t block_rows, int cap, int me,
                         const uint64_t* peer_base, int64_t cnt_offset_bytes, void* stream) {
  using namespace reid;
  REID_CHECK_ARG(part && part_cnt && peer_base, "reid_peer_push_lists: NULL pointer");
  REID_CHECK_ARG(world >= 1 && block_rows >= 0 && cap >= 1 && me >= 0 && me < world && cnt_offset_bytes >= 0 &&
                     cnt_offset_bytes % 4 == 0,
                 "reid_peer_push_lists: bad arguments");
  const int64_t slots = (int64_t)world * block_rows;
  if (slots == 0) return REID_OK;
  peer_push_lists_kernel<<<(unsigned)((slots + 7) / 8), 256, 0, (cudaStream_t)stream>>>(
      (const unsigned long long*)part, part_cnt, world, block_rows, cap, me, (const unsigned long long*)peer_base,
      cnt_offset_bytes);
  REID_LAUNCH_CHECK();
  return REID_OK;
}

int reid_peer_push_records(const int32_t* cnt, const int64_t* ptr, const int32_t* idx, const float* val, int64_t n_rows,
                           int64_t max_rows, int stride, int me, int world, const uint64_t* peer_base,
                           int64_t rec_offset_bytes, void* stream) {
  using namespace reid;
  REID_CHECK_ARG(peer_base && stride >= 1 && n_rows >= 0 && max_rows >= n_rows && me >= 0 && me < world &&
                     rec_offset_bytes >= 0 && rec_offset_bytes % 4 == 0,
                 "reid_peer_push_records: bad arguments");
  REID_CHECK_ARG(n_rows == 0 || (cnt && ptr && idx), "reid_peer_push_records: NULL pointer");
  if (max_rows == 0) return REID_OK;
  const int words = 1 + stride * (val ? 2 : 1);
  peer_push_records_kernel<<<(unsigned)((max_rows + 7) / 8), 256, 0, (cudaStream_t)stream>>>(
      cnt, ptr, idx, val, n_rows, max_rows, stride, words, me, world, (const unsigned long long*)peer_base, rec_offset_bytes);
  REID_LAUNCH_CHECK();
  return REID_OK;
}

int reid_peer_allgather(const void* src, int64_t block_bytes, int me, int world, const uint64_t* peer_base,
                        int64_t dst_offset_bytes, void* stream) {
  using namespace reid;
  REID_CHECK_ARG(src && peer_base && block_bytes >= 0 && block_bytes % 4 == 0 && me >= 0 && me < world &&
                     dst_offset_bytes >= 0 && dst_offset_bytes % 4 == 0 && ((uintptr_t)src & 3) == 0,
                 "reid_peer_allgather: bad arguments (4-byte granularity)");
  if (block_bytes == 0) return REID_OK;
  const int64_t n4 = block_bytes / 4;
  int64_t grid = (n4 + 255) / 256;
  if (grid > 4 * num_sms()) grid = 4 * num_sms();
  peer_allgather_kernel<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>((const uint32_t*)src, n4, me, world,
                                                                         (const unsigned long long*)peer_base,
                                                                         dst_offset_bytes);
  REID_LAUNCH_CHECK();
  return REID_OK;
}

int reid_peer_scatter_rows(const float* src, int64_t n_rows, int64_t D, const int32_t* dst_rows, int64_t M, int world,
                           const uint64_t* peer_base, int64_t dst_offset_bytes, uint64_t* bad_count, void* stream) {
  using namespace reid;
  REID_CHECK_ARG(n_rows == 0 || (src && dst_rows), "reid_peer_scatter_rows: NULL pointer");
  REID_CHECK_ARG(peer_base && n_rows >= 0 && M >= 1 && world >= 1 && D >= 1 && dst_offset_bytes >= 0,
                 "reid_peer_scatter_rows: bad arguments");
  REID_CHECK_ARG(D % 4 == 0, "reid_peer_scatter_rows: D=%lld is not a multiple of 4", (long long)D);
  REID_CHECK_ARG(((uintptr_t)src & 15) == 0 && dst_offset_bytes % 16 == 0,
                 "reid_peer_scatter_rows: src and dst_offset_bytes must be 16-byte aligned");
  if (n_rows == 0) return REID_OK;
  REID_CHECK_ARG((n_rows + 7) / 8 < (1LL << 31), "reid_peer_scatter_rows: too many rows");
  peer_scatter_rows_kernel<<<(unsigned)((n_rows + 7) / 8), 256, 0, (cudaStream_t)stream>>>(
      (const float4*)src, n_rows, D / 4, dst_rows, M, world, (const unsigned long long*)peer_base, dst_offset_bytes,
      (unsigned long long*)bad_count);
  REID_LAUNCH_CHECK();
  return REID_OK;
}
}
