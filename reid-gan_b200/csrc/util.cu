// Error plumbing + the count->pointer scan used between the two-pass (count / fill) stages.
#include <stdarg.h>

#include <map>
#include <mutex>
#include <utility>

#include "common.cuh"

namespace reid {

static thread_local char g_err[512] = "";
unsigned long long g_launches = 0;

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// count -> pointer scan, single pass over many CTAs ("decoupled look-back"): a CTA takes the next tile of
// 256 x 8 counts by ticket, publishes the tile's total, sums the published totals of the tiles before it (32 per
// step, stopping at the first tile that already knows its inclusive prefix), publishes its own inclusive prefix and
// writes its 2048 pointers.  All sums are 64-bit (a row of reid_jaccard_bounds alone may reach 2^31 - 1).  The
// stats (total, max, sum of squares) come out of the same pass; the CTA that finishes last writes them and
// clears the state, so the state buffer is zero again when the kernel ends (no memset per call).
constexpr int kScanThreads = 256;
constexpr int kScanPer = 8;
constexpr int kScanTile = kScanThreads * kScanPer;
constexpr unsigned long long kScanAgg = 1ull << 62, kScanIncl = 2ull << 62, kScanMask = (1ull << 62) - 1ull;

struct ScanState {
  unsigned ticket, done;
  int max;
  int pad;
  unsigned long long sq;
  unsigned long long tiles[1];        // n_tiles entries: status (2 bits) | value (62 bits)
};

__global__ void __launch_bounds__(kScanThreads) scan_counts_kernel(const int32_t* __restrict__ cnt, int64_t n,
                                                                   int64_t* __restrict__ ptr, int64_t* __restrict__ stats,
                                                                   ScanState* __restrict__ st, unsigned n_tiles) {
  __shared__ unsigned s_tile, s_last;
  __shared__ long long s_warp[kScanThreads / 32];
  __shared__ long long s_prefix;
  __shared__ int s_max[kScanThreads / 32];
  __shared__ unsigned long long s_sq[kScanThreads / 32];
  const int t = threadIdx.x, lane = t & 31, w = t >> 5;
  if (t == 0) s_tile = atomicAdd(&st->ticket, 1u);
  __syncthreads();
  const unsigned tile = s_tile;
  const int64_t i0 = (int64_t)tile * kScanTile + (int64_t)t * kScanPer;
  int32_t c[kScanPer];
  if ((((uintptr_t)cnt) & 15) == 0 && i0 + kScanPer <= n) {
#pragma unroll
    for (int q = 0; q < kScanPer / 4; ++q) {
      const int4 v = *reinterpret_cast<const int4*>(cnt + i0 + 4 * q);
      c[4 * q] = v.x; c[4 * q + 1] = v.y; c[4 * q + 2] = v.z; c[4 * q + 3] = v.w;
    }
  } else {
#pragma unroll
    for (int j = 0; j < kScanPer; ++j) c[j] = i0 + j < n ? cnt[i0 + j] : 0;
  }
  long long s = 0;
  unsigned long long sq = 0;
  int mx = 0;
#pragma unroll
  for (int j = 0; j < kScanPer; ++j) {
    mx = max(mx, c[j]);
    sq += (unsigned long long)((long long)c[j] * c[j]);
    s += c[j];
  }
  long long inc = s;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const long long v = __shfl_up_sync(kFull, inc, o);
    if (lane >= o) inc += v;
  }
  mx = warp_max(mx);
  sq = warp_sum(sq);
  if (lane == 31) s_warp[w] = inc;
  if (lane == 0) {
    s_max[w] = mx;
    s_sq[w] = sq;
  }
  __syncthreads();
  if (w == 0) {
    long long wt = lane < kScanThreads / 32 ? s_warp[lane] : 0;
    long long wi = wt;
#pragma unroll
    for (int o = 1; o < kScanThreads / 32; o <<= 1) {
      const long long v = __shfl_up_sync(kFull, wi, o);
      if (lane >= o) wi += v;
    }
    if (lane < kScanThreads / 32) s_warp[lane] = wi - wt;          // exclusive offset of each warp inside the tile
    const long long total = __shfl_sync(kFull, wi, kScanThreads / 32 - 1);
    volatile unsigned long long* tiles = st->tiles;
    long long excl = 0;
    if (tile > 0) {
      if (lane == 0) tiles[tile] = kScanAgg | (unsigned long long)total;
      for (int64_t j = (int64_t)tile - 1;; j -= 32) {
        const int64_t jj = j - lane;
        unsigned long long v;
        do {                                                       // tickets are handed out in order: tile jj is running
          v = jj >= 0 ? tiles[jj] : (2ull << 62);
        } while (__any_sync(kFull, (v >> 62) == 0ull));
        const unsigned incl = __ballot_sync(kFull, (v >> 62) == 2ull);
        const int first = incl ? __ffs(incl) - 1 : 32;
        excl += warp_sum(lane <= first ? (long long)(v & kScanMask) : 0ll);
        if (incl) break;
      }
    }
    if (lane == 0) {
      tiles[tile] = kScanIncl | (unsigned long long)(excl + total);
      s_prefix = excl;
      int m = 0;
      unsigned long long q = 0;
      for (int u = 0; u < kScanThreads / 32; ++u) {
        m = max(m, s_max[u]);
        q += s_sq[u];
      }
      atomicMax(&st->max, m);
      atomicAdd(&st->sq, q);
    }
  }
  __syncthreads();
  long long run = s_prefix + s_warp[w] + (inc - s);
#pragma unroll
  for (int j = 0; j < kScanPer; ++j) {
    if (i0 + j < n) ptr[i0 + j] = run;
    run += c[j];
  }
  __threadfence();
  __syncthreads();
  if (t == 0) s_last = atomicAdd(&st->done, 1u) == n_tiles - 1u;
  __syncthreads();
  if (s_last) {                                                    // every other CTA has published and left
    __threadfence();
    volatile unsigned long long* tiles = st->tiles;
    if (t == 0) {
      const long long total = (long long)(tiles[n_tiles - 1] & kScanMask);
      ptr[n] = total;
      if (stats) {
        stats[0] = total;
        stats[1] = *(volatile int*)&st->max;
        stats[2] = (long long)*(volatile unsigned long long*)&st->sq;
      }
    }
    __syncthreads();
    for (unsigned u = t; u < n_tiles; u += kScanThreads) tiles[u] = 0ull;
    if (t == 0) {
      st->ticket = 0u;
      st->done = 0u;
      st->max = 0;
      st->sq = 0ull;
    }
  }
}

// Scan state per (device, stream): zero-filled once, left zeroed by every launch.  Grown on demand (never while a
// stream capture is running: call the scan once before capturing).
struct ScanSlot {
  ScanState* state;
  size_t tiles;
};
static std::mutex g_scan_mu;
static std::map<std::pair<int, cudaStream_t>, ScanSlot> g_scan_slots;

static int scan_state_for(cudaStream_t stream, size_t n_tiles, ScanState** out) {
  int dev = 0;
  REID_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(g_scan_mu);
  ScanSlot& slot = g_scan_slots[std::make_pair(dev, stream)];
  if (slot.tiles < n_tiles) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    REID_CUDA(cudaStreamIsCapturing(stream, &cs));
    if (cs != cudaStreamCaptureStatusNone) {
      set_error("reid_scan_counts: the scan state must exist before a stream capture (run the pass once first)");
      return REID_ERR_UNSUPPORTED;
    }
    size_t want = slot.tiles ? slot.tiles : 1024;
    while (want < n_tiles) want *= 2;
    if (slot.state) {
      REID_CUDA(cudaStreamSynchronize(stream));
      REID_CUDA(cudaFree(slot.state));
      slot.state = nullptr;
      slot.tiles = 0;
    }
    const size_t bytes = sizeof(ScanState) + sizeof(unsigned long long) * want;
    void* p = nullptr;
    REID_CUDA(cudaMalloc(&p, bytes));
    REID_CUDA(cudaMemset(p, 0, bytes));
    slot.state = (ScanState*)p;
    slot.tiles = want;
  }
  *out = slot.state;
  return REID_OK;
}

}  // namespace reid

extern "C" {

int reid_abi_version(void) { return 5; }
const char* reid_last_error(void) { return reid::g_err; }
uint64_t reid_launch_count(void) { return reid::g_launches; }

int reid_scan_counts(const int32_t* cnt, int64_t n, int64_t* ptr_out, int64_t* stats_out, void* stream) {
  using namespace reid;
  REID_CHECK_ARG(n >= 0 && ptr_out, "reid_scan_counts: bad arguments");
  REID_CHECK_ARG(n == 0 || cnt, "reid_scan_counts: cnt is NULL");
  cudaStream_t st = (cudaStream_t)stream;
  if (n == 0) {
    REID_CUDA(cudaMemsetAsync(ptr_out, 0, sizeof(int64_t), st));
    if (stats_out) REID_CUDA(cudaMemsetAsync(stats_out, 0, 3 * sizeof(int64_t), st));
    return REID_OK;
  }
  const size_t n_tiles = (size_t)((n + kScanTile - 1) / kScanTile);
  ScanState* state = nullptr;
  int rc = scan_state_for(st, n_tiles, &state);
  if (rc != REID_OK) return rc;
  scan_counts_kernel<<<(unsigned)n_tiles, kScanThreads, 0, st>>>(cnt, n, ptr_out, stats_out, state, (unsigned)n_tiles);
  REID_LAUNCH_CHECK();
  return REID_OK;
}
}
