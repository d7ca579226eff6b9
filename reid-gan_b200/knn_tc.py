"""a1 on the tensor cores: fp16 tcgen05 candidate GEMM with fused top-K, exact re-score with a
per-row certificate, exact CUDA-core search for the rows that cannot be certified
(replaces faiss IndexFlatL2 / GpuIndexFlatL2.search, utils/faiss_rerank.py:39-62).

The result is bit-identical to the all-exact search whatever the fp16 arithmetic does: a row is
accepted only when the certificate of knn_rescore.cu holds, otherwise it is recomputed exactly.
"""
import ctypes

import torch

from . import _lib
from ._lib import call, check, ptr, stream_ptr

TC_CAP = 512
KEEP_MAX = 64
SCALE_LOG2 = 4          # features are scaled by 2^4 before rounding to fp16 (keeps them out of the subnormals)
CTA_GROUP = 2                 # 2 = CTA pairs (tcgen05 cta_group::2); 1 = single CTAs (developer comparison: set the attribute)
ORDER_ROWS = True             # cluster-locality visiting order of the re-score stage
SLACK = 34              # K = k + SLACK candidates are kept per (row, column range)


UNIT_NORM_TOL = 1e-4    # rows count as "one norm" when max ||x||^2 <= (1 + tol) min ||x||^2 (see one_norm)


def one_norm(sqnorm_range):
    """sqnorm_range = [max ||x||^2, min ||x||^2] (reid_features_to_half).  faiss IndexFlatL2 ranks by squared L2, which
    is the inner-product order the tensor-core search produces iff all rows have the same norm.  Rows normalised in
    fp32 by the backbone (models/resnet.py:90-94) differ by ~1e-7 -- below what the reference's own fp32 search
    resolves; beyond UNIT_NORM_TOL the search is redone with the squared-L2 key (reid_knn_exact_l2)."""
    mx, mn = float(sqnorm_range[0]), float(sqnorm_range[1])
    return mx <= mn * (1.0 + UNIT_NORM_TOL)


def sqnorm_range_of(x, sqnorm_range):
    """[max, min] squared norms of the rows of x, from the range reid_features_to_half reported.  That maximum is +inf
    when a feature overflowed the fp16 operand (|x| * 2^SCALE_LOG2 >= 65520; it makes eps infinite, so no row is
    certified); the true range is then computed again, so that an overflow alone never picks the squared-L2 key."""
    rng = sqnorm_range.tolist()
    if rng[0] == float("inf"):
        r = torch.empty(2, dtype=torch.float32, device=x.device)
        call("reid_sqnorm_range", ptr(x), x.shape[0], x.shape[1], ptr(r), stream_ptr())
        rng = r.tolist()
    return rng


def new_sqnorm_range(dev):
    """{max, min} accumulator for reid_features_to_half_acc: identities {0, 3.4e38}."""
    r = torch.empty(2, dtype=torch.float32, device=dev)
    call("reid_sqnorm_range_reset", ptr(r), stream_ptr())
    return r


def err_bound(max_sqnorm):
    """|fp16-GEMM score - exact dot| <= 2^-10 ||x_i|| ||x_j|| (both operands rounded to 11 significant
    bits, Cauchy-Schwarz) + fp32 accumulation allowance."""
    return float(max_sqnorm) * (2.0 ** -10) * 1.02 + 2.0 ** -14


SYM = True                    # symmetric search when the shard is the whole matrix
SYM_MIN_N = 8192        # below this the sample cannot give a tight threshold; the one-sided kernel is used
SYM_CAP = 1024          # list capacity per row in the symmetric search
SYM_RANK = 16           # tau_i = SYM_RANK-th best sample score ...
SYM_TARGET = 256        # ... with the sample sized so that about SYM_TARGET columns beat it (k <= 32; twice that above)
SYM_MAX_K = 64          # rank positions live in one 64-bit mask (REID_MAX_K1)


def sym_rank(k):
    """tau_i is the sym_rank(k)-th best of the m sample scores of row i, so about sym_rank / m * N columns beat it:
    SYM_TARGET for k <= 32 and twice that for 32 < k <= 64 (the lists must hold the k best with room for the
    certificate's window) -- the sample itself stays the same size."""
    return SYM_RANK * (1 if k <= 32 else 2)


def sample_size(N, k=30):
    """Rows in the threshold sample (see sym_rank)."""
    return min(N, max(1024, -(-(SYM_RANK * N // SYM_TARGET) // 256) * 256))
_tile_cache = {}


def prepass_splits(n_rows, m, pair_slots=74, max_splits=4):
    """Column splits of the sampling prepass over `n_rows` rows: as many (<= max_splits, <= sample tiles) as keep the
    (256-row unit x split) count within one wave of the CTA-pair slots."""
    units = (n_rows + 255) // 256
    s = 1
    while s < max_splits and units * s * 2 <= pair_slots and s * 2 <= m // 256:
        s *= 2
    return s


def _tile_order(n_t, dev, sb=16):
    """Upper-triangle 256 x 256 tiles in super-blocks of sb x sb: the ~74 tiles in flight share a few dozen operand
    blocks, so they stream out of L2.  Cached per (n_t, device)."""
    key_ = (n_t, str(dev))
    if key_ not in _tile_cache:
        out = []
        nb = (n_t + sb - 1) // sb
        for bi in range(nb):
            for bj in range(bi, nb):
                for i in range(bi * sb, min(n_t, (bi + 1) * sb)):
                    for j in range(max(i, bj * sb), min(n_t, (bj + 1) * sb)):
                        out.append((i, j))
        _tile_cache[key_] = torch.tensor(out, dtype=torch.int32).to(dev).contiguous()
    return _tile_cache[key_]


SYM_WIDE = False              # True: 256 x 512 strips (reid_knn_candidates_sym_wide).  Measured slower (1.71 vs 1.53 ms at N = 32,621, DESIGN.md 4): off
_unit_cache = {}


def pair_units(tiles):
    """(n, 2) int32 tile list -> (u, 3) int32 units (I, J0, J1): consecutive tiles of one row block are paired into a
    256 x 512 strip, J1 = -1 for a tile left alone (odd runs).  Order preserved."""
    import numpy as np
    t = tiles.cpu().numpy().reshape(-1, 2)
    n = t.shape[0]
    if n == 0:
        return torch.empty((0, 3), dtype=torch.int32)
    I = t[:, 0]
    start = np.r_[True, I[1:] != I[:-1]]
    run_start = np.flatnonzero(start)[np.cumsum(start) - 1]
    first = np.flatnonzero((np.arange(n) - run_start) % 2 == 0)
    nxt = np.minimum(first + 1, n - 1)
    has = (first + 1 < n) & (I[nxt] == I[first]) & (run_start[nxt] == run_start[first])
    units = np.stack([I[first], t[first, 1], np.where(has, t[nxt, 1], -1)], axis=1).astype(np.int32)
    return torch.from_numpy(np.ascontiguousarray(units))


def candidates_sym_launch(xh, N, D, tau, tiles, cap, cand, cnt, reset, sp):
    """One launch of the symmetric candidate kernel over `tiles` (a cached, persistent (n, 2) int32 device tensor)."""
    if not SYM_WIDE:
        call("reid_knn_candidates_sym", ptr(xh), N, D, SCALE_LOG2, ptr(tau), ptr(tiles), tiles.shape[0], cap, ptr(cand),
             ptr(cnt), reset, sp)
        return
    key_ = (tiles.data_ptr(), int(tiles.shape[0]))
    ent = _unit_cache.get(key_)
    if ent is None or ent[0] is not tiles:                     # first use of this list (a host synchronisation, cached)
        ent = (tiles, pair_units(tiles).to(tiles.device))
        _unit_cache[key_] = ent
    units = ent[1]
    call("reid_knn_candidates_sym_wide", ptr(xh), N, D, SCALE_LOG2, ptr(tau), ptr(units), units.shape[0], cap, ptr(cand),
         ptr(cnt), reset, sp)


_stride_cache = {}


def _sample_stride(N, m=None):
    """~N / golden ratio, coprime with N: (i * stride) mod N, i < m, walks the rows with low discrepancy.  a / N is only
    close to the golden ratio: past the last Fibonacci denominator below m its continued fraction has large terms and the
    first m points bunch up (N = 32,621, m = 2,048, a = round(0.618 N): gaps of 4, 65 and 69 rows).  So among the strides
    within +-64 of round(0.618 N) the one whose first m points leave the smallest largest gap is taken (ties: the
    closest).  m = None: plain rounding."""
    import math
    a0 = max(1, int(round(N * 0.6180339887498949)))
    if m is None or m < 2 or m >= N:
        a = a0
        while math.gcd(a, N) != 1:
            a += 1
        return a
    key_ = (N, m)
    if key_ not in _stride_cache:
        import numpy as np
        best = None
        idx = np.arange(m, dtype=np.int64)
        for d in sorted(range(-64, 65), key=abs):
            a = a0 + d
            if a < 1 or a >= N or math.gcd(a, N) != 1:
                continue
            p = np.sort((idx * a) % N)
            gap = int(max(np.diff(p).max(), p[0] + N - p[-1]))
            if best is None or gap < best[0]:
                best = (gap, a)
        _stride_cache[key_] = best[1] if best else _sample_stride(N)
    return _stride_cache[key_]


def _candidates_sym(xh, N, D, sp, dev, k=30):
    """Prepass (sample thresholds) + symmetric main pass.  Returns (cand, cand_cnt, tau_ord, cap, stats)."""
    m = sample_size(N, k)
    xs = torch.empty((m, D), dtype=torch.float16, device=dev)
    call("reid_features_sample", ptr(xh), N, D, m, _sample_stride(N, m), ptr(xs), sp)
    cand = torch.empty(N * max(2 * TC_CAP, SYM_CAP), dtype=torch.int64, device=dev)     # prepass lists, then main lists
    pre_cnt = torch.zeros(N * 2, dtype=torch.int32, device=dev)
    pre_tau = torch.empty(N, dtype=torch.int32, device=dev)
    call("reid_knn_candidates_tc_ab", ptr(xh), N, ptr(xs), m, D, SCALE_LOG2, 0, N, -sym_rank(k), 1, 2, ptr(cand), ptr(pre_cnt),
         ptr(pre_tau), sp)
    tau = torch.empty(N, dtype=torch.float32, device=dev)
    tau_ord = torch.empty(N, dtype=torch.int32, device=dev)
    call("reid_knn_sample_tau", ptr(cand), ptr(pre_cnt), ptr(pre_tau), 2, N, sym_rank(k), ptr(tau), ptr(tau_ord), sp)
    tiles = _tile_order((N + 255) // 256, dev)
    cnt = torch.empty(N, dtype=torch.int32, device=dev)
    candidates_sym_launch(xh, N, D, tau, tiles, SYM_CAP, cand, cnt, 1, sp)
    return cand, cnt, tau_ord, SYM_CAP, dict(sample=m, tiles=int(tiles.shape[0]))


SYM_SAMPLE_FIRST = True       # sample-first layout: the prepass scores are handed to the main lists and the symmetric pass
                              # skips the sample blocks (device-resident single-GPU search; see _candidates_sym_sf)
_sf_cache = {}
_side_streams = {}


def _side_stream(dev):
    """One forked stream per device (created once: a stream made under graph capture would not outlive it)."""
    key_ = str(dev)
    if key_ not in _side_streams:
        _side_streams[key_] = torch.cuda.Stream(device=dev)
    return _side_streams[key_]


def _sample_first_maps(N, m, dev):
    """(pos_of, orig_of) int32 device tensors of the sample-first layout: positions [0, m) hold the low-discrepancy
    sample rows (p * stride) mod N, positions [m, N) the other rows in their original order.  Cached per (N, m, dev)."""
    key_ = (N, m, str(dev))
    if key_ not in _sf_cache:
        import numpy as np
        samp = (np.arange(m, dtype=np.int64) * _sample_stride(N, m)) % N
        is_s = np.zeros(N, dtype=bool)
        is_s[samp] = True
        orig_of = np.concatenate([samp, np.flatnonzero(~is_s)]).astype(np.int32)
        pos_of = np.empty(N, dtype=np.int32)
        pos_of[orig_of] = np.arange(N, dtype=np.int32)
        _sf_cache[key_] = (torch.from_numpy(pos_of).to(dev), torch.from_numpy(orig_of).to(dev))
    return _sf_cache[key_]


def _tile_order_from(n_t, first, dev):
    """_tile_order over the blocks [first, n_t): the upper triangle without the sample blocks.  Cached."""
    key_ = ("from", n_t, first, str(dev))
    if key_ not in _tile_cache:
        _tile_cache[key_] = (_tile_order(n_t - first, "cpu") + first).to(dev).contiguous()
    return _tile_cache[key_]


def _sample_block_tiles(n_t, s_t, dev):
    """The tiles (I, J), I < s_t <= J: the block column of the sample against the other rows, column block by column
    block (the s_t sample blocks stay in L2, every other block is read by s_t tiles in a row).  Cached."""
    key_ = ("sample", n_t, s_t, str(dev))
    if key_ not in _tile_cache:
        out = [(i, j) for j in range(s_t, n_t) for i in range(s_t)]
        _tile_cache[key_] = torch.tensor(out, dtype=torch.int32).reshape(-1, 2).to(dev).contiguous()
    return _tile_cache[key_]


def _tau_floor(tau, tau_ord, m, N, sp):
    """tau[m:] = tau_ord[m:] = tau', the provisional threshold of the rows outside the sample: the smallest sample-row
    threshold (reid_knn_tau_floor).  A higher choice (the 8th or 32nd smallest of 2,048) measured no faster at
    N = 32,621: lists 2-3 % shorter, the same re-score time, and up to 30x more rows left at tau'."""
    call("reid_knn_tau_floor", ptr(tau), ptr(tau_ord), m, N, sp)


def _candidates_sym_sf(x, N, D, sp, dev, k, msq):
    """Symmetric search in the sample-first layout.  The fp16 operand is written with the m threshold-sample rows first,
    so the rows against the sample are the block column [0, m) of the similarity matrix:
      A. sample rows x sample  -> thresholds of the sample rows; their listed scores above the threshold are their
         candidates among the sample (reid_knn_sample_tau_emit).  Then tau' (_tau_floor) for the other rows;
      B. the symmetric kernel on the tiles (I, J), I < m / 256 <= J (reid_knn_candidates_sym_tiles): sample row i lists
         column j above its threshold, row j lists sample column i above tau'.  reid_knn_list_tau then raises tau' of
         row j to the r-th best of its listed sample scores (they are all of them above tau');
      C. the symmetric kernel on the tiles (I, J), m / 256 <= I <= J, appending to the same lists.
    Every pair of rows is scored exactly once; all lists and thresholds are indexed by POSITION (reid_knn_rescore_mapped
    translates).  Needs m % 256 == 0 and N - m >= 256.  Returns (cand, cnt, tau_ord, cap, stats, xh, maps)."""
    m = sample_size(N, k)
    pos_of, orig_of = _sample_first_maps(N, m, dev)
    xh = torch.empty((N, D), dtype=torch.float16, device=dev)
    r = sym_rank(k)
    cand = torch.empty(N * SYM_CAP, dtype=torch.int64, device=dev)
    cnt = torch.zeros(N, dtype=torch.int32, device=dev)
    tau = torch.empty(N, dtype=torch.float32, device=dev)
    tau_ord = torch.empty(N, dtype=torch.int32, device=dev)
    n_rest = N - m
    splits_a = prepass_splits(m, m, max_splits=8)
    # fp16 operand, sample rows first.  Phase A needs only those: it runs on a forked stream (64 tile units for 74 CTA
    # pairs, tensor bound) under the conversion of the other rows (HBM bound); with its own list buffers.
    call("reid_sqnorm_range_reset", ptr(msq), sp)
    call("reid_features_to_half_gather", ptr(x), ptr(orig_of), m, D, SCALE_LOG2, ptr(xh), ptr(msq), sp)
    pre_a = torch.empty(m * 2 * splits_a * TC_CAP, dtype=torch.int64, device=dev)
    pre_a_cnt = torch.zeros(m * 2 * splits_a, dtype=torch.int32, device=dev)
    pre_a_tau = torch.empty(m, dtype=torch.int32, device=dev)
    main = torch.cuda.current_stream()
    side = _side_stream(dev)
    side.wait_stream(main)
    with torch.cuda.stream(side):
        sp_a = stream_ptr()
        # A: the sample rows against the sample (a few row units: their columns are split over CTA pairs)
        call("reid_knn_candidates_tc_abt", ptr(xh), N, ptr(xh), m, D, SCALE_LOG2, 0, m, -r, splits_a, 2, ptr(pre_a), ptr(pre_a_cnt),
             ptr(pre_a_tau), 1, None, None, None, 0, sp_a)
        call("reid_knn_sample_tau_emit", ptr(pre_a), ptr(pre_a_cnt), ptr(pre_a_tau), 2 * splits_a, m, r, ptr(tau), ptr(tau_ord),
             ptr(cand), ptr(cnt), SYM_CAP, 0, sp_a)
        _tau_floor(tau, tau_ord, m, N, sp_a)
    call("reid_features_to_half_gather", ptr(x), ptr(orig_of[m:]), n_rest, D, SCALE_LOG2, ptr(xh[m:]), ptr(msq), sp)
    main.wait_stream(side)
    # B: the sample block column, both directions, then the other rows' thresholds
    n_t = (N + 255) // 256
    b_tiles = _sample_block_tiles(n_t, m // 256, dev)
    call("reid_knn_candidates_sym_tiles", ptr(xh), N, D, SCALE_LOG2, ptr(tau), ptr(b_tiles), b_tiles.shape[0], SYM_CAP, ptr(cand),
         ptr(cnt), 0, sp)
    call("reid_knn_list_tau", ptr(cand), ptr(cnt), SYM_CAP, m, n_rest, r, ptr(tau), ptr(tau_ord), sp)
    # C: the rest of the upper triangle
    tiles = _tile_order_from(n_t, m // 256, dev)
    candidates_sym_launch(xh, N, D, tau, tiles, SYM_CAP, cand, cnt, 0, sp)
    return cand, cnt, tau_ord, SYM_CAP, dict(sample=m, tiles=int(tiles.shape[0]), layout="sample-first"), xh, (pos_of, orig_of)


def sym_eligible(N, D, k):
    return SYM and N >= SYM_MIN_N and k <= SYM_MAX_K and D % 64 == 0


UPLOAD_CHUNKS = None          # None: about five 256-row blocks per chunk, 4..24 chunks (measured: scripts/dev_e2e_ab.py --
                              # N = 32,621: 12 -> 7.51, 24 -> 7.45, 32 -> 7.64, 48 -> 8.6 ms; N = 12,936: 8-12 best)


def upload_bounds(n_t, chunks):
    """Block boundaries (in 256-row tile blocks, chunks + 1 of them) of the chunked upload: equal chunks.  Chunks that
    shrink towards the end (so that less tensor work is left when the last byte lands) were measured and are slower
    (7.80 vs 7.58 ms end to end, scripts/dev_e2e_ab.py): every chunk carries ~0.15 ms of fixed latency -- conversion,
    a prepass that runs at the latency of one row unit, the thresholds, a partial wave of tiles -- and the small last
    chunks put that, not their tiles, behind the copy."""
    return [n_t * c // chunks for c in range(chunks)] + [n_t]


def knn_search_upload(x_host, k, dev, idx=None, key=None, info=None, defer=False, chunks=None, uncert_count=None):
    """a1 for features that still live in (pinned) HOST memory: the upload is cut into `chunks` row blocks on a copy
    stream and the candidate search follows it block by block -- fp16 conversion, sampling prepass and thresholds
    of the block's rows, then every upper-triangle tile whose rows are all resident -- so that when the last block
    lands only its own share of the tiles is left.  The threshold sample (rows at two interleaved regular strides,
    one cudaMemcpy2DAsync each) goes up first.  Returns (x_dev, idx, key, info); same results as knn_search."""
    L = _lib.lib()
    N, D = x_host.shape
    if chunks is None:
        chunks = UPLOAD_CHUNKS if UPLOAD_CHUNKS else max(4, min(24, ((N + 255) // 256) // 5))
    assert x_host.dtype == torch.float32 and x_host.is_contiguous() and not x_host.is_cuda
    info = {} if info is None else info
    main = torch.cuda.current_stream()
    copy = torch.cuda.Stream(device=dev)
    sp = stream_ptr()
    x = torch.empty((N, D), dtype=torch.float32, device=dev)
    xh = torch.empty((N, D), dtype=torch.float16, device=dev)
    msq = new_sqnorm_range(dev)
    # sample: two interleaved regular strides (odd, different) so that no single period of the row order can bias it
    m = sample_size(N, k)
    s = max(2, N // m)
    halves = [(0, 2 * s - 1), (s // 2, 2 * s - 3 if s > 2 else 2 * s - 1)]
    rows_h = [min(m // 2, (N - 1 - o) // st + 1) for o, st in halves]
    m = sum(rows_h)
    xs32 = torch.empty((m, D), dtype=torch.float32, device=dev)
    xs = torch.empty((m, D), dtype=torch.float16, device=dev)
    n_t = (N + 255) // 256
    bounds = [min(N, 256 * t) for t in upload_bounds(n_t, chunks)[:-1]] + [N]
    copy.wait_stream(main)                       # the destination buffers were just allocated on `main`
    events = []
    with torch.cuda.stream(copy):
        cp = ctypes.c_void_p(copy.cuda_stream)
        base = x_host.data_ptr()
        done = 0
        for (o, st), nr in zip(halves, rows_h):
            call("reid_upload_rows_strided", ptr(xs32[done:]), ctypes.c_void_p(base + o * D * 4), D * 4, st * D * 4, nr, cp)
            done += nr
        ev_s = torch.cuda.Event()
        ev_s.record(copy)
        for c in range(chunks):
            a, b = bounds[c], bounds[c + 1]
            if b > a:
                x[a:b].copy_(x_host[a:b], non_blocking=True)
            e = torch.cuda.Event()
            e.record(copy)
            events.append(e)
    main.wait_event(ev_s)
    msq_s = torch.zeros(2, dtype=torch.float32, device=dev)
    call("reid_features_to_half", ptr(xs32), m, D, SCALE_LOG2, ptr(xs), ptr(msq_s), sp)
    cand = torch.empty(N * SYM_CAP, dtype=torch.int64, device=dev)
    cnt = torch.zeros(N, dtype=torch.int32, device=dev)
    tau = torch.empty(N, dtype=torch.float32, device=dev)
    tau_ord = torch.empty(N, dtype=torch.int32, device=dev)
    chunks = len(bounds) - 1
    max_rows = max(bounds[c + 1] - bounds[c] for c in range(chunks))
    splits = prepass_splits(max_rows, m)         # a chunk is ~11 row units for 74 CTA-pair slots: split its sample columns
    pre = torch.empty(max_rows * 2 * splits * TC_CAP, dtype=torch.int64, device=dev)
    pre_cnt = torch.empty(max_rows * 2 * splits, dtype=torch.int32, device=dev)
    pre_tau = torch.empty(max_rows, dtype=torch.int32, device=dev)
    order = _tile_order(n_t, dev)
    n_tiles = 0
    for c in range(chunks):
        a, b = bounds[c], bounds[c + 1]
        main.wait_event(events[c])
        if b <= a:
            continue
        call("reid_features_to_half_acc", ptr(x[a:]), b - a, D, SCALE_LOG2, ptr(xh[a:]), ptr(msq), sp)
        pre_cnt.zero_()
        call("reid_knn_candidates_tc_ab", ptr(xh), N, ptr(xs), m, D, SCALE_LOG2, a, b, -sym_rank(k), splits, 2, ptr(pre), ptr(pre_cnt),
             ptr(pre_tau), sp)
        call("reid_knn_sample_tau", ptr(pre), ptr(pre_cnt), ptr(pre_tau), 2 * splits, b - a, sym_rank(k), ptr(tau[a:]), ptr(tau_ord[a:]), sp)
        key_ = ("chunk", n_t, chunks, c, str(dev))
        if key_ not in _tile_cache:                            # tiles whose larger block index falls into this chunk
            t0, t1 = a // 256, (b + 255) // 256
            sel = (order[:, 1] >= t0) & (order[:, 1] < t1)
            _tile_cache[key_] = order[sel].contiguous()
        tiles = _tile_cache[key_]
        n_tiles += int(tiles.shape[0])
        if tiles.shape[0]:
            candidates_sym_launch(xh, N, D, tau, tiles, SYM_CAP, cand, cnt, 0, sp)
    if idx is None:
        idx = torch.empty((N, k), dtype=torch.int32, device=dev)
        key = torch.empty((N, k), dtype=torch.float32, device=dev)
    x.record_stream(copy)
    idx, key, info = knn_search_tc(x, k, 0, N, idx, key, info, xh=xh, defer=defer, uncert_count=uncert_count,
                                   cands=(cand, cnt, tau_ord, SYM_CAP, dict(sample=m, tiles=n_tiles, chunks=chunks), msq))
    return x, idx, key, info


def knn_search_tc(x, k, r0, r1, idx, key, info, xh=None, max_sqnorm=None, defer=False, cands=None, uncert_count=None):
    L = _lib.lib()
    from .faiss_rerank import _knn_exact_rows
    N, D = x.shape
    dev = x.device
    n = r1 - r0
    sp = stream_ptr()
    sym = SYM and r0 == 0 and r1 == N and N >= SYM_MIN_N and k <= SYM_MAX_K
    maps = None
    sf = None
    if cands is None and xh is None and sym and SYM_SAMPLE_FIRST and sample_size(N, k) % 256 == 0 and N - sample_size(N, k) >= 256:
        msq = torch.zeros(2, dtype=torch.float32, device=dev)
        sf = _candidates_sym_sf(x, N, D, sp, dev, k, msq)
        xh, maps = sf[5], sf[6]
        max_sqnorm = None
    elif cands is not None:
        msq = cands[5]
        max_sqnorm = None
    elif xh is None:
        xh = torch.empty((N, D), dtype=torch.float16, device=dev)
        msq = torch.zeros(2, dtype=torch.float32, device=dev)
        call("reid_features_to_half", ptr(x), N, D, SCALE_LOG2, ptr(xh), ptr(msq), sp)
        max_sqnorm = None
    else:
        msq = None
    keep = max(k, min(k + SLACK, KEEP_MAX))
    if sf is not None:
        cand, cand_cnt, row_tau, list_cap, sym_info = sf[:5]
        n_lists, s = 1, 0
    elif cands is not None:
        cand, cand_cnt, row_tau, list_cap, sym_info = cands[:5]
        n_lists, s, sym = 1, 0, True
    elif sym:
        cand, cand_cnt, row_tau, list_cap, sym_info = _candidates_sym(xh, N, D, sp, dev, k)
        n_lists, s = 1, 0
    else:
        n_splits = ctypes.c_int(1)
        call("reid_knn_tc_plan", N, n, CTA_GROUP, ctypes.byref(n_splits))
        s = n_splits.value
        n_lists = 2 * s                                        # two epilogue groups per column range
        list_cap, sym_info = TC_CAP, None
        cand = torch.empty(n * n_lists * TC_CAP, dtype=torch.int64, device=dev)
        cand_cnt = torch.zeros(n * n_lists, dtype=torch.int32, device=dev)
        row_tau = torch.empty(n, dtype=torch.int32, device=dev)
        call("reid_knn_candidates_tc", ptr(xh), N, D, SCALE_LOG2, r0, r1, keep, s, CTA_GROUP, ptr(cand), ptr(cand_cnt), ptr(row_tau), sp)
    eps = err_bound(max_sqnorm) if max_sqnorm is not None else 0.0   # else derived on device from msq
    flag = torch.empty(n, dtype=torch.int32, device=dev)
    max_err = torch.zeros(1, dtype=torch.float32, device=dev)
    ws = torch.empty(L.reid_knn_rescore_workspace_bytes(N, n), dtype=torch.uint8, device=dev)
    if maps is not None:      # the lists live in the sample-first positions
        call("reid_knn_rescore_mapped", ptr(x), N, D, r0, r1, ptr(cand), ptr(cand_cnt), ptr(row_tau), n_lists, list_cap, 0, k, eps,
             ptr(msq), 1 if ORDER_ROWS else 0, ptr(maps[0]), ptr(maps[1]), ptr(idx), ptr(key), ptr(flag), ptr(max_err), ptr(ws),
             ptr(uncert_count), sp)
    else:
        call("reid_knn_rescore", ptr(x), N, D, r0, r1, ptr(cand), ptr(cand_cnt), ptr(row_tau), n_lists, list_cap, 0, k, eps,
             ptr(msq), 1 if ORDER_ROWS else 0, ptr(idx), ptr(key), ptr(flag), ptr(max_err), ptr(ws), ptr(uncert_count), sp)

    def repair():
        """Exact CUDA-core search for the rows the certificate rejected (none on typical data)."""
        bad = torch.nonzero(flag).flatten().to(torch.int32)
        nb = bad.numel()
        if nb:
            rows = (bad + r0).contiguous()
            bi = torch.empty((nb, k), dtype=torch.int32, device=dev)
            bk = torch.empty((nb, k), dtype=torch.float32, device=dev)
            _knn_exact_rows(x, k, rows, 0, nb, bi, bk)
            idx[bad.long()] = bi
            key[bad.long()] = bk
        return nb

    if defer:            # the caller folds the flag count into its next read-back and calls repair() if needed
        n_bad = 0
        info["pending"] = dict(flag=flag, repair=repair)
    else:
        n_bad = repair()
    off = L.reid_knn_rescore_window_counts_offset(N, n)
    info["window_counts"] = ws[off:off + 4 * n].view(torch.int32)     # window size per row (reporting only)
    if ORDER_ROWS:                                                    # cluster-locality order of the rows (for a4)
        off = L.reid_knn_rescore_order_offset(N, n)
        info["visit_order"] = ws[off:off + 4 * n].view(torch.int32)
    info.update(mode="tc-sym" if sym else "tc", sym=sym_info, cand_cnt=cand_cnt if sym else None, cta_group=CTA_GROUP, n_splits=s, keep=keep, err_bound=eps if msq is None else None, max_sqnorm=msq, uncertified_rows=int(n_bad),
                max_abs_err=max_err, xh=xh)
    return idx, key, info
