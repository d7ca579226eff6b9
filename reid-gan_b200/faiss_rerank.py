"""Drop-in for clustercontrast/utils/faiss_rerank.py (reference lines cited per stage).

    compute_jaccard_distance(target_features, k1=20, k2=6, print_flag=True,
                             search_option=0, use_float16=False)

Same call surface as faiss_rerank.py:30.  Everything runs on the current CUDA device through
libreid_b200.so; there is no faiss, no backend dispatch (`search_option` is accepted and
validated, every value runs the same kernels) and no CPU fallback.

The reference returns a dense host float32 (N, N) matrix (:123).  Here the function returns a
`JaccardDistance`: a lazy view of that matrix.  `np.asarray(d)`, indexing, `.shape`,
`.dtype`, arithmetic ... materialise exactly the reference's matrix on first use, while
`reid_gan_b200.DBSCAN.fit_predict(d)` consumes the device-resident sparse form and never
builds the N x N matrix (4.26 GB and ~100 ms of PCIe at N = 32,621).
"""
import time

import numpy as np
import torch

from . import _lib
from ._lib import call, check, ptr, stream_ptr


TC_AVAILABLE = True      # the tcgen05 candidate kernel (csrc/simgemm_tc.cu) is part of the library


def half_k(k1):
    """faiss_rerank.py:69 -- int(np.around(k1/2)): round-half-to-even."""
    return int(np.around(k1 / 2))


def _device_of(t):
    if not torch.cuda.is_available():
        raise RuntimeError("reid_gan_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    if isinstance(t, torch.Tensor) and t.is_cuda:
        return t.device
    return torch.device("cuda", torch.cuda.current_device())


def _scan_async(cnt, n, dev, stats=None):
    """counts (int32, device) -> (ptr int64 (n+1), stats int64 (3) = [total, max, sum of squares]) -- no host sync.
    `stats`: an existing 3-element int64 device view to write into (a slice of a pass report)."""
    out = torch.empty(n + 1, dtype=torch.int64, device=dev)
    if stats is None:
        stats = torch.empty(3, dtype=torch.int64, device=dev)
    call("reid_scan_counts", ptr(cnt), n, ptr(out), ptr(stats), stream_ptr())
    return out, stats


def _scan(cnt, n, dev):
    """counts (int32, device) -> (ptr int64 (n+1), total, max) -- one small host sync."""
    out, stats = _scan_async(cnt, n, dev)
    total, mx, _ = stats.tolist()
    return out, int(total), int(mx)


# ---- speculative sizes of the sync-free single-GPU pass ---------------------------------------------------------
# A pass that reads sizes back between stages leaves the GPU idle for every round trip.  The single-GPU pass instead
# allocates upper bounds where a cheap one exists (|E| <= k1 + k1 (h + 1), nnz(V_qe) <= rows x table slots), guesses
# the two sizes that have no useful bound (the query-expansion table and the eps-neighbour slots), lets every kernel
# REPORT what did not fit instead of trusting the guess, and reads one small report at the END of the pass
# (RerankState.finish): a pass whose guesses held never synchronised in between, any other is redone with exact sizes.
QE_SPEC_SLOTS = 512          # query-expansion table / padded V_qe row (distinct columns <= 3/4 of it)
PARTNER_GUESS = True         # size each row's first Jaccard hash table from 3 x longest column + nnz (reid_jaccard_bounds P_cnt)
NBR_SPEC_PER_ROW = 256       # eps-neighbour slots per row on average (slots are dealt by the Markov bound S_i)
_nbr_cap_hint = {}           # N -> slot total of the last finished pass (the next pass allocates 1.25 x that)
# report (int64 x 16): [0:3] |E| total/max/sumsq  [3:6] nnz(V_qe) rows  [6:9] column counts: nnz, longest, sum len^2
#                      [9] uncertified kNN rows  [10] V_qe rows that overflowed the table  [11] rows that overflowed
#                      their eps-neighbour slots  [12:15] slot total/max/sumsq
#                      [15] rows that did not fit a fixed-stride exchange record (row-sharded pass)
#                      [16] rows the eps-graph stage had to move to a bigger hash table (the partner guess was too small)
R_E, R_Q, R_C, R_UNCERT, R_QE_OVF, R_NBR_OVF, R_S, R_XCHG_OVF, R_ESC = 0, 3, 6, 9, 10, 11, 12, 15, 16
REPORT_WORDS = 24
_guess_hint = {}             # N -> False once more than 3/4 of the rows outgrew the partner guess (Market-like shapes: 98 %;
                             # the hard set, where the guess still pays, 55 %)


def partner_guess_on(N):
    return PARTNER_GUESS and _guess_hint.get(N, True)
REC_STRIDE = {"V": 64, "Q": 128, "nbr": 128}     # exchange record strides of the row-sharded pass (entries per row)
_rec_stride_hint = {}        # (kind, N) -> longest row of the last finished pass


class RerankState:
    """Device-resident intermediates of one re-ranking pass (rows [row_begin,row_end) of N)."""

    def __init__(self):
        self.N = self.D = self.k1 = self.k2 = 0
        self.row_begin = self.row_end = 0
        self.rank = self.rank_key = None          # (N, k1) int32 / float32   faiss_rerank.py:62
        self.R_mask = self.Rh_mask = None         # uint64 bit masks           :65-69
        self.E_ptr = self.E_idx = self.V_val = None      # CSR of V            :72-85
        self.Q_ptr = self.Q_idx = self.Q_val = None      # CSR of V_qe         :89-94
        self.C_ptr = self.C_idx = self.C_val = None      # CSC of V_qe         :98-100
        self.timings = {}
        self.knn_info = {}
        self.report = None                        # device report of a speculative pass, until finish()
        self.report_vals = None
        self._redo = None

    def finish(self, check_nbr=False):
        """End of a speculative pass: ONE read-back of the report.  Returns the state to use: `self` when every guess
        held, else a new state recomputed with exact sizes (uncertified kNN rows are searched exactly first).
        check_nbr: also require that no row overflowed its eps-neighbour slots (-> (state, nbr_ok))."""
        if self.report is None:
            return (self, True) if check_nbr else self
        if getattr(self, "_comm", None) is not None:
            # every rank must take the same decision: the flags of the own rows are maximised over the ranks first
            import torch.distributed as dist
            dist.all_reduce(self.report, op=dist.ReduceOp.MAX, group=self._comm.group)
        vals = [int(v) for v in self.report.tolist()]
        self.report, self.report_vals = None, vals
        if getattr(self, "_check_norms", False) and not _one_norm_info(self.knn_info, self.x):
            st = self._redo("l2")
            self._redo = None
            return (st, False) if check_nbr else st
        self.knn_info["uncertified_rows"] = vals[R_UNCERT]
        if vals[R_E + 1] > self.e_stride:
            raise RuntimeError("reid_expand: an expansion set exceeded %d entries" % self.e_stride)
        ok = vals[R_UNCERT] == 0 and vals[R_QE_OVF] == 0 and vals[R_XCHG_OVF] == 0
        if ok:
            self.e_total, self.e_max = vals[R_E], vals[R_E + 1]
            self.q_total, self.c_max, self.t_total_all = vals[R_C], vals[R_C + 1], vals[R_C + 2]
            if vals[R_S]:
                _nbr_cap_hint[self.N] = vals[R_S]
                if PARTNER_GUESS and self.N not in _guess_hint and vals[R_ESC] * 4 > 3 * (self.row_end - self.row_begin):
                    _guess_hint[self.N] = False
            nbr_ok = vals[R_NBR_OVF] == 0
            return (self, nbr_ok) if check_nbr else self
        st = self._redo(vals)
        self._redo = None
        return (st, False) if check_nbr else st


def knn_search(x, k, mode="auto", rows=None, defer=False, uncert_count=None, metric="auto"):
    """a1: exact top-k neighbour lists (faiss_rerank.py:58-62).  Returns (idx int32, key fp32, info).
    mode "exact": CUDA-core fp64 search for every row; "tc": tensor-core candidates + exact
    re-score + certificate, uncertified rows redone exactly; "auto": "tc" when the shape allows.
    metric: the reference searches by squared L2 (IndexFlatL2).  "auto" = inner-product key when all rows have one norm
    (then both orders agree; the backbone L2-normalises, models/resnet.py:90-94), squared-L2 key otherwise; "ip" / "l2"
    force one (get_dist_nbr's IndexFlatIP is "ip").  info["metric"] tells which key `key` holds.
    defer: do not read anything back: info["pending"] holds the certificate flags and the repair closure,
    info["max_sqnorm"] the {max, min} squared norms the caller must check (knn_tc.one_norm); uncert_count: device
    scalar that receives the number of uncertified rows."""
    from .knn_tc import one_norm, sqnorm_range_of
    L = _lib.lib()
    N, D = x.shape
    dev = x.device
    if rows is None:
        r0, r1 = 0, N
    else:
        r0, r1 = rows
    n = r1 - r0
    idx = torch.empty((n, k), dtype=torch.int32, device=dev)
    key = torch.empty((n, k), dtype=torch.float32, device=dev)
    info = {"mode": mode, "uncertified_rows": 0, "metric": "ip"}
    if metric not in ("auto", "ip", "l2"):
        raise ValueError("unknown metric %r" % (metric,))
    if mode == "auto":
        mode = "tc" if (TC_AVAILABLE and D % 64 == 0 and N >= 256 and k <= 64 and metric != "l2") else "exact"
        info["mode"] = mode
    if mode == "tc":
        if metric == "l2":
            raise ValueError("the tensor-core search ranks by inner product; metric='l2' needs mode 'exact'")
        from .knn_tc import knn_search_tc
        idx, key, info = knn_search_tc(x, k, r0, r1, idx, key, info, defer=defer, uncert_count=uncert_count)
        info["metric"] = "ip"
        if metric == "auto" and not defer and not one_norm(sqnorm_range_of(x, info["max_sqnorm"])):
            _knn_exact_rows(x, k, None, r0, n, idx, key, metric="l2")      # rows of different norms: squared-L2 key
            info.update(mode="exact-l2", metric="l2", visit_order=None, uncertified_rows=0)
        return idx, key, info
    if mode != "exact":
        raise ValueError("unknown kNN mode %r" % (mode,))
    if metric == "auto":
        rng = torch.empty(2, dtype=torch.float32, device=dev)
        call("reid_sqnorm_range", ptr(x), N, D, ptr(rng), stream_ptr())
        metric = "ip" if one_norm(rng.tolist()) else "l2"
    _knn_exact_rows(x, k, None, r0, n, idx, key, metric=metric)
    info["metric"] = metric
    if metric == "l2":
        info["mode"] = "exact-l2"
    return idx, key, info


def _knn_exact_rows(x, k, rows_list, row_begin, n_rows, idx_out, key_out, metric="ip"):
    L = _lib.lib()
    N, D = x.shape
    if n_rows == 0:
        return
    budget = 1 << 30                                        # ~1 GiB of key rows per pass
    chunk = max(1, min(n_rows, budget // (4 * N)))
    head = (N * 8 + 255) // 256 * 256 if metric == "l2" else 0
    scratch = torch.empty(head + chunk * N * 4, dtype=torch.uint8, device=x.device)
    call("reid_knn_exact_l2" if metric == "l2" else "reid_knn_exact", ptr(x), N, D, ptr(rows_list), row_begin, n_rows, k,
         ptr(idx_out), ptr(key_out), ptr(scratch), scratch.numel(), stream_ptr())


def _check_shape(x, k1, k2):
    N, D = x.shape
    if not (1 <= k1 <= 64):
        raise ValueError("k1=%d outside the supported range 1..64" % k1)
    if k1 > N:
        raise ValueError("k1=%d exceeds the number of samples N=%d" % (k1, N))
    if not (1 <= k2 <= k1):
        raise ValueError("k2=%d must be in 1..k1" % k2)


def rerank_state_async(x, k1, k2, knn="auto", rows=None, timers=False, comm=None, knn_result=None, speculative=None,
                       metric="auto", half=False, report=None):
    """Run a1-a6 on device.  Single GPU: all rows.  Row-sharded (comm = sharded.RowComm): this rank
    computes rows [comm.r0, comm.r1) of every per-row stage and the stages' outputs are all-gathered
    (neighbour lists, V rows, V_qe rows), so the returned state always holds GLOBAL rank / V / V_qe /
    inverted index while `row_begin:row_end` remembers the rank's own rows.

    speculative (default: on for the unsharded pass): no host read-back between the stages -- sizes are upper
    bounds or guesses checked on the device, and the caller ends the pass with `st = st.finish()` (one read-back;
    see RerankState.finish).  speculative=False reads the sizes back where they are needed (two round trips)."""
    L = _lib.lib()
    assert (x.is_cuda or knn_result == "upload") and x.dtype == torch.float32 and x.is_contiguous()
    N, D = x.shape
    _check_shape(x, k1, k2)
    dev = x.device if x.is_cuda else torch.device("cuda", torch.cuda.current_device())
    if comm is not None:
        r0, r1 = comm.r0, comm.r1
    else:
        r0, r1 = (0, N) if rows is None else rows
    n = r1 - r0
    full = comm is None and r0 == 0 and r1 == N
    if speculative is None:
        speculative = full or (comm is not None and knn_result not in (None, "upload") and x.is_cuda)
    if speculative and not (full or comm is not None):
        raise ValueError("the speculative pass covers all rows of one GPU, or a communicator's row shard")
    st = RerankState()
    st._comm = comm
    st.N, st.D, st.k1, st.k2, st.row_begin, st.row_end = N, D, k1, k2, r0, r1
    st.half = bool(half)                                      # use_float16=True: fp16 roundings of V, V_qe, sums, J
    hp = 1 if half else 0
    sp = stream_ptr()
    ev = []

    def mark(name):
        if timers:
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            ev.append((name, e))

    external_knn = knn_result not in (None, "upload")
    if report is None:                                        # else: shared with the caller's search (sharded.py)
        report = torch.zeros(REPORT_WORDS, dtype=torch.int64, device=dev)
    mark("start")
    # a1 ------------------------------------------------------------------
    if knn_result == "upload":                               # x is still on the host: search while it is uploaded
        from .knn_tc import knn_search_upload
        x, rank_local, key_local, info = knn_search_upload(x, k1, dev, defer=True, uncert_count=report[R_UNCERT:])
        knn_result = None
    elif knn_result is not None:                             # searched elsewhere (sharded.knn_search_tiles): rows r0:r1 of it
        rank_g, key_g, info = knn_result
        rank_local, key_local = rank_g[r0:r1].contiguous(), key_g[r0:r1].contiguous()
    else:
        # unsharded: the certificate flags are not read back here -- their count rides on the pass report (or, in
        # the exact-size flavour, on the first unavoidable read-back); the rare uncertified rows are then repaired
        rank_local, key_local, info = knn_search(x, k1, knn, rows=(r0, r1), defer=comm is None,
                                                 uncert_count=report[R_UNCERT:], metric=metric)
    st.knn_info = info
    st.x = x
    if knn_result is not None:
        rank = knn_result[0].contiguous()
    else:
        rank = comm.gather_rows(rank_local) if comm is not None else rank_local  # global (N, k1)
    if rank.shape[0] != N:
        raise ValueError("a row shard needs the global neighbour lists (knn_result or comm)")
    st.rank, st.rank_key = rank, key_local
    mark("knn")
    h = half_k(k1)
    e_stride = min(k1 + k1 * (h + 1), 1024)                  # |E| <= |R| + |R| * |R_half|
    st.e_stride = e_stride
    R = torch.empty(max(n, 1), dtype=torch.int64, device=dev)
    Rh = torch.empty(N, dtype=torch.int64, device=dev)        # every rank needs R_half of all rows
    e_pad = torch.empty(max(n, 1) * e_stride, dtype=torch.int32, device=dev)
    e_cnt = torch.empty(max(n, 1), dtype=torch.int32, device=dev)

    def sets():
        # a2 ------------------------------------------------------------------
        call("reid_reciprocal_masks2", ptr(rank), N, k1, k1, h, r0, r1, ptr(R), ptr(Rh), sp)
        # a3 ------------------------------------------------------------------
        call("reid_expand", ptr(rank), N, k1, min(h + 1, k1), ptr(R), ptr(Rh), r0, r1, e_stride, ptr(e_pad), ptr(e_cnt), sp)
        return _scan_async(e_cnt, n, dev, stats=report[R_E:R_E + 3])

    e_ptr, e_stats = sets()
    pending = info.pop("pending", None)
    st.R_mask, st.Rh_mask = R, Rh
    mark("reciprocal")
    if speculative:
        e_total = e_max = None
        e_cap = max(n, 1) * e_stride                          # upper bound: no size needed on the host
    else:
        vals = report.tolist()                                # read-back 1 of 2: |E| sizes + certificate count
        if pending is not None and metric == "auto" and not _one_norm_info(info, x):
            # rows of different norms: the reference's L2 order is not the inner-product order that was searched
            return rerank_state_async(x, k1, k2, knn="exact", timers=timers, speculative=False, metric="l2", half=half)
        if pending is not None and vals[R_UNCERT]:            # uncertified rows: exact search for them, then redo a2/a3
            pending["repair"]()
            info["visit_order"] = None                        # only valid for the lists it was built from
            e_ptr, e_stats = sets()
            n_bad = vals[R_UNCERT]
            vals = report.tolist()
            info["uncertified_rows"] = int(n_bad)
        e_total, e_max = int(vals[R_E]), int(vals[R_E + 1])
        if e_max > e_stride:
            raise RuntimeError("reid_expand: an expansion set exceeded %d entries" % e_stride)
        e_cap = max(e_total, 1)
    mark("expand")
    # a4 ------------------------------------------------------------------
    e_idx = torch.empty(e_cap, dtype=torch.int32, device=dev)
    v_val = torch.empty(e_cap, dtype=torch.float32, device=dev)
    order = info.get("visit_order") if knn_result is None else None
    if order is not None and order.numel() != n:
        order = None                                          # only valid for exactly these rows
    # members that are among the row's k1 neighbours re-use the search key -- when that key IS the dot product
    reuse = info.get("metric", "ip") == "ip"
    call("reid_v_weights", ptr(x), N, D, ptr(e_pad), e_stride, ptr(e_ptr), r0, r1, ptr(rank_local) if reuse else None,
         ptr(key_local) if reuse else None, k1, ptr(order), ptr(e_idx), ptr(v_val), hp, sp)
    mark("v_weights")
    if comm is not None and speculative:                     # V rows of other shards are read by a5
        sv = _stride_for("V", N)
        e_ptr, e_idx, v_val = comm.gather_records(e_cnt[:n], e_ptr, e_idx, v_val, sv, overflow=report[R_XCHG_OVF:],
                                                  stats_out=report[R_E:R_E + 3], tag="V")[:3]
    elif comm is not None:
        e_ptr, e_idx, v_val, e_total, e_max = comm.gather_csr(e_cnt[:n], e_idx[:e_total], v_val[:e_total], row_ptr=e_ptr)
        _rec_stride_hint[("V", N)] = max(_rec_stride_hint.get(("V", N), 0), int(e_max))
    elif not full:                                           # a row shard without a communicator (tests): a5 cannot run
        st.E_ptr, st.E_idx, st.V_val, st.e_total, st.e_max = e_ptr, e_idx, v_val, e_total, e_max
        return st
    st.E_ptr, st.E_idx, st.V_val = e_ptr, e_idx, v_val       # global CSR when sharded
    st.e_total, st.e_max = e_total, e_max
    # a5 ------------------------------------------------------------------
    if k2 != 1:
        if speculative:
            q_stride = QE_SPEC_SLOTS
            nnz_guess = max(1, (QE_SPEC_SLOTS - QE_SPEC_SLOTS // 4) // k2)    # reid_query_expand_stride(k2, guess) == 512
        else:
            q_stride = L.reid_query_expand_stride(k2, max(e_max, 1))
            nnz_guess = max(e_max, 1)
        q_cnt = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
        qp_idx = torch.empty(max(n, 1) * q_stride, dtype=torch.int32, device=dev)
        qp_val = torch.empty(max(n, 1) * q_stride, dtype=torch.float32, device=dev)
        call("reid_query_expand", ptr(rank), N, k1, k2, ptr(e_ptr), ptr(e_idx), ptr(v_val), nnz_guess, r0, r1,
             ptr(q_cnt), ptr(qp_idx), ptr(qp_val), ptr(report[R_QE_OVF:]), hp, sp)
        if comm is None or speculative:
            # no read-back here -- the CSR is compacted into upper-bound storage and nnz stays on the device (the
            # exact-size flavour reads it with the inverted index's sizes: one read-back for a5 + a6)
            q_ptr, q_stats = _scan_async(q_cnt, n, dev, stats=report[R_Q:R_Q + 3] if comm is None else None)
            q_idx = torch.empty(max(n, 1) * q_stride, dtype=torch.int32, device=dev)
            q_val = torch.empty(max(n, 1) * q_stride, dtype=torch.float32, device=dev)
            q_total = None
        else:
            q_ptr, q_total, _ = _scan(q_cnt, n, dev)
            q_idx = torch.empty(max(q_total, 1), dtype=torch.int32, device=dev)
            q_val = torch.empty(max(q_total, 1), dtype=torch.float32, device=dev)
        call("reid_csr_compact", ptr(qp_idx), ptr(qp_val), q_stride, ptr(q_cnt), ptr(q_ptr), n, ptr(q_idx), ptr(q_val), sp)
        if comm is not None and speculative:
            sq = _stride_for("Q", N)
            q_ptr, q_idx, q_val = comm.gather_records(q_cnt[:n], q_ptr, q_idx, q_val, sq, overflow=report[R_XCHG_OVF:],
                                                      stats_out=report[R_Q:R_Q + 3], tag="Q")[:3]
        elif comm is not None:
            q_ptr, q_idx, q_val, q_total, q_mx = comm.gather_csr(q_cnt[:n], q_idx[:q_total], q_val[:q_total], row_ptr=q_ptr)
            _rec_stride_hint[("Q", N)] = max(_rec_stride_hint.get(("Q", N), 0), int(q_mx))
    else:                                                    # faiss_rerank.py:89: skipped when k2 == 1
        q_ptr, q_idx, q_val, q_total = e_ptr, e_idx, v_val, e_total
    st.Q_ptr, st.Q_idx, st.Q_val = q_ptr, q_idx, q_val        # global CSR (N + 1)
    mark("query_expand")
    # a6 (replicated on every rank: it needs every row of V_qe and is tiny) ---------------------
    c_cnt = torch.empty(N, dtype=torch.int32, device=dev)
    if q_total is None:
        call("reid_transpose_count", ptr(q_idx), q_idx.numel(), ptr(q_ptr[q_ptr.numel() - 1:]), N, ptr(c_cnt), sp)
    else:
        call("reid_transpose_count", ptr(q_idx), q_total, None, N, ptr(c_cnt), sp)
    c_ptr, c_stats = _scan_async(c_cnt, N, dev, stats=report[R_C:R_C + 3])
    if speculative:
        c_cap, c_max = q_idx.numel(), 0                       # nnz(V_qe) <= its storage; longest column unknown
    else:
        q_total, c_max, c_sq = (int(v) for v in c_stats.tolist())   # read-back 2 of 2; total of the counts == nnz(V_qe)
        c_cap = max(q_total, 1)
        st.q_total, st.c_max, st.t_total_all = q_total, c_max, c_sq   # sum_c |col(c)|^2 = sum_i T_i over ALL rows
    c_idx = torch.empty(c_cap, dtype=torch.int32, device=dev)
    c_val = torch.empty(c_cap, dtype=torch.float32, device=dev)
    call("reid_transpose_fill", ptr(q_ptr), ptr(q_idx), ptr(q_val), N, N, ptr(c_ptr), ptr(c_cnt), ptr(c_idx),
         ptr(c_val), int(c_max), sp)
    st.C_ptr, st.C_idx, st.C_val = c_ptr, c_idx, c_val
    mark("transpose")
    if speculative:
        st.report = report

        st._check_norms = (pending is not None or info.get("max_sqnorm") is not None) and metric == "auto" \
            and info.get("metric", "ip") == "ip"

        def redo(vals):
            # a guess did not hold (or rows were uncertified): exact sizes, read back where they are needed
            if comm is not None or external_knn:              # the search ran elsewhere (sharded.py): the caller redoes the
                return None                                   # whole pass, search included, with sizes read back
            if vals == "l2":                                  # rows of different norms: search again with the L2 key
                return rerank_state_async(x, k1, k2, knn="exact", timers=timers, speculative=False, metric="l2", half=half)
            if vals[R_UNCERT] and pending is not None:
                pending["repair"]()
                info["visit_order"] = None
            info["uncertified_rows"] = int(vals[R_UNCERT])
            info["speculation_failed"] = dict(uncertified=int(vals[R_UNCERT]), qe_overflow_rows=int(vals[R_QE_OVF]))
            return rerank_state_async(x, k1, k2, knn=knn, timers=timers, knn_result=(rank_local, key_local, info),
                                      speculative=False, half=half)

        st._redo = redo
    if timers:
        torch.cuda.synchronize()
        for (_, a), (nm, b) in zip(ev[:-1], ev[1:]):
            st.timings[nm] = a.elapsed_time(b) * 1e-3
    return st


def rerank_state(x, k1, k2, **kw):
    """a1-a6 on device, finished: `rerank_state_async(...).finish()` (the pass itself does not synchronise; finish()
    reads its report once and redoes the pass with exact sizes in the rare case a guessed size did not hold)."""
    return rerank_state_async(x, k1, k2, **kw).finish()


def _stride_for(kind, N):
    """Record stride of a row-sharded exchange: the default, or 1.25 x the longest row the last pass saw."""
    hint = _rec_stride_hint.get((kind, N), 0)
    return max(REC_STRIDE[kind], -(-int(hint * 1.25) // 32) * 32)


def _one_norm_info(info, x):
    from .knn_tc import one_norm, sqnorm_range_of
    rng = info.get("max_sqnorm")
    return True if rng is None else one_norm(sqnorm_range_of(x, rng))


def rank_digest(st):
    """sha256 of the (N, k1) int32 neighbour lists -- what bench.py prints as config.rank_sha256."""
    import hashlib
    return hashlib.sha256(np.ascontiguousarray(st.rank.cpu().numpy().astype(np.int32)).tobytes()).hexdigest()


def query_expand_rows(st, row_begin, row_end):
    """a5 for rows [row_begin, row_end) against the state's GLOBAL V (what a rank of the row-sharded plan computes
    after the all-gather of the V rows).  Returns (q_cnt int32, q_idx int32, q_val fp32) compact in row order."""
    L = _lib.lib()
    dev = st.rank.device
    n = row_end - row_begin
    sp = stream_ptr()
    e_max = int((st.E_ptr[1:] - st.E_ptr[:-1]).max().item())
    q_stride = L.reid_query_expand_stride(st.k2, max(e_max, 1))
    q_cnt = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
    qp_idx = torch.empty(max(n, 1) * q_stride, dtype=torch.int32, device=dev)
    qp_val = torch.empty(max(n, 1) * q_stride, dtype=torch.float32, device=dev)
    call("reid_query_expand", ptr(st.rank), st.N, st.k1, st.k2, ptr(st.E_ptr), ptr(st.E_idx), ptr(st.V_val), max(e_max, 1),
         row_begin, row_end, ptr(q_cnt), ptr(qp_idx), ptr(qp_val), None, 1 if st.half else 0, sp)
    q_ptr, q_total, _ = _scan(q_cnt, n, dev)
    q_idx = torch.empty(max(q_total, 1), dtype=torch.int32, device=dev)
    q_val = torch.empty(max(q_total, 1), dtype=torch.float32, device=dev)
    call("reid_csr_compact", ptr(qp_idx), ptr(qp_val), q_stride, ptr(q_cnt), ptr(q_ptr), n, ptr(q_idx), ptr(q_val), sp)
    return q_cnt[:n], q_idx, q_val


def jaccard_neighbors(st, eps, with_values=False, speculative=None, owned=False):
    """a7 (sparse form): eps-neighbourhoods of the shard's rows.  Returns (slot_ptr int64 (n+1),
    nbr_idx int32, nbr_cnt int32 (n), nbr_val or None): row r's list is nbr_idx[slot_ptr[r] : +nbr_cnt[r]].

    Exact-size flavour: slots from T_i = sum_c |col(c)| (an upper bound of the partner count), total read back.
    Speculative flavour (default while the state's report is pending, i.e. inside a sync-free pass): slots from the
    Markov bound S_i (reid_jaccard_bounds), storage guessed, every kernel guarded; rows that did not fit are counted
    in the report (finish(check_nbr=True) tells).
    owned: every unordered pair {i, j} is accumulated and listed by ONE of its rows only (csrc/jaccard.cu pair_owned;
    J is bit-symmetric) -- half the table updates; dbscan_from_neighbors(owned=True) consumes such lists."""
    L = _lib.lib()
    dev = st.Q_ptr.device
    r0, r1 = st.row_begin, st.row_end
    n = r1 - r0
    sp = stream_ptr()
    if speculative is None:
        speculative = st.report is not None
    eps32 = float(np.float32(eps))
    t_cnt = torch.empty(n, dtype=torch.int32, device=dev)
    p_cnt = torch.empty(n, dtype=torch.int32, device=dev)       # partner-count guess: picks each row's first table class
    ws = torch.empty(L.reid_jaccard_eps_graph_workspace_bytes(st.N, n), dtype=torch.uint8, device=dev)
    if speculative:
        report = st.report
        s_cnt = torch.empty(n, dtype=torch.int32, device=dev)
        call("reid_jaccard_bounds", ptr(st.Q_ptr), ptr(st.Q_idx), ptr(st.Q_val), ptr(st.C_ptr), r0, r1, eps32, ptr(t_cnt),
             ptr(s_cnt), ptr(p_cnt), sp)
        slot_ptr, _ = _scan_async(s_cnt, n, dev, stats=report[R_S:R_S + 3])
        cap = max(n * NBR_SPEC_PER_ROW, int(_nbr_cap_hint.get(st.N, 0) * 1.25), 1)
        nbr_idx = torch.empty(cap, dtype=torch.int32, device=dev)
        nbr_val = torch.empty(cap, dtype=torch.float32, device=dev) if with_values else None
        nbr_cnt = torch.empty(n, dtype=torch.int32, device=dev)
        call("reid_jaccard_eps_graph", ptr(st.Q_ptr), ptr(st.Q_idx), ptr(st.Q_val), ptr(st.C_ptr), ptr(st.C_idx),
             ptr(st.C_val), st.N, r0, r1, eps32, ptr(t_cnt), ptr(p_cnt) if partner_guess_on(st.N) else None, ptr(slot_ptr),
             ptr(nbr_idx), ptr(nbr_val), ptr(nbr_cnt), cap, ptr(report[R_NBR_OVF:]), 1 if st.half else 0, 1 if owned else 0,
             ptr(report[R_ESC:]) if report.numel() > R_ESC else None, ptr(ws), sp)
        return slot_ptr, nbr_idx, nbr_cnt, nbr_val
    call("reid_jaccard_bounds", ptr(st.Q_ptr), ptr(st.Q_idx), None, ptr(st.C_ptr), r0, r1, eps32, ptr(t_cnt), None, ptr(p_cnt), sp)
    if r0 == 0 and r1 == st.N and getattr(st, "t_total_all", None) is not None:
        slot_ptr, _ = _scan_async(t_cnt, n, dev)              # the total is already known (rerank_state, a6)
        t_total = st.t_total_all
    else:
        slot_ptr, t_total, _ = _scan(t_cnt, n, dev)
    nbr_idx = torch.empty(max(t_total, 1), dtype=torch.int32, device=dev)
    nbr_val = torch.empty(max(t_total, 1), dtype=torch.float32, device=dev) if with_values else None
    nbr_cnt = torch.empty(n, dtype=torch.int32, device=dev)
    call("reid_jaccard_eps_graph", ptr(st.Q_ptr), ptr(st.Q_idx), ptr(st.Q_val), ptr(st.C_ptr), ptr(st.C_idx),
                                   ptr(st.C_val), st.N, r0, r1, eps32, ptr(t_cnt), ptr(p_cnt) if partner_guess_on(st.N) else None,
                                   ptr(slot_ptr), ptr(nbr_idx), ptr(nbr_val), ptr(nbr_cnt), 0, None, 1 if st.half else 0,
                                   1 if owned else 0, None, ptr(ws), sp)
    return slot_ptr, nbr_idx, nbr_cnt, nbr_val


def jaccard_dense_rows(st, out, row_begin, row_end):
    """a7 (dense form): rows [row_begin,row_end) of the reference's return value into `out` (device, (rows, N))."""
    L = _lib.lib()
    call("reid_jaccard_dense", ptr(st.Q_ptr), ptr(st.Q_idx), ptr(st.Q_val), ptr(st.C_ptr), ptr(st.C_idx),
                               ptr(st.C_val), st.N, row_begin, row_end, ptr(out), out.stride(0),
                               1 if getattr(st, "half", False) else 0, stream_ptr())


class JaccardDistance:
    """Lazy view of the float32 (N, N) Jaccard distance matrix (faiss_rerank.py:123)."""

    __array_priority__ = 100

    def __init__(self, state):
        self._state = state
        self._dense = None
        self.shape = (state.N, state.N)
        # use_float16=True returns a float16 matrix (faiss_rerank.py:36,101); the device rows hold fp16-representable fp32
        self.dtype = np.dtype(np.float16 if getattr(state, "half", False) else np.float32)
        self.ndim = 2

    # -- device-side consumers -------------------------------------------------
    @property
    def state(self):
        return self._state

    def dense_device(self, row_begin=0, row_end=None):
        """Rows of the matrix as a CUDA tensor (no host copy)."""
        st = self._state
        row_end = st.N if row_end is None else row_end
        out = torch.empty((row_end - row_begin, st.N), dtype=torch.float32, device=st.Q_ptr.device)
        jaccard_dense_rows(st, out, row_begin, row_end)
        return out

    # -- host-side (reference) view ---------------------------------------------
    def numpy(self):
        if self._dense is None:
            st = self._state
            N = st.N
            host = np.empty((N, N), dtype=self.dtype)
            block = max(1, min(N, (256 << 20) // (4 * N)))
            for a in range(0, N, block):
                b = min(N, a + block)
                host[a:b] = self.dense_device(a, b).cpu().numpy()      # exact: the values are float16 numbers already
            self._dense = host
        return self._dense

    def __array__(self, dtype=None, copy=None):
        a = self.numpy()
        if dtype is not None and np.dtype(dtype) != a.dtype:
            return a.astype(dtype)
        return a.copy() if copy else a

    def __len__(self):
        return self.shape[0]

    def __getitem__(self, item):
        return self.numpy()[item]

    def __setitem__(self, item, value):
        self.numpy()[item] = value

    def __getattr__(self, name):                              # min(), max(), mean(), T, astype, ...
        if name.startswith("_"):
            raise AttributeError(name)
        return getattr(self.numpy(), name)

    def _binop(name):
        def f(self, other):
            return getattr(self.numpy(), name)(np.asarray(other) if isinstance(other, JaccardDistance) else other)
        return f

    for _n in ("__add__", "__radd__", "__sub__", "__rsub__", "__mul__", "__rmul__", "__truediv__", "__lt__",
               "__le__", "__gt__", "__ge__", "__eq__", "__ne__"):
        locals()[_n] = _binop(_n)
    del _n, _binop

    def __repr__(self):
        return "JaccardDistance(N=%d, materialised=%s)" % (self.shape[0], self._dense is not None)

    __hash__ = None


def compute_jaccard_distance(target_features, k1=20, k2=6, print_flag=True, search_option=0, use_float16=False,
                             knn="auto"):
    """Drop-in for faiss_rerank.py:30.  `target_features`: (N, D) float32 tensor (CPU or CUDA) or ndarray,
    rows L2-normalised as the reference's backbone emits them (models/resnet.py:90-94)."""
    end = time.time()
    if print_flag:
        print('Computing jaccard distance...')
    if search_option not in (0, 1, 2, 3):
        raise ValueError("search_option must be 0..3 (faiss_rerank.py:39-62), got %r" % (search_option,))
    if isinstance(target_features, np.ndarray):
        target_features = torch.from_numpy(target_features)
    if target_features.dim() != 2:
        raise ValueError("target_features must be (N, D)")
    dev = _device_of(target_features)
    with torch.cuda.device(dev), torch.no_grad():
        from .knn_tc import sym_eligible
        N, D = target_features.shape
        if (not target_features.is_cuda and target_features.dtype == torch.float32 and target_features.is_contiguous()
                and knn in ("auto", "tc") and sym_eligible(N, D, k1) and 1 <= k2 <= k1 <= N):
            st = rerank_state(target_features, k1, k2, knn=knn, knn_result="upload", half=bool(use_float16))   # search overlaps the upload
        else:
            x = target_features.to(device=dev, dtype=torch.float32, non_blocking=True).contiguous()
            st = rerank_state(x, k1, k2, knn=knn, half=bool(use_float16))   # finish(): the one host synchronisation of the call
        out = JaccardDistance(st)
    if print_flag:
        print("Jaccard distance computing time cost: {}".format(time.time() - end))
    return out
