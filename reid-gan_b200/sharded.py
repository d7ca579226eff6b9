"""Row-partitioned pseudo-label pass: one process per GPU, torch.distributed (NCCL over NVLink /
NVSwitch) for the exchange steps.  The reference has no multi-GPU hot path (its only sharding is
faiss.IndexShards for search_option=2, utils/faiss_utils.py:92-106); the path is row-separable
(SURVEY.md section 8e), so rank r owns the contiguous rows [N*r/W, N*(r+1)/W) of every per-row stage:

    features   : all-gather of the fp32 rows (skipped when every rank already holds all N rows)
    a1  kNN    : own query rows against all N columns            -> all-gather neighbour lists (N x k1 int32)
    a2-a4      : own rows (R_half masks for all rows are recomputed locally: cheaper than a gather)
                                                                 -> all-gather V rows (CSR)
    a5  V_qe   : own rows                                        -> all-gather V_qe rows (CSR)
    a6  index  : replicated (tiny)
    a7  graph  : own rows of the eps-graph                       -> all-gather neighbour lists
    a8  labels : replicated union-find on the global graph (N x ~30 edges)

Outputs are byte-identical for every world size: each row's arithmetic is independent of the
partition and all accumulation orders are fixed.
The helpers only use torch.distributed collectives on whatever device the tensors live on, so the
host logic is testable on CPU with the gloo backend (tests/test_sharded_cpu.py).
"""
import torch
import torch.distributed as dist


TRACE_STEPS = False           # developer switch (scripts set the attribute): per-step CUDA-event times in knn_info["steps_ms"]
RECORD_GATHER = True          # one-collective ragged gathers
ROWS_PLAN_MIN_N = 65536     # from this N on the sparse stages are row-sharded too (see pseudo_labels)


_bounds_cache = {}


def partition(N, world, rank):
    """Contiguous row block of `rank`: [N*rank//world, N*(rank+1)//world)."""
    return (N * rank) // world, (N * (rank + 1)) // world


class RowComm:
    """All-gathers of row-sharded arrays (fixed-width rows and CSR pieces) over a process group."""

    def __init__(self, N, group=None):
        self.group = group
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        self.N = N
        self.bounds = [partition(N, self.world, r) for r in range(self.world)]
        self.r0, self.r1 = self.bounds[self.rank]
        self.max_rows = max(b - a for a, b in self.bounds)
        self._into_tensor = dist.get_backend(group) == "nccl"

    def _all_gather_padded(self, t, length, max_len):
        """t: (>=length, ...) local; returns a (world, max_len, ...) tensor after a padded all-gather."""
        shape = (max_len,) + tuple(t.shape[1:])
        if t.shape[0] == max_len and t.is_contiguous():
            send = t
        else:
            send = torch.empty(shape, dtype=t.dtype, device=t.device)
            if length:
                send[:length] = t[:length]
            if length < max_len:
                send[length:].zero_()
        out = torch.empty((self.world,) + shape, dtype=t.dtype, device=t.device)
        if self._into_tensor:
            dist.all_gather_into_tensor(out, send, group=self.group)
        else:
            dist.all_gather(list(out.unbind(0)), send, group=self.group)
        return out

    def gather_rows(self, t):
        """(n_local, ...) -> (N, ...): fixed-width rows in rank order."""
        n = self.r1 - self.r0
        out = self._all_gather_padded(t, n, self.max_rows)
        if self.N == self.max_rows * self.world:            # even split: the gathered buffer IS the result
            return out.reshape((self.N,) + tuple(t.shape[1:]))
        return torch.cat([out[r, : b - a] for r, (a, b) in enumerate(self.bounds)], dim=0)

    def gather_lengths(self, length, dev):
        """One int64 per rank (tensor all-gather + a single host read-back)."""
        mine = torch.tensor([int(length)], dtype=torch.int64, device=dev)
        out = self._all_gather_padded(mine, 1, 1)
        return [int(v) for v in out.flatten().tolist()]

    def gather_concat(self, t, length, lens=None):
        """1-D local array with `length` valid entries -> concatenation over ranks, and the lengths."""
        if lens is None:
            lens = self.gather_lengths(length, t.device)
        out = self._all_gather_padded(t, length, max(max(lens), 1))
        return torch.cat([out[r, :l] for r, l in enumerate(lens)], dim=0), lens

    def gather_records(self, cnt, row_ptr, idx, val, stride, overflow=None, stats_out=None, tag="rec"):
        """CUDA only: ragged rows (cnt, row starts `row_ptr` into idx / val) -> global CSR through ONE all-gather of
        fixed-stride records (csrc/rerank_sparse.cu rows_pack / rows_unpack).  Returns (g_ptr, g_idx, g_val, total,
        max, g_cnt), or None when some row is longer than `stride` (every rank sees the same gathered counts, so
        all ranks take the fallback together)."""
        from ._lib import call, ptr as p_, stream_ptr
        from .faiss_rerank import _scan_async
        dev = idx.device
        n = self.r1 - self.r0
        words = 1 + stride * (2 if val is not None else 1)
        pb = None
        if overflow is not None:                             # sync-free pass: peer stores instead of pack + NCCL all-gather
            # one buffer per exchange (tag): two exchanges of one pass must never share a receive buffer -- a fast rank
            # could push the second while a slow one still unpacks the first
            pb = _peer_buffer("rec:" + tag, self.world * self.max_rows * words * 4, dev, self.group)
        if pb is not None:
            call("reid_peer_push_records", p_(cnt), p_(row_ptr), p_(idx), p_(val), n, self.max_rows, stride, self.rank,
                 self.world, p_(pb.peer_base), 0, stream_ptr())
            pb.barrier()
            out = pb.buf.view(torch.int32)[: self.world * self.max_rows * words]
        else:
            rec = torch.empty((self.max_rows, words), dtype=torch.int32, device=dev)
            call("reid_rows_pack", p_(cnt), p_(row_ptr), p_(idx), p_(val), n, self.max_rows, stride, p_(rec), stream_ptr())
            out = torch.empty((self.world, self.max_rows, words), dtype=torch.int32, device=dev)
            dist.all_gather_into_tensor(out, rec, group=self.group)
        key_ = (self.N, self.world, str(dev))
        if key_ not in _bounds_cache:                         # cached across passes: no H2D copy inside a captured pass
            _bounds_cache[key_] = torch.tensor([a for a, _ in self.bounds] + [self.N], dtype=torch.int64, device=dev)
        self._bounds_dev = _bounds_cache[key_]
        g_cnt = torch.empty(self.N, dtype=torch.int32, device=dev)
        if overflow is not None:
            # sync-free flavour: upper-bound storage, rows that did not fit are counted in `overflow` (device scalar)
            call("reid_rows_unpack_counts", p_(out), stride, 1 if val is not None else 0, self.world, self.max_rows,
                 p_(self._bounds_dev), self.N, p_(g_cnt), p_(overflow), stream_ptr())
            g_ptr, stats = _scan_async(g_cnt, self.N, dev, stats=stats_out)
            g_idx = torch.empty(self.N * stride, dtype=torch.int32, device=dev)
            g_val = torch.empty(self.N * stride, dtype=torch.float32, device=dev) if val is not None else None
            call("reid_rows_unpack_fill", p_(out), stride, self.world, self.max_rows, p_(self._bounds_dev), self.N, p_(g_ptr),
                 p_(g_idx), p_(g_val), stream_ptr())
            return g_ptr, g_idx, g_val, None, None, g_cnt
        call("reid_rows_unpack_counts", p_(out), stride, 1 if val is not None else 0, self.world, self.max_rows,
             p_(self._bounds_dev), self.N, p_(g_cnt), None, stream_ptr())
        g_ptr, stats = _scan_async(g_cnt, self.N, dev)
        total, mx, _ = (int(v) for v in stats.tolist())
        if mx > stride:
            return None
        g_idx = torch.empty(max(total, 1), dtype=torch.int32, device=dev)
        g_val = torch.empty(max(total, 1), dtype=torch.float32, device=dev) if val is not None else None
        call("reid_rows_unpack_fill", p_(out), stride, self.world, self.max_rows, p_(self._bounds_dev), self.N, p_(g_ptr),
             p_(g_idx), p_(g_val), stream_ptr())
        return g_ptr, g_idx, g_val, total, mx, g_cnt

    def gather_csr(self, cnt, idx, val, row_ptr=None, stride=128):
        """Local CSR pieces (row counts, column indices, values) -> global (ptr, idx, val, nnz, max_row_nnz)."""
        from .faiss_rerank import _scan
        if idx.is_cuda and row_ptr is not None and RECORD_GATHER:
            got = self.gather_records(cnt, row_ptr, idx, val, stride)
            if got is not None:
                return got[:5]
        g_cnt = self.gather_rows(cnt)
        if g_cnt.is_cuda:
            g_ptr, total, mx = _scan(g_cnt, self.N, g_cnt.device)
            edges = g_ptr[[a for a, _ in self.bounds] + [self.N]].tolist()      # per-rank nnz without a 2nd collective
        else:                                   # CPU (gloo) test path: same arithmetic in torch
            g_ptr = torch.zeros(self.N + 1, dtype=torch.int64)
            g_ptr[1:] = torch.cumsum(g_cnt.to(torch.int64), 0)
            total, mx = int(g_ptr[-1]), int(g_cnt.max()) if self.N else 0
            edges = [int(g_ptr[a]) for a, _ in self.bounds] + [total]
        lens = [edges[r + 1] - edges[r] for r in range(self.world)]
        g_idx, _ = self.gather_concat(idx, lens[self.rank], lens)
        g_val, _ = self.gather_concat(val, lens[self.rank], lens)
        if g_idx.numel() == 0:
            g_idx = torch.zeros(1, dtype=idx.dtype, device=idx.device)
            g_val = torch.zeros(1, dtype=val.dtype, device=val.device)
        return g_ptr, g_idx, g_val, total, mx

    def gather_neighbors(self, slot_ptr, nbr_idx, nbr_cnt, overflow=None, stride=128):
        """Per-row neighbour lists stored at slot_ptr (upper-bound slots) -> compact global lists:
        (ptr int64 (N+1), idx, cnt int32 (N)).  overflow (device scalar): sync-free flavour, see gather_records."""
        n = self.r1 - self.r0
        if overflow is not None:
            got = self.gather_records(nbr_cnt, slot_ptr, nbr_idx, None, stride, overflow=overflow, tag="nbr")
            return got[0], got[1], got[5]
        if nbr_idx.is_cuda and RECORD_GATHER:
            got = self.gather_records(nbr_cnt, slot_ptr, nbr_idx, None, 128)
            if got is not None:
                g_idx = got[1] if got[3] else torch.zeros(1, dtype=torch.int32, device=nbr_idx.device)
                return got[0], g_idx, got[5]
        g_cnt = self.gather_rows(nbr_cnt[:n])
        dev = nbr_idx.device
        if g_cnt.is_cuda:
            from .faiss_rerank import _scan
            from ._lib import call, ptr as p_, stream_ptr
            g_ptr, total_all, _ = _scan(g_cnt, self.N, dev)
            edges = g_ptr[[a for a, _ in self.bounds] + [self.N]].tolist()
            lens = [edges[r + 1] - edges[r] for r in range(self.world)]
            compact = torch.empty(max(lens[self.rank], 1), dtype=torch.int32, device=dev)
            loc_ptr = (g_ptr[self.r0:self.r1 + 1] - edges[self.rank]).contiguous()
            call("reid_lists_compact", p_(slot_ptr), p_(nbr_idx), p_(nbr_cnt), p_(loc_ptr), n, p_(compact), stream_ptr())
        else:
            cnt64 = nbr_cnt[:n].to(torch.int64)
            total = int(cnt64.sum())
            if total:
                row_of = torch.repeat_interleave(torch.arange(n), cnt64)
                first = torch.cumsum(cnt64, 0) - cnt64
                pos = slot_ptr[:n][row_of] + (torch.arange(total) - first[row_of])
                compact = nbr_idx[pos]
            else:
                compact = nbr_idx[:0]
            g_ptr = torch.zeros(self.N + 1, dtype=torch.int64)
            g_ptr[1:] = torch.cumsum(g_cnt.to(torch.int64), 0)
            edges = [int(g_ptr[a]) for a, _ in self.bounds] + [int(g_ptr[-1])]
            lens = [edges[r + 1] - edges[r] for r in range(self.world)]
        g_idx, _ = self.gather_concat(compact, lens[self.rank], lens)
        if g_idx.numel() == 0:
            g_idx = torch.zeros(1, dtype=nbr_idx.dtype, device=dev)
        return g_ptr, g_idx, g_cnt.contiguous()


def block_partition(N, world, rank):
    """Equal blocks of B = ceil(N / world) rows (the last ranks may hold fewer): row -> owner is row // B, which
    lets an all-to-all address per-rank partial lists without a lookup.  Used by the tile-sharded search."""
    B = -(-N // world)
    return min(N, rank * B), min(N, (rank + 1) * B), B


_my_tiles_cache = {}
_peer_cache = {}
PEER_EXCHANGE = True      # False: the NCCL all-to-all carries the exchange (tests flip it to compare the two)


class PeerLists:
    """Receive buffer of the tile-sharded search in symmetric (peer-mapped) memory: W * B * cap candidate entries
    + W * B counts on every rank, each rank holding the base addresses of all of them (torch.distributed.
    _symmetric_memory does the mapping; the stores are csrc/peer_exchange.cu).  One per (N, W, cap, device)."""

    def __init__(self, W, B, cap, dev, group):
        import torch.distributed._symmetric_memory as symm
        self.cnt_off = W * B * cap * 8
        nbytes = self.cnt_off + W * B * 4
        self.buf = symm.empty((nbytes + 7) // 8, dtype=torch.int64, device=dev)
        self.handle = symm.rendezvous(self.buf, group if group is not None else dist.group.WORLD)
        self.peer_base = torch.tensor([int(p) for p in self.handle.buffer_ptrs], dtype=torch.int64, device=dev)
        self.recv = self.buf[: W * B * cap].view(W * B, cap)
        self.recv_cnt = self.buf.view(torch.int32)[self.cnt_off // 4: self.cnt_off // 4 + W * B]

    def barrier(self):
        self.handle.barrier(channel=0)


class PeerBuffer:
    """nbytes of symmetric (peer-mapped) memory on every rank + the device array of all ranks' base addresses."""

    def __init__(self, nbytes, dev, group):
        import torch.distributed._symmetric_memory as symm
        self.buf = symm.empty((nbytes + 7) // 8, dtype=torch.int64, device=dev)
        self.handle = symm.rendezvous(self.buf, group if group is not None else dist.group.WORLD)
        self.peer_base = torch.tensor([int(p) for p in self.handle.buffer_ptrs], dtype=torch.int64, device=dev)

    def barrier(self):
        self.handle.barrier(channel=0)


def _peer_buffer(name, nbytes, dev, group):
    """Cached per (name, size): creating one is a collective (rendezvous) and must not happen inside a captured pass.
    None when the box cannot map peer memory (NCCL then carries the exchange)."""
    if not PEER_EXCHANGE:
        return None
    key_ = (name, nbytes, str(dev), id(group))
    if key_ not in _peer_cache:
        try:
            _peer_cache[key_] = PeerBuffer(nbytes, dev, group)
        except Exception as e:
            import warnings
            warnings.warn("peer-memory exchange unavailable (%r): using NCCL collectives" % (e,))
            _peer_cache[key_] = None
    return _peer_cache[key_]


def peer_all_gather(name, block, group=None):
    """all_gather_into_tensor over peer stores: `block` (contiguous, same shape on every rank) -> (W * len(block), ...)
    on every rank, in rank order.  Falls back to NCCL when peer memory is unavailable."""
    from ._lib import call, ptr, stream_ptr
    W, me = dist.get_world_size(group), dist.get_rank(group)
    nbytes = block.numel() * block.element_size()
    pb = _peer_buffer(name, W * nbytes, block.device, group) if nbytes % 4 == 0 else None
    shape = (W * block.shape[0],) + tuple(block.shape[1:])
    if pb is None:
        out = torch.empty(shape, dtype=block.dtype, device=block.device)
        dist.all_gather_into_tensor(out, block, group=group)
        return out
    call("reid_peer_allgather", ptr(block), nbytes, me, W, ptr(pb.peer_base), 0, stream_ptr())
    pb.barrier()
    return pb.buf.view(torch.uint8)[: W * nbytes].view(block.dtype).view(shape)


def _peer_lists(W, B, cap, dev, group):
    key_ = (W, B, cap, str(dev), id(group))
    if key_ not in _peer_cache:
        try:
            _peer_cache[key_] = PeerLists(W, B, cap, dev, group)
        except Exception as e:                              # no peer mapping on this box: NCCL carries the exchange
            import warnings
            warnings.warn("peer-memory exchange unavailable (%r): using the NCCL all-to-all" % (e,))
            _peer_cache[key_] = None
    return _peer_cache[key_]


def _my_tiles(N, W, me, dev):
    """Upper-triangle tiles dealt to this rank: tile (I, J) goes to rank (I + J) mod W -- balanced for the rows of
    block I (J varies) AND for the rows of block J (I varies), so every row's candidates split evenly over the W
    partial lists.  Cached (the selection is a boolean-mask gather, i.e. a host synchronisation)."""
    from . import knn_tc as kt
    key_ = (N, W, me, str(dev))
    if key_ not in _my_tiles_cache:
        tiles = kt._tile_order((N + 255) // 256, dev)
        _my_tiles_cache[key_] = tiles[((tiles[:, 0] + tiles[:, 1]) % W) == me].contiguous()
    return _my_tiles_cache[key_]


@torch.no_grad()
def knn_search_tiles(x, k, group=None, report=None):
    """a1 on W GPUs, symmetric form: every rank holds all N feature rows; the sampling prepass is split by rows
    (all-gather of the N thresholds), the upper-triangle tiles of the similarity are dealt round-robin to the
    ranks, each rank appends the survivors of ITS tiles to per-row partial lists, one all-to-all hands every
    row's W partial lists to the row's owner, the owner re-scores and certifies its rows, and the final lists
    are all-gathered.  Returns (rank (N, k) int32, key (N, k) fp32, info) -- identical on every rank and
    bit-identical to the single-GPU search (the exact key and the (key desc, index asc) order decide, not
    the candidate sets).

    report (the int64 pass report of faiss_rerank.py): sync-free flavour -- nothing is read back here; the number of
    uncertified rows is accumulated in report[R_UNCERT] and info["max_sqnorm"] carries the {max, min} squared norms,
    both checked by RerankState.finish(), which has the whole pass redone (with the repairs below) if needed."""
    from . import knn_tc as kt
    from ._lib import call, lib, ptr, stream_ptr
    from .faiss_rerank import R_UNCERT, _knn_exact_rows
    L = lib()
    W, me = dist.get_world_size(group), dist.get_rank(group)
    N, D = x.shape
    dev = x.device
    sp = stream_ptr()
    marks = []

    def mark(name):
        if TRACE_STEPS:
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            marks.append((name, e))

    mark("start")
    b0, b1, B = block_partition(N, W, me)
    nb = b1 - b0
    xh = torch.empty((N, D), dtype=torch.float16, device=dev)
    msq = torch.empty(2, dtype=torch.float32, device=dev)
    call("reid_features_to_half", ptr(x), N, D, kt.SCALE_LOG2, ptr(xh), ptr(msq), sp)
    # 1. thresholds of my rows from the sample; the float thresholds are all-gathered (the main pass compares the rows
    #    AND the columns of a tile), their order-preserving images stay with the owner (certificate)
    m = kt.sample_size(N, k)
    xs = torch.empty((m, D), dtype=torch.float16, device=dev)
    call("reid_features_sample", ptr(xh), N, D, m, kt._sample_stride(N, m), ptr(xs), sp)
    t_f = torch.empty(B, dtype=torch.float32, device=dev)
    t_o = torch.empty(B, dtype=torch.int32, device=dev)
    if nb:
        # A rank's block is a few 256-row units (16 at W = 8) for 74 CTA-pair slots: the prepass then runs at the
        # latency of ONE unit.  The sample columns of a unit are split over up to 4 CTA pairs (every (row, split,
        # epilogue group) keeps its own list; the threshold is the r-th best over all of a row's lists).
        splits = kt.prepass_splits(nb, m)
        pre = torch.empty(nb * 2 * splits * kt.TC_CAP, dtype=torch.int64, device=dev)
        pre_cnt = torch.zeros(nb * 2 * splits, dtype=torch.int32, device=dev)
        pre_tau = torch.empty(nb, dtype=torch.int32, device=dev)
        call("reid_knn_candidates_tc_ab", ptr(xh), N, ptr(xs), m, D, kt.SCALE_LOG2, b0, b1, -kt.sym_rank(k), splits, 2, ptr(pre),
             ptr(pre_cnt), ptr(pre_tau), sp)
        call("reid_knn_sample_tau", ptr(pre), ptr(pre_cnt), ptr(pre_tau), 2 * splits, nb, kt.sym_rank(k), ptr(t_f), ptr(t_o), sp)
    mark("prepass")
    if report is not None:
        tau = peer_all_gather("tau", t_f, group)                       # rows >= N are padding (never read)
    else:
        tau = torch.empty(W * B, dtype=torch.float32, device=dev)
        dist.all_gather_into_tensor(tau, t_f, group=group)
    mark("gather_tau")
    # 2. my share of the tiles -> partial lists of ALL rows (W * B row slots so that slot == row)
    tiles = _my_tiles(N, W, me, dev)
    cap = max(128, kt.SYM_CAP // W)
    part = torch.empty((W * B, cap), dtype=torch.int64, device=dev)
    part_cnt = torch.empty(W * B, dtype=torch.int32, device=dev)
    if tiles.shape[0]:
        kt.candidates_sym_launch(xh, N, D, tau, tiles, cap, part, part_cnt, 1, sp)
    else:
        part_cnt.zero_()
    mark("tiles")
    # 3. all-to-all: block w of `part` (rows owned by rank w) goes to rank w; I receive W partial lists per own row.
    #    Over NVLink peer memory when the box maps it: every rank STORES the valid entries of its lists straight into
    #    the owners' receive buffers (csrc/peer_exchange.cu), a barrier separates the stores from the readers.  The
    #    buffer is reused by the next pass: its readers (the re-score below) are done on every rank before anyone
    #    can reach the next push, because the all-gather of the final lists (step 5) needs every rank's re-score.
    peer = _peer_lists(W, B, cap, dev, group) if PEER_EXCHANGE else None
    if peer is not None:
        call("reid_peer_push_lists", ptr(part), ptr(part_cnt), W, B, cap, me, ptr(peer.peer_base), peer.cnt_off, sp)
        peer.barrier()
        recv, recv_cnt = peer.recv, peer.recv_cnt
    else:
        recv = torch.empty_like(part)
        recv_cnt = torch.empty_like(part_cnt)
        dist.all_to_all_single(recv, part, group=group)
        dist.all_to_all_single(recv_cnt, part_cnt, group=group)
    mark("all_to_all")
    # 4. exact re-score + certificate of my rows (list q of local row r at q * B + r)
    idx = torch.empty((B, k), dtype=torch.int32, device=dev)
    key = torch.empty((B, k), dtype=torch.float32, device=dev)
    n_bad = 0
    metric = "ip"
    max_err = torch.zeros(1, dtype=torch.float32, device=dev)
    if nb:
        flag = torch.empty(nb, dtype=torch.int32, device=dev)
        ws = torch.empty(L.reid_knn_rescore_workspace_bytes(N, nb), dtype=torch.uint8, device=dev)
        call("reid_knn_rescore", ptr(x), N, D, b0, b1, ptr(recv), ptr(recv_cnt), ptr(t_o), W, cap, B, k, 0.0, ptr(msq),
             1 if kt.ORDER_ROWS else 0, ptr(idx), ptr(key), ptr(flag), ptr(max_err), ptr(ws),
             ptr(report[R_UNCERT:]) if report is not None else None, sp)
        if report is None:
            bad = torch.nonzero(flag).flatten().to(torch.int32)
            n_bad = bad.numel()
            if not kt.one_norm(kt.sqnorm_range_of(x, msq)):  # rows of different norms (every rank sees the same features):
                metric = "l2"                              # the reference's L2 order needs the squared-L2 key
                _knn_exact_rows(x, k, None, b0, nb, idx[:nb], key[:nb], metric="l2")
                n_bad = 0
            elif n_bad:                                    # uncertified rows: exact CUDA-core search
                rows = (bad + b0).contiguous()
                bi = torch.empty((n_bad, k), dtype=torch.int32, device=dev)
                bk = torch.empty((n_bad, k), dtype=torch.float32, device=dev)
                _knn_exact_rows(x, k, rows, 0, n_bad, bi, bk)
                idx[bad.long()] = bi
                key[bad.long()] = bk
    elif report is None and not kt.one_norm(kt.sqnorm_range_of(x, msq)):
        metric = "l2"
    mark("rescore")
    # 5. final lists of all rows on every rank
    if report is not None:
        g_idx = peer_all_gather("rank", idx, group)
        g_key = peer_all_gather("rkey", key, group)
    else:
        g_idx = torch.empty((W * B, k), dtype=torch.int32, device=dev)
        g_key = torch.empty((W * B, k), dtype=torch.float32, device=dev)
        dist.all_gather_into_tensor(g_idx, idx, group=group)
        dist.all_gather_into_tensor(g_key, key, group=group)
    mark("gather_lists")
    steps = None
    if TRACE_STEPS:
        torch.cuda.synchronize()
        steps = {b[0]: round(a[1].elapsed_time(b[1]), 3) for a, b in zip(marks[:-1], marks[1:])}
    info = dict(mode="tc-sym-tiles" if metric == "ip" else "exact-l2", metric=metric, steps_ms=steps, world=W,
                sym=dict(sample=m, tiles=int(tiles.shape[0])), n_splits=0, keep=cap,
                uncertified_rows=int(n_bad), max_abs_err=max_err, xh=xh, cand_cnt=recv_cnt,
                max_sqnorm=msq if report is not None else None)
    return g_idx[:N], g_key[:N], info


@torch.no_grad()
def pseudo_labels(x, k1=30, k2=6, eps=0.6, min_samples=4, knn="auto", centroids=False, group=None, N=None,
                  timers=False, plan="auto", speculative=True, graph=False):
    """Row-sharded pass.  `x`: either all N rows (every rank holds a replica) or this rank's row block
    (then N must be given and the blocks are all-gathered first).  Returns the same dict as
    pipeline.pseudo_labels with GLOBAL labels on every rank."""
    from ._lib import call, ptr, stream_ptr
    from .dbscan import dbscan_from_neighbors
    from .faiss_rerank import jaccard_neighbors, rerank_state_async
    if not x.is_cuda:
        raise RuntimeError("sharded.pseudo_labels needs CUDA tensors; there is no CPU fallback")
    with torch.cuda.device(x.device):
        if N is None or x.shape[0] == N:
            N = x.shape[0]
            comm = RowComm(N, group)
        else:
            comm = RowComm(N, group)
            if x.shape[0] != comm.r1 - comm.r0:
                raise ValueError("rank %d holds %d rows, expected %d" % (comm.rank, x.shape[0], comm.r1 - comm.r0))
            x = comm.gather_rows(x.contiguous())                    # collective (1): features
        # kNN: tile-sharded symmetric search when the shape allows it, else own rows x all columns.
        # Sparse stages a2-a8: plan "tiles" REPLICATES them on every rank (they total ~1.5 ms at N = 32,621 and on two
        # GPUs their exchange steps cost more than sharding saves); plan "tiles+rows" / "rows" shards every per-row
        # stage with the all-gathers listed in the module docstring (default from 4 GPUs or ROWS_PLAN_MIN_N rows on).
        from . import knn_tc as kt
        sym_ok = (knn in ("auto", "tc") and kt.SYM and N >= kt.SYM_MIN_N and k1 <= kt.SYM_MAX_K and x.shape[1] % 64 == 0)
        if plan == "auto":
            # measured at N = 32,621 with the peer-store exchanges and graph replay (profiles/): 2 GPUs 2.81 ms (tiles)
            # vs 2.57 ms (tiles+rows), 8 GPUs 2.16 vs 1.78 ms: the per-row stages are sharded from 2 GPUs on
            plan = "tiles+rows" if sym_ok else "rows"
        if plan in ("tiles", "tiles+rows") and not sym_ok:
            raise ValueError("plan %r needs the symmetric tensor-core search (N >= %d, k1 <= %d, D %% 64 == 0)" % (plan, kt.SYM_MIN_N, kt.SYM_MAX_K))
        from .faiss_rerank import REPORT_WORDS, R_XCHG_OVF, _stride_for, _rec_stride_hint, partner_guess_on
        from .pipeline import _labels_from_state
        x = x.contiguous()
        dev = x.device

        def run(spec):
            """One pass.  spec: the sync-free flavour (no host read-back between the stages: upper-bound / guessed sizes,
            fixed-stride exchange records, every kernel reports what did not fit); else sizes are read back where needed."""
            report = torch.zeros(REPORT_WORDS, dtype=torch.int64, device=dev) if spec else None
            res = None
            if plan in ("tiles", "tiles+rows"):
                res = knn_search_tiles(x, k1, group, report=report)
            if plan == "tiles":
                # every rank runs the (replicated) sparse stages like pipeline.pseudo_labels
                st = rerank_state_async(x, k1, k2, knn_result=res, timers=timers, report=report, speculative=spec)
                labels, core, ncl, nbr_cnt = _labels_from_state(st, eps, min_samples, timers)
            else:
                st = rerank_state_async(x, k1, k2, knn=knn, comm=comm, timers=timers, knn_result=res, report=report,
                                        speculative=spec and res is not None)
                slot_ptr, nbr_idx, nbr_cnt, _ = jaccard_neighbors(st, eps, owned=True)
                if st.report is not None:
                    g_ptr, g_idx, g_cnt = comm.gather_neighbors(slot_ptr, nbr_idx, nbr_cnt, overflow=st.report[R_XCHG_OVF:],
                                                                stride=_stride_for("nbr", N))
                else:
                    g_ptr, g_idx, g_cnt = comm.gather_neighbors(slot_ptr, nbr_idx, nbr_cnt)
                    _rec_stride_hint[("nbr", N)] = max(_rec_stride_hint.get(("nbr", N), 0), int(g_cnt.max().item()) if N else 0)
                labels, core, ncl = dbscan_from_neighbors(N, g_ptr, g_idx, g_cnt, min_samples, owned=True)
            cen = None
            if centroids:
                cen = torch.empty((max(N, 1), x.shape[1]), dtype=torch.float32, device=dev)
                from ._lib import lib as _L
                cws = torch.empty(max(1, _L().reid_centroids_workspace_bytes(N, max(N, 1))), dtype=torch.uint8, device=dev)
                call("reid_centroids_dev", ptr(x), N, x.shape[1], ptr(labels), ptr(ncl), max(N, 1), 1, ptr(cen), ptr(cws), stream_ptr())
            return st, labels, core, ncl, nbr_cnt, cen

        if graph and speculative and not timers:
            # the whole pass, collectives included, replayed from one CUDA graph (pipeline.PassGraph)
            from .pipeline import PassGraph, _graph_key
            g = PassGraph.get(_graph_key(x, k1, k2, float(eps), min_samples, knn, bool(centroids), plan, comm.world, N,
                                         partner_guess_on(N)),
                              lambda: run(True) + (None,))
            if getattr(g, "report", None) is None:
                g.report = g.result[0].report
            g.graph.replay()
            st, labels, core, ncl, nbr_cnt, cen = g.result[:6]
            st.report = g.report
        else:
            st, labels, core, ncl, nbr_cnt, cen = run(speculative)
        st2, nbr_ok = st.finish(check_nbr=True)
        if st2 is None or st2 is not st or not nbr_ok:               # a guess did not hold / rows uncertified / other norms
            info = st.knn_info
            st, labels, core, ncl, nbr_cnt, cen = run(False)
            st.finish()
            st.knn_info["speculation_failed"] = dict(report=getattr(st2 or st, "report_vals", None), first=info.get("mode"))
        out = dict(labels=labels, core=core, num_clusters=ncl, state=st, nbr_cnt=nbr_cnt)
        if centroids:
            out["centroids"] = cen[: int(ncl.item())]
        return out


@torch.no_grad()
def pseudo_labels_host(x_host, k1=30, k2=6, eps=0.6, min_samples=4, knn="auto", group=None):
    """End-to-end variant: `x_host` = all N rows in (pinned) host memory on every rank; each rank uploads
    only ITS row block, the blocks are all-gathered over NVLink, labels come back to the host."""
    N = x_host.shape[0]
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    r0, r1 = partition(N, world, rank)
    dev = torch.device("cuda", torch.cuda.current_device())
    x_local = x_host[r0:r1].to(dev, non_blocking=True)
    out = pseudo_labels(x_local, k1, k2, eps, min_samples, knn=knn, group=group, N=N)
    return out["labels"].cpu().numpy()
