"""DistributedEvaluator: Evaluator.evaluate with one process per GPU.

The reference evaluates under nn.DataParallel (evaluators.py:127-142, test.py:84): the backbone runs on all GPUs.  Here
each rank extracts its share of the test images (eval_shard: the union of query and gallery, sorted by file name, in
contiguous blocks), and reid_peer_scatter_rows stores every extracted row, as NVLink peer stores, straight into its
query and gallery positions of the (M, D) matrix x = [query; gallery] of EVERY rank (M = Q + G).  Then:

    distances and metrics : rank r scores the query rows partition(Q, W, r) against all G gallery rows; the per-query
                            AP, has-positive flag and CMC contributions are all-gathered, and every rank reduces them
                            in query order (mAP: mean_ap's host arithmetic; CMC: reid_cmc_reduce)
    rerank=True           : colmax (farthest-row search) and the neighbour lists initial_rank[:, :k1+1] are split by
                            the rows partition(M, W, r) and all-gathered; the sparse stages are replicated (a query's
                            Jaccard row reads the inverted index of all M rows); the Jaccard rows and the blend run
                            for the rank's query rows only, against its own (Q_r, G) distance block

Every per-row value is computed with the arithmetic of the single-process path and every sum runs in its order, so
each rank returns the same mAP and CMC as Evaluator.evaluate, byte for byte, for every world size -- given the same
extracted rows.  The backbone itself is outside that promise: its kernels may depend on the batch size (the GEMM of an
nn.Linear gives other bits for some rows in a 50-row batch than in a 64-row one on a B200), and a rank's share is cut
into other batches than one loader over all images, so such a model can change the last bits of some rows before
evaluation starts.  Without a peer
mapping (sharded.PEER_EXCHANGE = False, or a box that cannot map peer memory) the collectives carry the exchanges.

single_gallery_shot (a host twin of np.random over the full distance matrix) is not offered: no rank ever holds
the full matrix, and evaluate_all never asks for it.
"""
import numpy as np
import torch
import torch.distributed as dist

from . import sharded
from ._lib import call, ptr, stream_ptr
from .evaluators import Evaluator, _print_cmc, eval_shard, extract_features
from .sharded import partition

TRACE_STEPS = False      # developer switch (scripts set the attribute): per-stage CUDA-event times in evaluator.steps_ms
CMC_TOPK = 100           # evaluation.cmc's default topk, the one evaluate_all uses


def _positions(query, gallery):
    """file name -> row of x = [query; gallery], once per list."""
    qpos = {f: i for i, (f, _, _) in enumerate(query)}
    gpos = {f: len(query) + j for j, (f, _, _) in enumerate(gallery)}
    if len(qpos) != len(query) or len(gpos) != len(gallery):
        raise ValueError("DistributedEvaluator: a file name occurs twice in the query or in the gallery list")
    return qpos, gpos


def dst_table(names, qpos, gpos, dev):
    """(n, 2) int32 destinations of the extracted rows `names` for reid_peer_scatter_rows (-1: not in that list)."""
    rows = [[qpos.get(f, -1), gpos.get(f, -1)] for f in names]
    return torch.tensor(rows, dtype=torch.int32).reshape(len(rows), 2).to(dev)


def scatter_features(src, n, table, M, group=None):
    """x = [query; gallery] (M, D) on every rank from each rank's n extracted rows src[:n] and their destinations."""
    D = src.shape[1]
    dev = src.device
    W = dist.get_world_size(group)
    sp = stream_ptr()
    pb = sharded._peer_buffer("eval_x:%dx%d" % (M, D), M * D * 4, dev, group)
    if pb is not None:
        call("reid_peer_scatter_rows", ptr(src), n, D, ptr(table), M, W, ptr(pb.peer_base), 0, None, sp)
        pb.barrier()
        return pb.buf.view(torch.float32)[: M * D].view(M, D)
    # collective fallback: one all-gather of [table | rows] blocks (an even row count keeps the rows 16-byte aligned),
    # then the same kernel once per source rank into the local matrix
    B = -(-M // W)
    B += B & 1
    blk = torch.full((2 * B + B * D,), -1, dtype=torch.int32, device=dev)
    blk[: 2 * n] = table.flatten()
    blk[2 * B: 2 * B + n * D] = src[:n].reshape(-1).view(torch.int32)
    out = torch.empty(W * blk.numel(), dtype=torch.int32, device=dev)
    dist.all_gather_into_tensor(out, blk, group=group)
    x = torch.empty((M, D), dtype=torch.float32, device=dev)
    base = torch.full((1,), x.data_ptr(), dtype=torch.int64, device=dev)
    for w in range(W):
        o = w * blk.numel()
        call("reid_peer_scatter_rows", ptr(out[o + 2 * B:]), B, D, ptr(out[o:]), M, 1, ptr(base), 0, None, sp)
    return x


def device_ids(query, gallery, dev):
    """(q_ids, g_ids, q_cams, g_cams) int64 CUDA tensors."""
    def col(items, k):
        return torch.tensor([it[k] for it in items], dtype=torch.int64).to(dev)
    return col(query, 1), col(gallery, 1), col(query, 2), col(gallery, 2)


def block_metrics(d, q0, ids, topk, rows):
    """reid_rank_metrics on the distance rows of queries [q0, q0 + len(d)) against the whole gallery -> one float64
    (rows, 2 + topk) block: AP, has-positive flag, CMC contributions (market1501: no separate camera set, first match
    break), zero-padded to `rows` rows for a fixed-size all-gather."""
    qi, gi, qc, gc = ids
    dev = qi.device
    out = torch.zeros((rows, 2 + topk), dtype=torch.float64, device=dev)
    if d is None or d.shape[0] == 0:
        return out
    m, n = d.shape
    ap = torch.empty(m, dtype=torch.float64, device=dev)
    has = torch.empty(m, dtype=torch.int32, device=dev)
    contrib = ret = None
    if topk:
        contrib = torch.empty((m, topk), dtype=torch.float64, device=dev)
        ret = torch.empty(topk, dtype=torch.float64, device=dev)
    q1 = q0 + m
    call("reid_rank_metrics", ptr(d), m, n, n, ptr(qi[q0:q1]), ptr(gi), ptr(qc[q0:q1]), ptr(gc), 0, int(topk), 1, ptr(ap),
         ptr(has), ptr(contrib), ptr(ret), stream_ptr())
    out[:m, 0] = ap
    out[:m, 1] = has.to(torch.float64)
    if topk:
        out[:m, 2:] = contrib
    return out


def metrics_from_rows(rows, topk):
    """(Q, 2 + topk) rows of all queries in query order -> (mAP, cmc scores or None), the arithmetic of mean_ap / cmc."""
    Q = rows.shape[0]
    ret = None
    if topk:
        contrib = rows[:, 2:].contiguous()
        ret = torch.empty(topk, dtype=torch.float64, device=rows.device)
        call("reid_cmc_reduce", ptr(contrib), Q, topk, ptr(ret), stream_ptr())
    h = rows[:, :2].cpu().numpy()
    ap, has = h[:, 0].copy(), h[:, 1].astype(np.int32)
    if (has < 0).any():
        raise RuntimeError("a query has more positives than reid_rank_metrics handles")
    aps = ap[has > 0]
    if len(aps) == 0:
        raise RuntimeError("No valid query")
    mAP = np.mean(aps)
    if not topk:
        return mAP, None
    return mAP, ret.cpu().numpy().cumsum() / int((has > 0).sum())


def gather_blocks(name, t, N, group=None):
    """This rank's rows partition(N, W, rank) of an (N, ...) array -> all N rows on every rank (peer stores into a
    cached buffer, or the collective fallback)."""
    W = dist.get_world_size(group)
    B = -(-N // W)
    send = torch.zeros((B,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
    send[: t.shape[0]] = t
    out = sharded.peer_all_gather(name, send, group)
    return torch.cat([out[w * B: w * B + (b - a)] for w, (a, b) in enumerate(partition(N, W, r) for r in range(W))])


def rerank_rows(x, sqnorm, cols, r0, r1):
    """colmax and the neighbour lists initial_rank[:, :cols] of the rows [r0, r1) of x: the values the single-process
    farthest_colmax(x) / knn_search(x, cols, "auto") give those rows (both are exact per row)."""
    from .faiss_rerank import knn_search
    from .rerank import farthest_colmax
    colmax, _ = farthest_colmax(x, sqnorm, rows=(r0, r1))
    rank, _, _ = knn_search(x, cols, "auto", rows=(r0, r1))
    return colmax, rank


def _check_shares(names, share, D, dev, group):
    """One small all-gather, the only host synchronisation before the metrics: every rank extracted exactly its
    eval_shard share, and all with the same feature width D (% 4 == 0).  Every rank raises the same ValueError."""
    W = dist.get_world_size(group)
    mine = torch.tensor([int(sorted(names) == [f for f, _, _ in share]), D], dtype=torch.int64, device=dev)
    got = torch.empty(2 * W, dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(got, mine, group=group)
    flags = got.view(W, 2).tolist()
    bad = [r for r, (ok, _) in enumerate(flags) if not ok]
    if bad:
        raise ValueError("DistributedEvaluator: rank(s) %s extracted other files than eval_shard(query, gallery) "
                         "assigns them" % bad)
    if len({d for _, d in flags}) != 1:
        raise ValueError("DistributedEvaluator: the ranks extracted features of different widths %s" % [d for _, d in flags])
    if D % 4:
        raise ValueError("DistributedEvaluator: feature width D=%d is not a multiple of 4" % D)


class DistributedEvaluator(Evaluator):
    """Evaluator over the ranks of `group` (default: the world group), one process per GPU.  Give each rank a test
    loader over eval_shard(query, gallery) and call evaluate(data_loader, query, gallery, cmc_flag, rerank) with the
    full query and gallery lists on every rank: every rank returns the single-process Evaluator's values; rank 0
    prints the reference's lines.  Without an initialised process group, or with one rank, it is an Evaluator."""

    def __init__(self, model, group=None):
        super(DistributedEvaluator, self).__init__(model)
        self.group = group
        self.steps_ms = None

    def evaluate(self, data_loader, query, gallery, cmc_flag=False, rerank=False):
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(self.group) == 1:
            return super(DistributedEvaluator, self).evaluate(data_loader, query, gallery, cmc_flag, rerank)
        from .evaluation import pairwise_distance_device
        from .rerank import _check_k, _rr_blend, _rr_sparse
        group = self.group
        W, me = dist.get_world_size(group), dist.get_rank(group)
        Q, G = len(query), len(gallery)
        M = Q + G
        qpos, gpos = _positions(query, gallery)
        share = eval_shard(query, gallery, group)
        if len(qpos.keys() | gpos.keys()) < W:
            raise ValueError("DistributedEvaluator: %d distinct test images for %d ranks" % (len(qpos.keys() | gpos.keys()), W))
        features, _ = extract_features(self.model, data_loader)
        names = list(features.keys())
        dev = features.device if features.device is not None else torch.device("cuda", torch.cuda.current_device())
        D = features._buf.shape[1] if names else 0
        marks = []

        def mark(name):
            if TRACE_STEPS:
                e = torch.cuda.Event(enable_timing=True)
                e.record()
                marks.append((name, e))

        _check_shares(names, share, D, dev, group)
        with torch.cuda.device(dev), torch.no_grad():
            mark("start")
            x = scatter_features(features._buf, len(names), dst_table(names, qpos, gpos, dev), M, group)
            mark("scatter")
            del features
            ids = device_ids(query, gallery, dev)
            topk = CMC_TOPK if cmc_flag else 0
            q0, q1 = partition(Q, W, me)
            Bq = -(-Q // W)
            qg = pairwise_distance_device(x[q0:q1], x[Q:]) if q1 > q0 else None
            results = self._gather_metrics(block_metrics(qg, q0, ids, topk, Bq), Q, topk, cmc_flag, me)
            mark("distance_metrics")
            if not rerank:
                self._steps(marks)
                return results
            if me == 0:
                print('Applying person re-ranking ...')
            k1, k2, lam = 20, 6, 0.3
            cols = _check_k(k1, k2, M)
            sqnorm = torch.empty(M, dtype=torch.float64, device=dev)
            call("reid_rr_row_sqnorm64", ptr(x), M, D, ptr(sqnorm), stream_ptr())
            r0, r1 = partition(M, W, me)
            colmax_r, rank_r = rerank_rows(x, sqnorm, cols, r0, r1)
            colmax = gather_blocks("eval_colmax", colmax_r, M, group)
            rank = gather_blocks("eval_rank", rank_r, M, group)
            mark("rerank_search")
            sparse = _rr_sparse(x, sqnorm, colmax, rank, k1, k2)
            mark("sparse_stages")
            out = _rr_blend(x, sparse, colmax, Q, lam, qg, q0, q1) if q1 > q0 else None
            del sparse
            results = self._gather_metrics(block_metrics(out, q0, ids, topk, Bq), Q, topk, cmc_flag, me)
            mark("rerank_blend_metrics")
            self._steps(marks)
            return results

    def _gather_metrics(self, block, Q, topk, cmc_flag, me):
        W = dist.get_world_size(self.group)
        B = block.shape[0]
        out = sharded.peer_all_gather("eval_metrics", block, self.group)
        rows = torch.cat([out[w * B: w * B + (b - a)] for w, (a, b) in enumerate(partition(Q, W, r) for r in range(W))])
        mAP, cmc_scores = metrics_from_rows(rows, topk)
        if me == 0:
            print('Mean AP: {:4.1%}'.format(mAP))
            if cmc_flag:
                _print_cmc(cmc_scores, (1, 5, 10))
        return (cmc_scores, mAP) if cmc_flag else mAP

    def _steps(self, marks):
        if TRACE_STEPS:
            torch.cuda.synchronize()
            self.steps_ms = {b[0]: a[1].elapsed_time(b[1]) for a, b in zip(marks[:-1], marks[1:])}
