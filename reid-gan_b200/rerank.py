"""Drop-in for clustercontrast/utils/rerank.py (SURVEY.md section 8f, row f2):

    distmat = re_ranking(distmat.numpy(), distmat_qq.numpy(), distmat_gg.numpy())     # evaluators.py:141
    re_ranking(q_g_dist, q_q_dist, g_g_dist, k1=20, k2=6, lambda_value=0.3) -> float32 (Q, G)

the evaluation-time k-reciprocal re-ranking behind Evaluator.evaluate(rerank=True).  Same mathematics as the
pseudo-label path on a (query+gallery)^2 matrix of column-max-normalised squared distances (rerank.py:36-41), with
exp(-d) weights (:66-67) and the blend (1 - lambda) * Jaccard + lambda * original (:95-96).  The set / sparse / Jaccard
stages are the kernels of the pseudo-label path; csrc/eval_rerank.cu holds the dense front and back ends.
Everything runs on the current CUDA device through libreid_b200.so; there is no CPU fallback.

    re_ranking_features(query_features, gallery_features, k1=20, k2=6, lambda_value=0.3) -> float32 (Q, G)

is the same function of the features, re_ranking(pairwise_distance(q, g), pairwise_distance(q, q),
pairwise_distance(g, g), ...), without any (Q+G)^2 or G^2 buffer (35 GB each at MSMT17's test split).  A row of the
normalised matrix is a row of squared-squared distances times a constant, so: the neighbour lists are the squared-L2
kNN of the union [q; g] (knn_search), the column maxima are a farthest-neighbour search (farthest_colmax), the
weights are gathered from feature rows, and the blend reads the Q x G distance block (csrc/eval_features.cu).
"""
import numpy as np
import torch

from . import _lib
from ._lib import call, ptr, stream_ptr
from .faiss_rerank import _device_of, _scan, half_k, knn_search


def _dev_f32(a, dev):
    if isinstance(a, np.ndarray):
        a = torch.from_numpy(np.ascontiguousarray(a))
    return a.to(device=dev, dtype=torch.float32).contiguous()


def _check_k(k1, k2, M):
    cols = k1 + 1                                                # initial_rank[i, :k1+1]   (rerank.py:51-52)
    if not (1 <= k1 and cols <= 64 and cols <= M):
        raise ValueError("k1=%d outside the supported range (k1 + 1 <= min(64, Q + G))" % k1)
    if not (1 <= k2 <= cols):
        raise ValueError("k2=%d must be in 1..k1+1" % k2)
    return cols


def _sparse_stages(rank, M, k1, k2, weights, dev):
    """rerank.py:50-78 on the (M, k1+1) neighbour lists: k-reciprocal sets, expansion, weights (`weights(e_pad,
    e_stride, e_ptr, e_idx, v_val)` fills the CSR values), query expansion and inverted index.  Returns the CSR of V_qe
    and its CSC, what the Jaccard rows read, plus the expansion CSR (ptr, idx) for callers that inspect the sets."""
    L = _lib.lib()
    sp = stream_ptr()
    cols = rank.shape[1]
    # :50-64  k-reciprocal sets and their expansion
    h = half_k(k1)
    R = torch.empty(M, dtype=torch.int64, device=dev)
    Rh = torch.empty(M, dtype=torch.int64, device=dev)
    call("reid_reciprocal_masks", ptr(rank), M, cols, k1, 0, M, ptr(R), sp)
    call("reid_reciprocal_masks", ptr(rank), M, cols, h, 0, M, ptr(Rh), sp)
    half_cols = min(h + 1, cols)
    e_stride = min(cols + cols * half_cols, 1024)
    e_pad = torch.empty(M * e_stride, dtype=torch.int32, device=dev)
    e_cnt = torch.empty(M, dtype=torch.int32, device=dev)
    call("reid_expand", ptr(rank), M, cols, half_cols, ptr(R), ptr(Rh), 0, M, e_stride, ptr(e_pad), ptr(e_cnt), sp)
    e_ptr, e_total, e_max = _scan(e_cnt, M, dev)
    if e_max > e_stride:
        raise RuntimeError("re_ranking: an expansion set exceeded %d entries" % e_stride)
    # :66-67  weights
    e_idx = torch.empty(max(e_total, 1), dtype=torch.int32, device=dev)
    v_val = torch.empty(max(e_total, 1), dtype=torch.float32, device=dev)
    weights(e_pad, e_stride, e_ptr, e_idx, v_val)
    # :69-74  query expansion
    if k2 != 1:
        q_stride = L.reid_query_expand_stride(k2, max(e_max, 1))
        q_cnt = torch.empty(M, dtype=torch.int32, device=dev)
        qp_idx = torch.empty(M * q_stride, dtype=torch.int32, device=dev)
        qp_val = torch.empty(M * q_stride, dtype=torch.float32, device=dev)
        call("reid_query_expand", ptr(rank), M, cols, k2, ptr(e_ptr), ptr(e_idx), ptr(v_val), max(e_max, 1), 0, M,
             ptr(q_cnt), ptr(qp_idx), ptr(qp_val), None, 0, sp)
        q_ptr, q_total, _ = _scan(q_cnt, M, dev)
        q_idx = torch.empty(max(q_total, 1), dtype=torch.int32, device=dev)
        q_val = torch.empty(max(q_total, 1), dtype=torch.float32, device=dev)
        call("reid_csr_compact", ptr(qp_idx), ptr(qp_val), q_stride, ptr(q_cnt), ptr(q_ptr), M, ptr(q_idx), ptr(q_val), sp)
        del qp_idx, qp_val
    else:
        q_ptr, q_idx, q_val, q_total = e_ptr, e_idx, v_val, e_total
    # :76-78  inverted index
    c_cnt = torch.empty(M, dtype=torch.int32, device=dev)
    call("reid_transpose_count", ptr(q_idx), q_total, None, M, ptr(c_cnt), sp)
    c_ptr, _, c_max = _scan(c_cnt, M, dev)
    c_idx = torch.empty(max(q_total, 1), dtype=torch.int32, device=dev)
    c_val = torch.empty(max(q_total, 1), dtype=torch.float32, device=dev)
    call("reid_transpose_fill", ptr(q_ptr), ptr(q_idx), ptr(q_val), M, M, ptr(c_ptr), ptr(c_cnt), ptr(c_idx), ptr(c_val),
         int(c_max), sp)
    return dict(Q=(q_ptr, q_idx, q_val), C=(c_ptr, c_idx, c_val), E=(e_ptr, e_idx[:e_total], v_val[:e_total]))


def _jaccard_blend(sparse, M, Q, lambda_value, blend, dev):
    """rerank.py:80-96: Jaccard rows of the queries in blocks of rows (<= 512 MB each); `blend(J, r0, r1, 1 - lambda,
    lambda)` writes rows [r0, r1) of the result."""
    sp = stream_ptr()
    q_ptr, q_idx, q_val = sparse["Q"]
    c_ptr, c_idx, c_val = sparse["C"]
    block = max(1, min(Q, (512 << 20) // (4 * M)))
    a_ = float(np.float32(1 - lambda_value))
    b_ = float(np.float32(lambda_value))
    for r0 in range(0, Q, block):
        r1 = min(Q, r0 + block)
        J = torch.empty((r1 - r0, M), dtype=torch.float32, device=dev)
        call("reid_jaccard_dense", ptr(q_ptr), ptr(q_idx), ptr(q_val), ptr(c_ptr), ptr(c_idx), ptr(c_val), M, r0, r1, ptr(J),
             M, 0, sp)
        blend(J, r0, r1, a_, b_)


def re_ranking(q_g_dist, q_q_dist, g_g_dist, k1=20, k2=6, lambda_value=0.3, return_device=False):
    _lib.lib()
    dev = _device_of(q_g_dist if isinstance(q_g_dist, torch.Tensor) else None)
    with torch.cuda.device(dev), torch.no_grad():
        qg, qq, gg = _dev_f32(q_g_dist, dev), _dev_f32(q_q_dist, dev), _dev_f32(g_g_dist, dev)
        Q, G = qg.shape
        if qq.shape != (Q, Q) or gg.shape != (G, G):
            raise ValueError("expected q_g (Q, G), q_q (Q, Q), g_g (G, G); got %s %s %s" % (tuple(qg.shape), tuple(qq.shape), tuple(gg.shape)))
        M = Q + G
        cols = _check_k(k1, k2, M)
        sp = stream_ptr()
        # :36-41  normalised squared distances, transposed
        scratch = torch.empty((M, M), dtype=torch.float32, device=dev)
        colmax = torch.empty(M, dtype=torch.float32, device=dev)
        dist = torch.empty((M, M), dtype=torch.float32, device=dev)
        call("reid_rr_normalised_distance", ptr(qg), ptr(qq), ptr(gg), Q, G, ptr(scratch), ptr(colmax), ptr(dist), sp)
        del scratch
        # :43  initial_rank (only the first k1+1 columns are ever read)
        rank = torch.empty((M, cols), dtype=torch.int32, device=dev)
        call("reid_select_rows", ptr(dist), M, M, cols, 1, ptr(rank), None, sp)

        def weights(e_pad, e_stride, e_ptr, e_idx, v_val):
            call("reid_rr_weights", ptr(dist), M, ptr(e_pad), e_stride, ptr(e_ptr), M, ptr(e_idx), ptr(v_val), sp)

        def blend(J, r0, r1, a_, b_):
            call("reid_rr_final", ptr(J), M, ptr(dist[r0:]), r1 - r0, G, a_, b_, ptr(out[r0:]), sp)

        out = torch.empty((Q, G), dtype=torch.float32, device=dev)
        _jaccard_blend(_sparse_stages(rank, M, k1, k2, weights, dev), M, Q, lambda_value, blend, dev)
        if return_device:
            return out
        return out.cpu().numpy()


FARTHEST_TC_MIN = 4096       # below this many rows the exact scan is cheap; the tensor-core search needs D % 64 == 0
FARTHEST_KEEP = 16           # candidates kept per list (per row: 2 x column splits lists)
FARTHEST_BLOCK = 16384       # rows per candidate pass: their lists take 2 x splits x 512 x 8 B = 8..32 KB a row


def farthest_colmax(x, sqnorm=None, mode="auto"):
    """colmax[i] = max_j fp32(sq(i, j)^2) over all rows j of the (M, D) float32 CUDA tensor x (rerank.py:41's
    np.max(original_dist, axis=0) of the union).  Returns (colmax float32 (M,), info).

    mode "tc" (what "auto" picks for M >= FARTHEST_TC_MIN, D % 64 == 0 and rows of one norm): the fp16 tcgen05 candidate
    kernel of the kNN search run against the NEGATED operand keeps the few smallest approximate dot products per row;
    reid_rr_farthest_certify re-scores the window and certifies the row; the rows it cannot certify
    (info["uncertified_rows"]) go through the exact scan.  mode "exact": the exact CUDA-core scan for every row."""
    import ctypes
    from .knn_tc import SCALE_LOG2, TC_CAP, CTA_GROUP, one_norm
    _device_of(x)
    if not (x.is_cuda and x.dtype == torch.float32 and x.dim() == 2 and x.is_contiguous()):
        raise ValueError("farthest_colmax takes a contiguous float32 (M, D) CUDA tensor")
    M, D = x.shape
    dev = x.device
    sp = stream_ptr()
    if sqnorm is None:
        sqnorm = torch.empty(M, dtype=torch.float64, device=dev)
        call("reid_rr_row_sqnorm64", ptr(x), M, D, ptr(sqnorm), sp)
    colmax = torch.empty(M, dtype=torch.float32, device=dev)
    info = {"mode": mode, "uncertified_rows": 0}
    if mode not in ("auto", "tc", "exact"):
        raise ValueError("unknown farthest-search mode %r" % (mode,))
    if mode == "auto":
        mode = "tc" if (D % 64 == 0 and M >= FARTHEST_TC_MIN) else "exact"
    if mode == "tc":
        xh = torch.empty((M, D), dtype=torch.float16, device=dev)
        msq = torch.zeros(2, dtype=torch.float32, device=dev)
        call("reid_features_to_half", ptr(x), M, D, SCALE_LOG2, ptr(xh), ptr(msq), sp)
        if info["mode"] == "auto" and not one_norm(msq.tolist()):
            mode = "exact"                                    # rows of different norms: no useful certificate
            del xh
    info["mode"] = mode
    if mode == "exact":
        call("reid_rr_farthest_exact", ptr(x), M, D, ptr(sqnorm), None, 0, M, ptr(colmax), sp)
        return colmax, info
    xn = torch.neg(xh)
    flag = torch.empty(M, dtype=torch.int32, device=dev)
    for r0 in range(0, M, FARTHEST_BLOCK):
        r1 = min(M, r0 + FARTHEST_BLOCK)
        n = r1 - r0
        s = ctypes.c_int(1)
        call("reid_knn_tc_plan", M, n, CTA_GROUP, ctypes.byref(s))
        n_lists = 2 * s.value
        cand = torch.empty(n * n_lists * TC_CAP, dtype=torch.int64, device=dev)
        cand_cnt = torch.zeros(n * n_lists, dtype=torch.int32, device=dev)
        tau = torch.empty(n, dtype=torch.int32, device=dev)
        call("reid_knn_candidates_tc_ab", ptr(xh), M, ptr(xn), M, D, SCALE_LOG2, r0, r1, FARTHEST_KEEP, s.value, CTA_GROUP,
             ptr(cand), ptr(cand_cnt), ptr(tau), sp)
        call("reid_rr_farthest_certify", ptr(x), M, D, ptr(sqnorm), ptr(cand), ptr(cand_cnt), ptr(tau), n_lists, TC_CAP, r0, r1,
             ptr(msq), ptr(colmax), ptr(flag[r0:]), None, sp)
        del cand, cand_cnt, tau
    del xh, xn
    bad = torch.nonzero(flag).flatten().to(torch.int32).contiguous()
    if bad.numel():
        call("reid_rr_farthest_exact", ptr(x), M, D, ptr(sqnorm), ptr(bad), 0, bad.numel(), ptr(colmax), sp)
    info["uncertified_rows"] = int(bad.numel())
    return colmax, info


def _as_features(a, dev, what):
    if isinstance(a, np.ndarray):
        a = torch.from_numpy(np.ascontiguousarray(a))
    if not isinstance(a, torch.Tensor) or a.dim() != 2:
        raise ValueError("%s must be a 2-D (rows, D) array or tensor" % what)
    return a.to(device=dev, dtype=torch.float32).contiguous()


def _re_ranking_features(query_features, gallery_features, k1=20, k2=6, lambda_value=0.3, q_g_dist=None):
    """re_ranking_features on the device; returns (out (Q, G) CUDA tensor, parts).  q_g_dist: the (Q, G)
    pairwise_distance_device(q, g) block when the caller has it already (Evaluator.evaluate), else it is computed."""
    from .evaluation import pairwise_distance_device
    _lib.lib()
    _check_k(k1, k2, 64)                                      # k1 + 1 <= 64 before anything touches a device
    ref = query_features if isinstance(query_features, torch.Tensor) else None
    dev = _device_of(ref)
    with torch.cuda.device(dev), torch.no_grad():
        q = _as_features(query_features, dev, "query_features")
        g = _as_features(gallery_features, dev, "gallery_features")
        Q, D = q.shape
        G = g.shape[0]
        if g.shape[1] != D or Q < 1 or G < 1:
            raise ValueError("expected (Q, D) and (G, D) features; got %s %s" % (tuple(q.shape), tuple(g.shape)))
        M = Q + G
        cols = _check_k(k1, k2, M)
        if q_g_dist is not None and (tuple(q_g_dist.shape) != (Q, G) or not q_g_dist.is_cuda
                                     or q_g_dist.dtype != torch.float32 or not q_g_dist.is_contiguous()):
            raise ValueError("q_g_dist must be the contiguous float32 (Q, G) CUDA block of pairwise_distance_device(q, g)")
        sp = stream_ptr()
        x = torch.cat([q, g]).contiguous()
        del q
        sqnorm = torch.empty(M, dtype=torch.float64, device=dev)
        call("reid_rr_row_sqnorm64", ptr(x), M, D, ptr(sqnorm), sp)
        # :41  column maxima of the squared-squared distances (a farthest-neighbour search)
        colmax, far_info = farthest_colmax(x, sqnorm)
        # :43  initial_rank[:, :k1+1]: a row of dist is a row of orig over a positive constant -- the squared-L2 kNN
        rank, _, knn_info = knn_search(x, cols, "auto")

        def weights(e_pad, e_stride, e_ptr, e_idx, v_val):
            call("reid_rr_weights_features", ptr(x), M, D, ptr(sqnorm), ptr(colmax), ptr(e_pad), e_stride, ptr(e_ptr), M,
                 ptr(e_idx), ptr(v_val), sp)

        sparse = _sparse_stages(rank, M, k1, k2, weights, dev)
        if q_g_dist is None:
            q_g_dist = pairwise_distance_device(x[:Q], g)
        del g
        out = torch.empty((Q, G), dtype=torch.float32, device=dev)

        def blend(J, r0, r1, a_, b_):
            call("reid_rr_final_qg", ptr(J), M, ptr(q_g_dist), ptr(colmax), Q, G, r0, r1, a_, b_, ptr(out), sp)

        _jaccard_blend(sparse, M, Q, lambda_value, blend, dev)
        parts = dict(rank=rank, colmax=colmax, E=sparse["E"], knn_info=knn_info, farthest_info=far_info)
        return out, parts


def re_ranking_features(query_features, gallery_features, k1=20, k2=6, lambda_value=0.3, return_device=False):
    """re_ranking(pairwise_distance(q, g), pairwise_distance(q, q), pairwise_distance(g, g), k1, k2, lambda_value)
    from the (Q, D) query and (G, D) gallery features (CUDA tensors, host tensors or numpy), without any buffer of
    (Q+G)^2 or G^2 elements.  Returns the float32 (Q, G) matrix (numpy; a CUDA tensor with return_device=True)."""
    out, _ = _re_ranking_features(query_features, gallery_features, k1, k2, lambda_value)
    if return_device:
        return out
    return out.cpu().numpy()
