"""GPU (-m gpu): the argument behind every neighbour list of the tensor-core kNN search (knn_rescore.cu, DESIGN 4 K2),
one clause at a time, against float64 references computed here with torch / numpy:

  1. premise     -- a candidate producer leaves out of a row's lists only columns whose fp16 score is at most the
                    row's threshold (reid_knn_candidates_tc, _tc_ab, the symmetric search in both layouts);
  2. error model -- an fp16 score is within eps = 1.02 * 2^-10 * max ||x||^2 + 2^-14 of the exact dot, with the
                    max ||x||^2 that reid_features_to_half reports;
  3. certificate -- reid_knn_rescore(_mapped) certifies a row only when its lists hold the exact top-k, and then
                    returns that top-k with the canonical keys, ordered by (key desc, index asc).

approx_ref = the dots of the fp16 operands xh = fp16(16 x) in float64, times 2^-8 (what the tensor cores compute up
to the fp32 accumulation); exact_ref = float64 dots of the fp32 rows rounded once to fp32 (the canonical key)."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

BLOCK = 2048                    # row block of the reference products
SPIKE = 5000.0                  # 16 * 5000 > 65504: a component that overflows the fp16 operand


# ---- references -------------------------------------------------------------------------------------------------
def fp16_operand(x):
    return (x * 16.0).half()


def refs(x):
    """(approx_ref, |xh|.|xh| * 2^-8, exact_ref) as (N, N) device matrices: float64, float64, float32."""
    N = x.shape[0]
    xh = fp16_operand(x).double()
    xa = xh.abs()
    xd = x.double()
    approx = torch.empty((N, N), dtype=torch.float64, device=x.device)
    absp = torch.empty_like(approx)
    exact = torch.empty((N, N), dtype=torch.float32, device=x.device)
    for b in range(0, N, BLOCK):
        e = min(N, b + BLOCK)
        approx[b:e] = (xh[b:e] @ xh.T) * 2.0 ** -8
        absp[b:e] = (xa[b:e] @ xa.T) * 2.0 ** -8
        exact[b:e] = (xd[b:e] @ xd.T).float()
    return approx, absp, exact


def eps_of(max_sqnorm):
    """knn_tc.err_bound."""
    return float(max_sqnorm) * (2.0 ** -10) * 1.02 + 2.0 ** -14


def float_ord(f):
    """common.cuh float_ord, numpy: float32 -> order-preserving uint32."""
    b = np.ascontiguousarray(f, dtype=np.float32).view(np.uint32)
    return np.where(b & 0x80000000, ~b, b | 0x80000000).astype(np.uint32)


def ord_float(o):
    """common.cuh ord_float, numpy: the threshold image back to float32; 0 = no threshold = -inf."""
    o = np.ascontiguousarray(o).view(np.uint32)
    b = np.where(o & 0x80000000, o & 0x7FFFFFFF, ~o).astype(np.uint32)
    f = b.view(np.float32).copy()
    f[o == 0] = -np.inf
    return f


def decode(cand, cap):
    """List entries (fp32 score bits << 32) | column -> (score float32, column int64), shaped (lists, cap)."""
    c = cand.view(-1, cap)
    return (c >> 32).to(torch.int32).view(torch.float32), c & 0xFFFFFFFF


def pack(score, col):
    """numpy inverse of decode."""
    s = np.ascontiguousarray(score, dtype=np.float32).view(np.uint32).astype(np.uint64)
    return ((s << np.uint64(32)) | np.asarray(col).astype(np.uint64)).view(np.int64)


# ---- data -------------------------------------------------------------------------------------------------------
def spike_set(N, D, seed, mixed=False, norm=1e4, n_spike=6):
    """Rows of norm 1e4 (x0.5-1.5 with mixed) in clusters of ~16.  Every row has equal components 0 and 1; a few spike
    rows hold +5000 / -5000 there instead, and their other components point at their cluster.  The exact dot of a
    spike row with a cluster mate does not see the spike, and it is among the mate's top 30; its fp16 score is
    inf * h - inf * h = NaN."""
    import reid_gan_b200 as rg
    g = torch.Generator().manual_seed(seed + 101)
    x, _ = rg.synth(N, D, max(1, N // 16), 0.5, seed)
    x[:, 1] = x[:, 0]
    x = F.normalize(x, dim=1) * norm
    if mixed:
        x *= 0.5 + torch.rand(N, 1, generator=g)
    spikes = torch.randperm(N, generator=g)[:n_spike]
    for s in spikes.tolist():
        r = x[s].clone()
        r[:2] = 0.0
        r = r / r.norm() * math.sqrt(norm ** 2 - 2 * SPIKE ** 2)
        r[0], r[1] = SPIKE, -SPIKE
        x[s] = r
    return x.contiguous()


def family(name, N, D, seed=0):
    import reid_gan_b200 as rg
    g = torch.Generator().manual_seed(seed + 7)
    if name == "iso":
        x, _ = rg.synth(N, D, N, 1.0, seed)
    elif name == "clusters":                                  # ids = 8: windows far above 128 members
        x, _ = rg.synth(N, D, 8, 0.3, seed)
    elif name == "dup":                                       # exact duplicates: equal scores, the index decides
        x, _ = rg.synth(N, D, max(1, N // 31), 0.8, seed)
        d = min(300, N // 3)
        x[N - d:] = x[:d]
    elif name == "sorted":                                    # rows listed by identity
        x, ids = rg.synth(N, D, max(1, N // 31), 0.8, seed)
        x = x[torch.argsort(ids, stable=True)]
    elif name == "mixed":
        x, _ = rg.synth(N, D, max(1, N // 31), 0.8, seed)
        x = x * (0.5 + torch.rand(N, 1, generator=g))
    elif name == "big":
        x = rg.synth(N, D, max(1, N // 31), 0.8, seed)[0] * 1e3
    elif name == "tiny":
        x = rg.synth(N, D, max(1, N // 31), 0.8, seed)[0] * 1e-3
    elif name == "spike":
        x = spike_set(N, D, seed)
    elif name == "spike-mixed":
        x = spike_set(N, D, seed, mixed=True)
    else:
        raise ValueError(name)
    return x.contiguous().cuda()


def to_half(x):
    """(xh, [max, min] ||x||^2 as reid_features_to_half reports it)."""
    from reid_gan_b200._lib import call, ptr, stream_ptr
    N, D = x.shape
    xh = torch.empty((N, D), dtype=torch.float16, device=x.device)
    msq = torch.zeros(2, dtype=torch.float32, device=x.device)
    call("reid_features_to_half", ptr(x), N, D, 4, ptr(xh), ptr(msq), stream_ptr())
    return xh, msq


# ---- clause checks on the lists of a producer -------------------------------------------------------------------
def check_lists(tag, rows, cols, scores, tau, skip_rows, A, P, E, eps, D, keep=None, sym=False):
    """rows / cols / scores: every listed entry (device tensors); tau: float64 (n,) thresholds; skip_rows: bool (n,)
    rows whose lists overflowed (the re-score refuses them, so (c) and (d) do not apply).  A / P / E: approx_ref,
    |xh|.|xh| 2^-8 and exact_ref restricted to the producer's rows x columns.  Returns the largest
    |score - approx_ref| seen."""
    n, M = A.shape
    # (a) no column twice in a row's lists: the re-score ranks by counting strictly greater keys
    flat = rows * M + cols
    n_unique = torch.unique(flat).numel()
    assert n_unique == flat.numel(), "%s: %d duplicated entries" % (tag, flat.numel() - n_unique)
    # (b) listed scores are the fp16 dots up to fp32 accumulation in any order: D 2^-23 sum |xh_i,d xh_j,d| 2^-8
    a = A[rows, cols]
    s = scores.double()
    bound = D * 2.0 ** -23 * P[rows, cols]
    fin = torch.isfinite(a)
    dev_b = (s - a).abs()
    ok = torch.where(fin, dev_b <= bound, (s == a) | (torch.isnan(s) & torch.isnan(a)))
    bad = torch.nonzero(~ok).flatten()
    assert bad.numel() == 0, "%s: listed score off the fp16 reference: row %d col %d score %r approx %r bound %r" % (
        tag, int(rows[bad[0]]), int(cols[bad[0]]), float(s[bad[0]]), float(a[bad[0]]), float(bound[bad[0]]))
    max_dev = float(dev_b[fin].max()) if bool(fin.any()) else 0.0
    # (c) the premise: every column a row did not list has exact_ref <= tau + eps
    listed = torch.zeros((n, M), dtype=torch.bool, device=A.device)
    listed[rows, cols] = True
    tau_d = torch.as_tensor(tau, dtype=torch.float64, device=A.device)
    viol = ~listed & (E.double() > tau_d[:, None] + eps) & ~skip_rows[:, None]
    if bool(viol.any()):
        r, c = (int(v) for v in torch.nonzero(viol)[0])
        raise AssertionError("%s: premise broken on %d pairs, e.g. row %d col %d: exact %r > tau %r + eps %r (approx %r)"
                             % (tag, int(viol.sum()), r, c, float(E[r, c]), float(tau_d[r]), eps, float(A[r, c])))
    # (d) tc: at least `keep` listed scores >= tau (rows whose fp16 scores are all numbers)
    if keep is not None:
        ge = torch.zeros(n, dtype=torch.int64, device=A.device)
        ge.index_add_(0, rows, (s >= tau_d[rows]).long())
        finite_row = torch.isfinite(A).all(dim=1)
        short = (ge < keep) & finite_row & ~skip_rows
        assert not bool(short.any()), "%s: row %d lists %d scores >= its threshold, keep = %d" % (
            tag, int(torch.nonzero(short)[0]), int(ge[short][0]), keep)
    # (e) symmetric search: every pair clearly above both thresholds is listed in both directions
    if sym:
        above = (A > tau_d[:, None] + 2 * eps) & (A > tau_d[None, :] + 2 * eps)
        miss = above & ~(listed & listed.T)
        assert not bool(miss.any()), "%s: %d pairs above both thresholds not listed both ways, e.g. %s" % (
            tag, int(miss.sum()), torch.nonzero(miss)[0].tolist())
    return max_dev


def row_major_entries(cand, cnt, n, n_lists, cap):
    """Every listed entry of row-major lists: (rows, cols, scores, rows with an overflowed list)."""
    cnt = cnt[:n * n_lists].long()
    sc, col = decode(cand[:n * n_lists * cap], cap)
    valid = torch.arange(cap, device=cand.device)[None, :] < cnt.clamp(max=cap)[:, None]
    row = (torch.arange(n * n_lists, device=cand.device) // n_lists)[:, None].expand(-1, cap)
    over = (cnt.view(n, n_lists) > cap).any(dim=1)
    return row[valid], col[valid], sc[valid], over


REPORT = {}


def _report(fam, what, value, eps):
    cur = REPORT.setdefault((fam, what), [0.0, eps])
    cur[0] = max(cur[0], value)
    print("%-12s %-26s max %.3e   eps %.3e" % (fam, what, value, eps))


# ---- A. candidate producers keep their promise on every pair -----------------------------------------------------
@pytest.mark.parametrize("fam,N,D,k", [
    ("iso", 256, 64, 1),
    ("iso", 300, 192, 33),
    ("clusters", 1000, 512, 30),
    ("dup", 1000, 64, 64),
    ("sorted", 4173, 192, 30),
    ("mixed", 1000, 192, 30),
    ("big", 1000, 64, 30),
    ("tiny", 300, 64, 30),
    ("spike", 1000, 256, 30),
    ("iso", 300, 2048, 64),
])
def test_tc_producers_keep_the_premise(fam, N, D, k):
    """Premise and error model, one-sided kernel: reid_knn_candidates_tc (keep = min(k + 34, 64), the planned column
    splits and 1 / 2 / 4 forced) and reid_knn_candidates_tc_ab in prepass mode (negative keep, against the threshold
    sample).  Clauses (a)-(d) on all N^2 pairs; also |approx_ref - exact_ref| <= eps on all pairs."""
    import ctypes
    from reid_gan_b200 import knn_tc
    from reid_gan_b200._lib import call, ptr, stream_ptr
    x = family(fam, N, D)
    A, P, E = refs(x)
    xh, msq = to_half(x)
    assert torch.equal(xh, fp16_operand(x)), "reid_features_to_half must round like torch's .half() of 16 x"
    eps = eps_of(msq[0])
    true_sq = (x.double() ** 2).sum(dim=1)
    assert float(msq[0]) >= float(true_sq.max()) * (1 - 1e-6) and float(msq[1]) <= float(true_sq.min()) * (1 + 1e-6)
    err = (A - E.double()).abs()
    err[~torch.isfinite(A)] = math.inf
    _report(fam, "|approx - exact|", float(err[torch.isfinite(err)].max()), eps)
    assert float(err.max()) <= eps, "error model: |approx - exact| = %r > eps = %r" % (float(err.max()), eps)
    sp = stream_ptr()
    keep = max(k, min(k + knn_tc.SLACK, knn_tc.KEEP_MAX))
    planned = ctypes.c_int(1)
    call("reid_knn_tc_plan", N, N, knn_tc.CTA_GROUP, ctypes.byref(planned))
    n_t = (N + 255) // 256
    for s in sorted({planned.value, 1, 2, 4}):
        if s > n_t:
            continue
        n_lists = 2 * s
        cand = torch.empty(N * n_lists * knn_tc.TC_CAP, dtype=torch.int64, device=x.device)
        cnt = torch.zeros(N * n_lists, dtype=torch.int32, device=x.device)
        tau_o = torch.empty(N, dtype=torch.int32, device=x.device)
        call("reid_knn_candidates_tc", ptr(xh), N, D, 4, 0, N, keep, s, knn_tc.CTA_GROUP, ptr(cand), ptr(cnt), ptr(tau_o), sp)
        rows, cols, sc, over = row_major_entries(cand, cnt, N, n_lists, knn_tc.TC_CAP)
        tau = ord_float(tau_o.cpu().numpy()).astype(np.float64)
        d = check_lists("tc n_splits=%d" % s, rows, cols, sc, tau, over, A, P, E, eps, D, keep=keep)
        _report(fam, "|score - approx| tc", d, eps)
    # the sampling prepass: all rows against the threshold sample
    m = knn_tc.sample_size(N, k)
    samp = torch.as_tensor((np.arange(m) * knn_tc._sample_stride(N, m)) % N, device=x.device)
    xs = torch.empty((m, D), dtype=torch.float16, device=x.device)
    call("reid_features_sample", ptr(xh), N, D, m, knn_tc._sample_stride(N, m), ptr(xs), sp)
    assert torch.equal(xs, xh[samp])
    # prepass mode seeds each list's threshold, so row_tau bounds what the lists rejected only with publish_final
    # (reid_knn_candidates_tc_abt): clauses (a) and (b) for the plain entry, (a)-(c) with publish_final
    for publish in (0, 1):
        cand = torch.empty(N * 2 * knn_tc.TC_CAP, dtype=torch.int64, device=x.device)
        cnt = torch.zeros(N * 2, dtype=torch.int32, device=x.device)
        tau_o = torch.empty(N, dtype=torch.int32, device=x.device)
        if publish:
            call("reid_knn_candidates_tc_abt", ptr(xh), N, ptr(xs), m, D, 4, 0, N, -knn_tc.sym_rank(k), 1, 2, ptr(cand),
                 ptr(cnt), ptr(tau_o), 1, None, None, None, 0, sp)
            tau = ord_float(tau_o.cpu().numpy()).astype(np.float64)
        else:
            call("reid_knn_candidates_tc_ab", ptr(xh), N, ptr(xs), m, D, 4, 0, N, -knn_tc.sym_rank(k), 1, 2, ptr(cand),
                 ptr(cnt), ptr(tau_o), sp)
            tau = np.full(N, np.inf)                          # no premise without publish_final
        rows, cols, sc, over = row_major_entries(cand, cnt, N, 2, knn_tc.TC_CAP)
        d = check_lists("tc_ab prepass publish_final=%d" % publish, rows, cols, sc, tau, over, A[:, samp], P[:, samp],
                        E[:, samp], eps, D)
        _report(fam, "|score - approx| prepass", d, eps)


@pytest.mark.parametrize("fam,N,D,k", [
    ("iso", 8192, 64, 30),
    ("clusters", 8269, 192, 33),
    ("dup", 8192, 128, 64),
    ("sorted", 12345, 64, 30),
    ("mixed", 8269, 128, 1),
    ("big", 8192, 64, 30),
    ("tiny", 8192, 64, 30),
    ("spike", 8192, 256, 30),
    ("iso", 8192, 2048, 30),
    ("iso", 12345, 512, 64),
])
def test_symmetric_producers_keep_the_premise(fam, N, D, k):
    """Premise and error model, symmetric search: knn_tc._candidates_sym (separate sample) and _candidates_sym_sf
    (sample-first; positions mapped back with its (pos_of, orig_of)).  Clauses (a)-(c) and (e) on all N^2 pairs."""
    from reid_gan_b200 import knn_tc
    from reid_gan_b200._lib import stream_ptr
    x = family(fam, N, D)
    A, P, E = refs(x)
    xh, msq = to_half(x)
    eps = eps_of(msq[0])
    err = (A - E.double()).abs()
    err[~torch.isfinite(A)] = math.inf
    _report(fam, "|approx - exact|", float(err[torch.isfinite(err)].max()), eps)
    assert float(err.max()) <= eps, "error model: |approx - exact| = %r > eps = %r" % (float(err.max()), eps)
    sp = stream_ptr()
    cand, cnt, tau_o, cap, _ = knn_tc._candidates_sym(xh, N, D, sp, x.device, k)
    rows, cols, sc, over = row_major_entries(cand, cnt, N, 1, cap)
    tau = ord_float(tau_o.cpu().numpy()).astype(np.float64)
    d = check_lists("sym", rows, cols, sc, tau, over, A, P, E, eps, D, sym=True)
    _report(fam, "|score - approx| sym", d, eps)
    if knn_tc.sample_size(N, k) % 256 == 0 and N - knn_tc.sample_size(N, k) >= 256:
        msq_sf = torch.zeros(2, dtype=torch.float32, device=x.device)
        cand, cnt, tau_o, cap, _, xh_sf, (pos_of, orig_of) = knn_tc._candidates_sym_sf(x, N, D, sp, x.device, k, msq_sf)
        assert torch.equal(msq_sf, msq), "the sample-first conversion must report the same range"
        assert torch.equal(xh_sf, xh[orig_of.long()])
        rows, cols, sc, over = row_major_entries(cand, cnt, N, 1, cap)
        o = orig_of.long()
        tau_pos = ord_float(tau_o.cpu().numpy()).astype(np.float64)
        tau = np.empty_like(tau_pos)
        tau[o.cpu().numpy()] = tau_pos
        over_o = torch.empty_like(over)
        over_o[o] = over
        d = check_lists("sym sample-first", o[rows], o[cols], sc, tau, over_o, A, P, E, eps, D, sym=True)
        _report(fam, "|score - approx| sym-sf", d, eps)


# ---- B. the re-score certificate on crafted lists ----------------------------------------------------------------
B_EPS = 1e-3


def craft(a, tau, strict, n_lists, cap=None, list_major=False, seed=0):
    """Lists of every row r: the columns with a > tau[r] (strict) or a >= tau[r], in a random order, dealt
    round-robin over n_lists lists.  Unused slots hold (-inf, r).  Returns (cand, cnt, cap) as device tensors."""
    n, M = a.shape
    sel = np.where(strict[:, None], a > tau[:, None], a >= tau[:, None])
    rows, cols = np.nonzero(sel)
    rng = np.random.default_rng(seed)
    order = np.lexsort((rng.random(rows.size), rows))
    rows, cols = rows[order], cols[order]
    first = np.searchsorted(rows, rows)
    t = np.arange(rows.size) - first
    q, p = t % n_lists, t // n_lists
    li = q * n + rows if list_major else rows * n_lists + q
    cnt = np.zeros(n * n_lists, dtype=np.int32)
    np.add.at(cnt, li, 1)
    cap = int(cnt.max()) if cap is None else cap
    assert cnt.max() <= cap
    owner = (np.arange(n * n_lists) % n) if list_major else (np.arange(n * n_lists) // n_lists)
    cand = np.repeat(pack(np.full(n * n_lists, -np.inf, np.float32), owner), cap)
    cand[li * cap + p] = pack(a[rows, cols], cols)
    dev = torch.device("cuda")
    return torch.from_numpy(cand).to(dev), torch.from_numpy(cnt).to(dev), cap


def rescore(x, cand, cnt, tau, n_lists, cap, k, eps=B_EPS, pitch=0, locality=1, r0=0, r1=None, maps=None, count=None):
    """reid_knn_rescore(_mapped) with err_bound = eps; tau float32 numpy thresholds.  Returns (idx, key, flag, max_err)."""
    from reid_gan_b200 import _lib
    from reid_gan_b200._lib import call, ptr, stream_ptr
    N, D = x.shape
    r1 = N if r1 is None else r1
    n = r1 - r0
    dev = x.device
    tau_o = torch.from_numpy(float_ord(tau).view(np.int32).copy()).to(dev)
    idx = torch.empty((n, k), dtype=torch.int32, device=dev)
    key = torch.empty((n, k), dtype=torch.float32, device=dev)
    flag = torch.empty(n, dtype=torch.int32, device=dev)
    max_err = torch.zeros(1, dtype=torch.float32, device=dev)
    ws = torch.empty(_lib.lib().reid_knn_rescore_workspace_bytes(N, n), dtype=torch.uint8, device=dev)
    if maps is None:
        call("reid_knn_rescore", ptr(x), N, D, r0, r1, ptr(cand), ptr(cnt), ptr(tau_o), n_lists, cap, pitch, k, eps, None,
             locality, ptr(idx), ptr(key), ptr(flag), ptr(max_err), ptr(ws), ptr(count), stream_ptr())
    else:
        call("reid_knn_rescore_mapped", ptr(x), N, D, r0, r1, ptr(cand), ptr(cnt), ptr(tau_o), n_lists, cap, pitch, k, eps,
             None, locality, ptr(maps[0]), ptr(maps[1]), ptr(idx), ptr(key), ptr(flag), ptr(max_err), ptr(ws), ptr(count),
             stream_ptr())
    return idx, key, flag, float(max_err)


def exact_topk(E, k):
    """Top-k of exact_ref by (key desc, index asc), numpy: (idx, key)."""
    n, N = E.shape
    order = np.lexsort((np.broadcast_to(np.arange(N), E.shape), -E.astype(np.float64)), axis=1)[:, :k]
    return order.astype(np.int32), np.take_along_axis(E, order, 1)


def kth(v, k):
    return -np.sort(-v, axis=1)[:, k - 1]


class Crafted:
    """A cluster set with a 200-row duplicate block, exact_ref, and a = exact_ref + delta, |delta| <= eps / 2."""

    def __init__(self, N=2048, D=128, seed=3):
        import reid_gan_b200 as rg
        x, _ = rg.synth(N, D, 64, 0.6, seed)
        x[300:500] = x[300]                                   # rows 300..499: one point 200 times
        self.x = x.contiguous().cuda()
        self.E = refs(self.x)[2].cpu().numpy()
        rng = np.random.default_rng(seed)
        self.a = (self.E.astype(np.float64) + rng.uniform(-0.5, 0.5, self.E.shape) * B_EPS).astype(np.float32)
        self.N = N


@pytest.fixture(scope="module")
def crafted():
    return Crafted()


def expect_certified(a, tau, k, eps=B_EPS, margin=1e-5):
    """Rows whose certificate clearly holds: tau below a_(k) - 2 eps with room, window of k..128 members."""
    ak = kth(a, k)
    lo = ak - 2 * eps
    n_w = (a >= lo[:, None] - margin).sum(axis=1)
    n_w_hi = (a >= lo[:, None] + margin).sum(axis=1)
    return (tau < lo - margin) & (n_w <= 128) & (n_w_hi >= k)


@pytest.mark.parametrize("k", [1, 30, 64])
def test_rescore_certified_rows_are_exact_and_refusals_hold(crafted, k):
    """Certificate: on lists that keep the premise (built from exact_ref + delta, |delta| <= eps), a row with flag 0
    holds exactly the top-k of exact_ref -- indices and key bits, (key desc, index asc); rows whose certificate holds
    with room are certified.  Refusals: a threshold at or above a_(k) - 2 eps with a window member unlisted, an
    overflowed list, fewer than k entries, a window of more than 128 members (the 200-row duplicate block), a window
    member whose approximate score is off by 1.5 eps (max_err_out >= that error).  Flagged rows still hold valid
    indices: unfilled positions are the row itself with key -inf."""
    c = crafted
    N, a, E = c.N, c.a, c.E
    L = k + 34
    tau = kth(a, L).astype(np.float32)                        # keep L entries >= tau: every other column scores below
    strict = np.zeros(N, dtype=bool)
    ak = kth(a, k)
    ak1 = kth(a, k + 1)
    normal = np.ones(N, dtype=bool)
    normal[300:500] = False
    # refusal 1: tau = a_(k+1) >= a_(k) - 2 eps, lists {a > tau}: the (k+1)-th is a window member and unlisted
    r_hi = np.flatnonzero(normal & (ak1 >= ak - 2 * B_EPS) & (ak1 < ak))[:8]
    assert r_hi.size >= 3 or k == 1
    tau[r_hi], strict[r_hi] = ak1[r_hi], True
    # ... and tau = a_(k) - eps, lists {a > tau}, whatever lies below
    r_mid = np.setdiff1d(np.flatnonzero(normal), r_hi)[[3, 600, 1200]]
    tau[r_mid], strict[r_mid] = (ak[r_mid] - np.float32(B_EPS)).astype(np.float32), True
    r_hi = np.r_[r_hi, r_mid]
    # refusal 2: fewer than k entries -- tau = a_(k), lists {a > tau}
    r_few = np.flatnonzero(normal)[[5, 77, 1500]]
    tau[r_few], strict[r_few] = ak[r_few], True
    # refusal 3: the duplicate block lists all 200 copies (window > 128)
    tau[300:500] = kth(a[300:500], 230)
    cand, cnt, cap = craft(a, tau, strict, 1)
    # refusal 4: an overflowed list (count above cap: the kernel reads cap entries)
    r_ovf = np.flatnonzero(normal)[[11, 900]]
    cnt_np = cnt.cpu().numpy()
    cnt_np[r_ovf] = cap + 3
    cnt = torch.from_numpy(cnt_np).cuda()
    # refusal 5: one window member's approximate score off by 1.5 eps (the row's best column: a member for every k)
    r_err = int(np.flatnonzero(normal)[42])
    cand_np = cand.cpu().numpy().reshape(N, cap)
    sc = cand_np[r_err].view(np.uint64) >> np.uint64(32)
    cols = (cand_np[r_err].view(np.uint64) & np.uint64(0xFFFFFFFF)).astype(np.int64)
    used = np.arange(cap) < cnt_np[r_err]
    scores = sc.astype(np.uint32).view(np.float32)
    best = np.flatnonzero(used)[np.argmax(scores[used])]
    pushed = np.float32(np.float64(E[r_err, cols[best]]) + 1.5 * B_EPS)
    cand_np[r_err, best] = pack(np.array([pushed]), np.array([cols[best]]))[0]
    cand = torch.from_numpy(cand_np.reshape(-1)).cuda()
    a_used = a.copy()
    a_used[r_err, cols[best]] = pushed

    idx, key, flag, max_err = rescore(c.x, cand, cnt, tau, 1, cap, k)
    idx, key, flag = idx.cpu().numpy(), key.cpu().numpy(), flag.cpu().numpy()
    ie, ke = exact_topk(E, k)
    for name, rr in (("threshold >= a_(k) - 2 eps", r_hi), ("fewer than k", r_few), ("window > 128", np.arange(300, 500)),
                     ("overflowed list", r_ovf), ("error 1.5 eps", np.array([r_err]))):
        assert flag[rr].all(), "%s: rows %s certified" % (name, rr[flag[rr] == 0].tolist())
    assert max_err >= 1.5 * B_EPS * (1 - 1e-3), "max_err_out %r misses the 1.5 eps error" % max_err
    ok = flag == 0
    want = expect_certified(a_used, tau, k) & normal
    want[np.r_[r_hi, r_few, r_ovf, r_err]] = False
    assert want.sum() >= N // 4, "too few rows certify: the test would not test the certificate"
    assert ok[want].all(), "rows whose certificate holds were refused: %s" % np.flatnonzero(want & ~ok)[:10].tolist()
    diff = ok & ((idx != ie).any(axis=1) | (key.view(np.uint32) != ke.view(np.uint32)).any(axis=1))
    if diff.any():
        r = int(np.flatnonzero(diff)[0])
        j = int(np.flatnonzero(idx[r] != ie[r])[0]) if (idx[r] != ie[r]).any() else 0
        xd = c.x.double().cpu().numpy()
        raise AssertionError("certified row %d differs from exact_ref at position %d: kernel (%d, %r) reference (%d, %r); "
                             "fp64 dots %r / %r" % (r, j, idx[r, j], key[r, j], ie[r, j], ke[r, j],
                                                    float(xd[r] @ xd[idx[r, j]]), float(xd[r] @ xd[ie[r, j]])))
    assert ((idx >= 0) & (idx < N)).all(), "flagged rows must still hold valid indices"
    unfilled = np.isneginf(key)
    rows_of = np.broadcast_to(np.arange(N)[:, None], idx.shape)
    assert (idx[unfilled] == rows_of[unfilled]).all(), "unfilled positions hold the row itself"
    if k > 1:
        assert unfilled[r_few, -1].all(), "a row with k - 1 entries leaves its last position unfilled"


def test_rescore_results_do_not_depend_on_layout(crafted):
    """Certificate: the same lists as row-major or list-major, in 1 / 2 / 8 / 64 lists, with and without the locality
    order, as a shard with row_begin > 0, and through reid_knn_rescore_mapped with a random permutation give identical
    indices, key bits and flags; uncertified_count equals the sum of the flags and accumulates across calls."""
    c = crafted
    N, a, k = c.N, c.a, 30
    tau = kth(a, k + 34).astype(np.float32)
    strict = np.zeros(N, dtype=bool)
    cand, cnt, cap = craft(a, tau, strict, 1)
    count = torch.zeros(1, dtype=torch.int64, device=c.x.device)
    i0, k0, f0, _ = rescore(c.x, cand, cnt, tau, 1, cap, k, count=count)
    rescore(c.x, cand, cnt, tau, 1, cap, k, count=count)
    assert int(count) == 2 * int(f0.sum()), "uncertified_count must add the flags of every call"
    assert 0 < int(f0.sum()) < N, "the layout test needs certified and refused rows"

    def same(res, what, rows=slice(None)):
        i, kk, f, _ = res
        assert torch.equal(i, i0[rows]) and torch.equal(kk.view(torch.int32), k0[rows].view(torch.int32)), what
        assert torch.equal(f, f0[rows]), what + ": flags"

    same(rescore(c.x, cand, cnt, tau, 1, cap, k, locality=0), "locality order off")
    for n_lists in (2, 8, 64):
        cd, cn, cp = craft(a, tau, strict, n_lists, seed=n_lists)
        same(rescore(c.x, cd, cn, tau, n_lists, cp, k), "%d row-major lists" % n_lists)
        cd, cn, cp = craft(a, tau, strict, n_lists, list_major=True, seed=n_lists)
        same(rescore(c.x, cd, cn, tau, n_lists, cp, k, pitch=N), "%d list-major lists" % n_lists)
    r0, r1 = 700, 1900
    cd, cn, cp = craft(a[r0:r1], tau[r0:r1], strict[r0:r1], 2)
    same(rescore(c.x, cd, cn, tau[r0:r1], 2, cp, k, r0=r0, r1=r1), "shard [700, 1900)", slice(r0, r1))
    orig_of = np.random.default_rng(5).permutation(N)
    pos_of = np.argsort(orig_of)
    cd, cn, cp = craft(a[orig_of][:, orig_of], tau[orig_of], strict[orig_of], 2)
    maps = (torch.from_numpy(pos_of.astype(np.int32)).cuda(), torch.from_numpy(orig_of.astype(np.int32)).cuda())
    same(rescore(c.x, cd, cn, tau[orig_of], 2, cp, k, maps=maps), "mapped (random permutation)")


@pytest.mark.parametrize("D,offset", [(128, 0), (192, 0), (96, 0), (100, 0), (128, 1)])
def test_rescore_stage2_kernels_match_exact_keys(D, offset):
    """Certificate, stage 2: every exact re-score kernel a release build reaches gives the key bits of reid_knn_exact
    and of exact_ref -- rescore_mma_kernel (16-byte aligned x, D % 64 == 0) and rescore_exact_kernel<0> (D = 96, 100;
    x one float off 16-byte alignment).  rescore_group_kernel and rescore_exact_kernel<16/8/4/2> are reached only in a
    -DREID_DEV build and are not tested here."""
    import reid_gan_b200 as rg
    from reid_gan_b200.faiss_rerank import _knn_exact_rows
    N, k = 1500, 30
    x0, _ = rg.synth(N, D, 50, 0.7, 11)
    buf = torch.zeros(N * D + 4, dtype=torch.float32, device="cuda")
    buf[offset:offset + N * D] = x0.reshape(-1).cuda()
    x = buf[offset:offset + N * D].view(N, D)
    assert (x.data_ptr() % 16 == 0) == (offset == 0)
    E = refs(x)[2].cpu().numpy()
    tau = kth(E, k + 34).astype(np.float32)
    cand, cnt, cap = craft(E, tau, np.zeros(N, dtype=bool), 2)
    idx, key, flag, _ = rescore(x, cand, cnt, tau, 2, cap, k, eps=1e-5)
    ie = torch.empty((N, k), dtype=torch.int32, device="cuda")
    ke = torch.empty((N, k), dtype=torch.float32, device="cuda")
    _knn_exact_rows(x, k, None, 0, N, ie, ke)
    ok = flag == 0
    assert int(ok.sum()) >= N // 2
    assert torch.equal(idx[ok], ie[ok]) and torch.equal(key[ok].view(torch.int32), ke[ok].view(torch.int32)), \
        "re-score and reid_knn_exact disagree"
    ir, kr = exact_topk(E, k)
    okn = ok.cpu().numpy()
    bad = okn & ((idx.cpu().numpy() != ir).any(axis=1) | (key.cpu().numpy().view(np.uint32) != kr.view(np.uint32)).any(axis=1))
    if bad.any():
        r = int(np.flatnonzero(bad)[0])
        raise AssertionError("row %d: kernel %s %s, exact_ref %s %s" % (r, idx[r].tolist(), key[r].tolist(), ir[r].tolist(),
                                                                         kr[r].tolist()))


# ---- C. end to end at the magnitude edges ------------------------------------------------------------------------
@pytest.mark.parametrize("fam,N,D,k", [
    ("big", 1500, 64, 30),
    ("tiny", 1500, 64, 30),
    ("spike", 8192, 256, 30),            # one norm with spikes: metric "auto" takes the inner-product key
    ("spike-mixed", 3000, 256, 30),      # the one-sided kernel; "ip" whatever the norms (get_dist_nbr)
    ("iso", 8191, 128, 30),              # just below SYM_MIN_N: the one-sided kernel
    ("iso", 8193, 128, 64),              # just above: the symmetric search, k = 64
])
def test_knn_search_at_magnitude_edges(fam, N, D, k):
    """End to end: knn_search(x, k, "auto") and knn_search(x, k, "tc", metric="ip") give the lists and key bits of
    knn_search(x, k, "exact", metric=...) and of oracle.rerank.exact_knn (fp64).  The spike sets are the regression
    case of an fp16 overflow: their rows once scored NaN against their cluster mates and were left out of certified
    lists."""
    from reid_gan_b200 import faiss_rerank as fr
    from oracle import rerank as orr
    x = family(fam, N, D)
    xn = x.cpu().numpy()
    oracle = {}
    for mode, metric in (("auto", "auto"), ("tc", "ip")):
        it, kt, info = fr.knn_search(x, k, mode, metric=metric)
        ie, ke, info_e = fr.knn_search(x, k, "exact", metric=metric)
        assert info["metric"] == info_e["metric"], "%s: the key must not depend on the fp16 conversion" % mode
        assert torch.equal(it, ie), "%s/%s: neighbour lists differ from the exact search" % (mode, metric)
        assert torch.equal(kt.view(torch.int32), ke.view(torch.int32)), "%s/%s: keys differ" % (mode, metric)
        m = info_e["metric"]
        if m not in oracle:
            oracle[m] = orr.exact_knn(xn, k, return_keys=True, metric=m)
        io, ko = oracle[m]
        assert np.array_equal(it.cpu().numpy(), io), "%s/%s: lists differ from the fp64 oracle" % (mode, metric)
        assert np.array_equal(kt.cpu().numpy().view(np.uint32), ko.view(np.uint32)), "%s/%s: keys vs oracle" % (mode, metric)
    if fam.startswith("spike"):
        assert float(to_half(x)[1][0]) == math.inf, "an fp16 overflow must make eps infinite"


def test_get_dist_nbr_with_spikes():
    """End to end, infomap front end: get_dist_nbr on a spike set of one norm (the oracle's key is the inner product
    only then) equals oracle.infomap.get_dist_nbr."""
    from reid_gan_b200 import infomap_cluster as ic
    from oracle import infomap as oi
    x = spike_set(3000, 256, 1).numpy()
    d, n = ic.get_dist_nbr(x, k=30)
    d_ref, n_ref = oi.get_dist_nbr(x, k=30)
    assert np.array_equal(n, n_ref) and np.array_equal(d, d_ref)


def test_features_to_half_reports_overflow():
    """Error model: reid_features_to_half, _acc and _gather report max ||x||^2 = +inf exactly when a component
    rounds to +-inf in fp16 (|x| * 16 >= 65520); the minimum stays the true one; below that bound nothing changes."""
    from reid_gan_b200 import knn_tc
    from reid_gan_b200._lib import call, ptr, stream_ptr
    x = torch.full((64, 128), 0.5, device="cuda")
    x[7, 3] = 4094.0                                          # 65504 in fp16: finite
    xh, msq = to_half(x)
    assert torch.isfinite(xh).all() and abs(float(msq[0]) / float((x.double() ** 2).sum(1).max()) - 1) < 1e-6
    x[9, 100] = -4095.0                                       # 65520 rounds to -inf
    xh, msq = to_half(x)
    assert not torch.isfinite(xh).all() and float(msq[0]) == math.inf
    assert float(msq[1]) == float((x.double() ** 2).sum(1).min().float())
    rng = knn_tc.sqnorm_range_of(x, msq)
    assert rng[0] != math.inf and knn_tc.one_norm(rng) is False
    acc = knn_tc.new_sqnorm_range(x.device)
    sp = stream_ptr()
    call("reid_features_to_half_acc", ptr(x[:8]), 8, 128, 4, ptr(xh), ptr(acc), sp)
    assert float(acc[0]) != math.inf
    call("reid_features_to_half_acc", ptr(x[8:]), 56, 128, 4, ptr(xh[8:]), ptr(acc), sp)
    assert float(acc[0]) == math.inf
    src = torch.arange(63, -1, -1, dtype=torch.int32, device="cuda")
    g = knn_tc.new_sqnorm_range(x.device)
    call("reid_features_to_half_gather", ptr(x), ptr(src), 64, 128, 4, ptr(xh), ptr(g), sp)
    assert float(g[0]) == math.inf
