"""GPU (-m gpu): the provisional threshold tau' of the sample-first symmetric search (knn_tc._candidates_sym_sf).

The rows outside the threshold sample are scored against it by the symmetric kernel with tau[j] = tau' (the smallest
sample-row threshold); reid_knn_list_tau then raises tau[j] to the r-th best of row j's listed sample scores, or leaves
tau' when fewer than r are listed.  Whatever tau' is, the neighbour lists must be those of the exact search: a tau'
that is too low overflows lists (those rows are un-certified and redone), one that is too high leaves rows with short
lists (the same)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

K = 30


def float_ord(f):
    """common.cuh float_ord, numpy: float32 -> order-preserving uint32."""
    b = np.ascontiguousarray(f, dtype=np.float32).view(np.uint32)
    return np.where(b & 0x80000000, ~b, b | 0x80000000).astype(np.uint32)


def ord_float(o):
    """common.cuh ord_float, numpy: a threshold image back to float32."""
    o = np.asarray(o, dtype=np.uint32)
    return np.where(o & 0x80000000, o & 0x7FFFFFFF, ~o).astype(np.uint32).view(np.float32)


def search_sf(x, k=K):
    """_candidates_sym_sf on x: (list scores, list columns, counts, thresholds as uint32 images, m) on the host."""
    from reid_gan_b200 import knn_tc
    from reid_gan_b200._lib import stream_ptr
    N, D = x.shape
    msq = torch.zeros(2, dtype=torch.float32, device=x.device)
    cand, cnt, tau_o, cap, info, _, _ = knn_tc._candidates_sym_sf(x, N, D, stream_ptr(), x.device, k, msq)
    assert info["layout"] == "sample-first"
    c = cand.view(N, cap).cpu().numpy().view(np.uint64)
    sc = (c >> np.uint64(32)).astype(np.uint32).view(np.float32)
    col = (c & np.uint64(0xFFFFFFFF)).astype(np.int64)
    return sc, col, cnt.cpu().numpy(), tau_o.cpu().numpy().view(np.uint32), knn_tc.sample_size(N, k)


def check_list_tau(sc, col, cnt, tau_o, m, r, floor):
    """The threshold rule of every row outside the sample whose list did not overflow: its sample entries (columns
    < m) all score above tau', and its threshold is max(tau', r-th best of them rounded down to 16 bits) when at least
    r are listed, else tau'.  Returns the number of rows that kept tau'."""
    N, cap = sc.shape
    kept = 0
    for j in range(m, N):
        if cnt[j] > cap:
            continue
        s = sc[j, :cnt[j]][col[j, :cnt[j]] < m]
        o = float_ord(s)
        assert (o > floor).all(), "row %d lists a sample score at or below tau'" % j
        if o.size >= r:
            want = max(int(floor), int(np.sort(o)[::-1][r - 1]) & 0xFFFF0000)
        else:
            want = int(floor)
        assert int(tau_o[j]) == want, "row %d: threshold %#x, rule gives %#x (%d sample entries)" % (j, tau_o[j], want, o.size)
        kept += int(tau_o[j]) == int(floor)
    return kept


def assert_exact(x, k=K):
    """knn_search(x, k, "tc") gives the lists and key bits of the exact search; returns its info."""
    from reid_gan_b200 import faiss_rerank as fr
    it, kt, info = fr.knn_search(x, k, "tc")
    ie, ke, _ = fr.knn_search(x, k, "exact")
    assert torch.equal(it, ie), "neighbour lists differ from the exact search"
    assert torch.equal(kt.view(torch.int32), ke.view(torch.int32)), "keys differ from the exact search"
    return info


def forced_floor(value):
    """A stand-in for knn_tc._tau_floor that writes tau' = value."""
    o = int(float_ord(np.float32(value)).view(np.int32)[0])

    def f(tau, tau_ord, m, N, sp):
        tau[m:] = float(value)
        tau_ord[m:] = o
    return f


def planted_set(N, D, n_planted, seed):
    """Unit rows of clusters in the dimensions [8, D), plus n_planted rows outside the threshold sample that live in
    the dimensions [0, 8) only (a tight cluster of their own): they score exactly 0 against every other row, so no
    sample score of theirs is above tau' > 0."""
    import reid_gan_b200 as rg
    from reid_gan_b200 import knn_tc
    x, _ = rg.synth(N, D, max(1, N // 31), 0.8, seed)
    x[:, :8] = 0.0
    g = torch.Generator().manual_seed(seed + 1)
    m = knn_tc.sample_size(N, K)
    others = knn_tc._sample_first_maps(N, m, "cpu")[1][m:].long()
    planted = others[torch.randperm(others.numel(), generator=g)[:n_planted]]
    c = torch.randn(8, generator=g)
    p = torch.zeros(n_planted, D)
    p[:, :8] = c + 0.3 * torch.randn(n_planted, 8, generator=g)
    x[planted] = p
    return F.normalize(x, dim=1).contiguous().cuda(), planted


def test_rows_without_sample_scores_keep_tau_floor():
    """Rows with fewer than r sample scores above tau' keep tau' as their threshold, and the search still returns the
    exact lists for them and for every other row."""
    from reid_gan_b200 import knn_tc
    N, D = 9000, 128
    x, planted = planted_set(N, D, 48, 3)
    sc, col, cnt, tau_o, m = search_sf(x)
    floor = tau_o[:m].min()
    assert ord_float(floor) > 0, "the construction needs tau' > 0"
    pos_of = knn_tc._sample_first_maps(N, m, "cpu")[0].numpy()
    assert (pos_of[planted.numpy()] >= m).all()
    assert (tau_o[pos_of[planted.numpy()]] == floor).all(), "planted rows must keep tau'"
    kept = check_list_tau(sc, col, cnt, tau_o, m, knn_tc.sym_rank(K), floor)
    assert kept >= planted.numel()
    assert_exact(x)


def test_tau_floor_far_too_low(monkeypatch):
    """tau' below every score: each row outside the sample lists all m = 1024 sample columns, its list overflows in the
    symmetric pass, and the row is un-certified and searched exactly.  The sample rows are unaffected."""
    from reid_gan_b200 import knn_tc
    import reid_gan_b200 as rg
    N, D = 8192, 128
    m = knn_tc.sample_size(N, K)
    assert m == knn_tc.SYM_CAP
    x = rg.synth(N, D, N // 31, 0.8, 4)[0].cuda()
    monkeypatch.setattr(knn_tc, "_tau_floor", forced_floor(-1e30))
    info = assert_exact(x)
    assert info["uncertified_rows"] == N - m
    cnt = info["cand_cnt"]
    assert bool((cnt[m:] > knn_tc.SYM_CAP).all()) and bool((cnt[:m] <= knn_tc.SYM_CAP).all())


def test_tau_floor_too_high(monkeypatch):
    """tau' at the median threshold the rows outside the sample get by default: about half of them list fewer than r
    sample scores and keep tau'; the lists are still those of the exact search."""
    from reid_gan_b200 import knn_tc
    import reid_gan_b200 as rg
    N, D = 12345, 128
    x = rg.synth(N, D, N // 31, 0.8, 5)[0].cuda()
    _, _, _, tau_o, m = search_sf(x)
    hi_f = float(ord_float(np.median(tau_o[m:]))[()])
    monkeypatch.setattr(knn_tc, "_tau_floor", forced_floor(hi_f))
    sc, col, cnt, tau_o, m = search_sf(x)
    floor = float_ord(np.float32(hi_f))[0]
    kept = check_list_tau(sc, col, cnt, tau_o, m, knn_tc.sym_rank(K), floor)
    assert (N - m) // 4 <= kept < N - m, "%d of %d rows kept tau'" % (kept, N - m)
    assert_exact(x)
    monkeypatch.setattr(knn_tc, "_tau_floor", forced_floor(1e30))   # above every score: these rows list nothing
    info = assert_exact(x)
    assert info["uncertified_rows"] == N - m


@pytest.mark.parametrize("N", [8191, 8193, 12345])
def test_sample_first_edges(N):
    """Just below the symmetric search (8191: the one-sided kernel), just above it (8193: one row in the last block)
    and a size whose last block is partly filled: exact lists, nothing un-certified; where the sample-first layout
    runs, every row outside the sample follows the threshold rule and lists every sample column whose fp16 score is
    clearly above tau'."""
    from reid_gan_b200 import knn_tc
    import reid_gan_b200 as rg
    D = 128
    x = rg.synth(N, D, max(1, N // 31), 0.8, 6)[0].cuda()
    info = assert_exact(x)
    assert info["uncertified_rows"] == 0
    if N < knn_tc.SYM_MIN_N:
        assert info["mode"] == "tc"
        return
    assert info["sym"]["layout"] == "sample-first"
    sc, col, cnt, tau_o, m = search_sf(x)
    floor = tau_o[:m].min()
    check_list_tau(sc, col, cnt, tau_o, m, knn_tc.sym_rank(K), floor)
    # completeness of the sample block column in the column direction, against float64 dots of the fp16 operand
    orig_of = knn_tc._sample_first_maps(N, m, x.device)[1].long()
    xh = (x[orig_of] * 16.0).half().double()
    a = ((xh[m:] @ xh[:m].T) * 2.0 ** -8).cpu().numpy()
    slack = D * 2.0 ** -23 * ((xh[m:].abs() @ xh[:m].abs().T) * 2.0 ** -8).cpu().numpy()
    t = np.float64(ord_float(floor))
    listed = np.zeros((N - m, m), dtype=bool)
    for j in range(m, N):
        c = col[j, :cnt[j]]
        listed[j - m, c[c < m]] = True
    assert not (~listed & (a > t + slack)).any(), "a sample score clearly above tau' is missing from a list"
