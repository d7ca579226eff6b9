"""GPU: re_ranking_features (evaluation re-ranking from features, no (Q+G)^2 buffer), its farthest-neighbour search,
and the device-resident Evaluator / evaluate_all, against the oracle, the dense re_ranking and stored outputs."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _pdist(a, b):
    """evaluators.py:78-87 on the host (expand + addmm_), like oracle.eval_rerank.synthetic_distances."""
    m, n = a.size(0), b.size(0)
    d = torch.pow(a, 2).sum(dim=1, keepdim=True).expand(m, n) + torch.pow(b, 2).sum(dim=1, keepdim=True).expand(n, m).t()
    d = d.clone()
    d.addmm_(a, b.t(), beta=1, alpha=-2)
    return d


def cluster_features(n_clusters, D, seed, scaled=False, size=22):
    """Tie-free fixture: clusters of `size` rows x_m = (c + a_m u_m) / sqrt(1 + a_m^2) over a private orthonormal set
    {c, u_1..u_size}, with distinct a_m, so every row's nearest size - 1 rows are its cluster mates at well separated
    distances.  scaled: every cluster gets its own norm in [0.7, 1.5]."""
    rng = np.random.default_rng(seed)
    rows = []
    for _ in range(n_clusters):
        basis, _ = np.linalg.qr(rng.standard_normal((D, size + 1)))
        a = 0.3 + 0.3 * (rng.permutation(size) + 0.5 * rng.random(size)) / size
        x = (basis[:, :1].T + a[:, None] * basis[:, 1:].T) / np.sqrt(1 + a * a)[:, None]
        if scaled:
            x = x * rng.uniform(0.7, 1.5)
        rows.append(x)
    x = np.concatenate(rows)[rng.permutation(n_clusters * size)]
    return torch.from_numpy(np.ascontiguousarray(x.astype(np.float32)))


def _dense_colmax(x):
    from reid_gan_b200.evaluation import pairwise_distance_device
    out = []
    for r0 in range(0, x.shape[0], 2048):
        d = pairwise_distance_device(x, x[r0:r0 + 2048])
        out.append((d * d).max(dim=0).values)
    return torch.cat(out)


# (clusters of 22, Q, D, k1, k2, lambda, scaled): the three shapes of test_eval_rerank (k2 = 1 included), one with
# M >= 8192 and D % 64 == 0 (tensor-core kNN and farthest search), one with rows of different norms
SHAPES = [(41, 250, 64, 20, 6, 0.3, False), (23, 120, 32, 7, 1, 0.5, False), (137, 700, 128, 20, 6, 0.3, False),
          (410, 1000, 128, 20, 6, 0.3, False), (70, 300, 64, 20, 6, 0.3, True)]


@pytest.mark.parametrize("nc,Q,D,k1,k2,lam,scaled", SHAPES)
def test_matches_oracle_and_dense_path(nc, Q, D, k1, k2, lam, scaled):
    import reid_gan_b200 as rg
    from oracle import eval_rerank as oe
    from reid_gan_b200.evaluation import pairwise_distance_device
    from reid_gan_b200.rerank import _re_ranking_features
    x = cluster_features(nc, D, 7, scaled)
    q, g = x[:Q], x[Q:]
    ref, parts = oe.re_ranking(_pdist(q, g).numpy(), _pdist(q, q).numpy(), _pdist(g, g).numpy(), k1, k2, lam, return_parts=True)
    srt = np.sort(parts["dist"], axis=1)[:, :k1 + 2]
    assert np.diff(srt, axis=1).min() >= 1e-6, "fixture has a gap below 1e-6 inside the first k1+2 distances"
    out, got = _re_ranking_features(q.cuda(), g.cuda(), k1, k2, lam)
    assert np.array_equal(got["rank"].cpu().numpy(), parts["rank"])
    ep, ei, _ = got["E"]
    assert np.array_equal(ep.cpu().numpy(), parts["E"][0]) and np.array_equal(ei.cpu().numpy(), parts["E"][1])
    out = out.cpu().numpy()
    assert out.dtype == np.float32 and out.shape == (Q, x.shape[0] - Q)
    assert np.abs(out - ref).max() <= 1e-5
    qd, gd = q.cuda(), g.cuda()
    dense = rg.re_ranking(pairwise_distance_device(qd, gd), pairwise_distance_device(qd, qd), pairwise_distance_device(gd, gd),
                          k1=k1, k2=k2, lambda_value=lam)
    assert np.abs(out - dense).max() <= 1e-5
    # host tensors and numpy go through the same path
    assert np.array_equal(rg.re_ranking_features(q, g, k1, k2, lam), out)
    assert np.array_equal(rg.re_ranking_features(q.numpy(), g.numpy(), k1, k2, lam), out)
    if x.shape[0] >= 8192:
        assert got["knn_info"]["mode"].startswith("tc") and got["farthest_info"]["mode"] == "tc"
    if scaled:
        assert got["knn_info"]["metric"] == "l2" and got["farthest_info"]["mode"] == "exact"


def test_colmax_tensor_core_search_is_exact():
    from reid_gan_b200.rerank import farthest_colmax
    from reid_gan_b200 import synth
    x, _ = synth(9000, 128, 300, 0.8, 3)
    x = x.cuda()
    cm, info = farthest_colmax(x)
    assert info["mode"] == "tc"
    ref = _dense_colmax(x)
    assert ((cm - ref).abs() / ref).max().item() <= 2e-6
    cm_exact, info_exact = farthest_colmax(x, mode="exact")
    assert info_exact["mode"] == "exact" and ((cm_exact - ref).abs() / ref).max().item() <= 2e-6


def test_colmax_crowded_window_falls_back_to_the_exact_scan():
    """300 copies of one row u and 60 rows near -u: for those 60 rows the farthest candidates are 300 tied columns, more
    than the lists and the window hold -- they must be reported uncertified and still get the exact column maximum."""
    from reid_gan_b200.rerank import farthest_colmax
    from reid_gan_b200 import synth
    x, _ = synth(8192, 64, 200, 0.8, 4)
    u = x[0].clone()
    x[1:301] = u
    near = -u + 0.05 * torch.randn(60, 64, generator=torch.Generator().manual_seed(5))
    x[301:361] = torch.nn.functional.normalize(near, dim=1)
    x = x.contiguous().cuda()
    cm, info = farthest_colmax(x)
    assert info["mode"] == "tc" and info["uncertified_rows"] >= 60
    ref = _dense_colmax(x)
    assert ((cm - ref).abs() / ref).max().item() <= 2e-6


def test_peak_memory_stays_below_one_square_matrix():
    import reid_gan_b200 as rg
    Q, G, D = 500, 20000, 128
    x, _ = rg.synth(Q + G, D, 700, 0.8, 9)
    q, g = x[:Q].cuda(), x[Q:].cuda()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    out = rg.re_ranking_features(q, g, return_device=True)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    M = Q + G
    assert out.shape == (Q, G)
    assert peak < M * M * 4, "peak %.1f MB" % (peak / 2**20)


class _Model(torch.nn.Module):
    def __init__(self, d_in, d_out):
        super().__init__()
        self.fc = torch.nn.Linear(d_in, d_out, bias=False)
        with torch.no_grad():
            self.fc.weight.copy_(torch.randn(d_out, d_in, generator=torch.Generator().manual_seed(11)) / d_in ** 0.5)

    def forward(self, x):
        return torch.nn.functional.normalize(self.fc(x), dim=1)


def _loader(imgs, names, pids, cams, batch=64):
    return [(imgs[i:i + batch], names[i:i + batch], pids[i:i + batch], cams[i:i + batch], 0)
            for i in range(0, len(names), batch)]


def _eval_fixture(N=1200, Q=200, d_in=48, d_out=64, n_ids=60):
    import reid_gan_b200 as rg
    x, ids = rg.synth(N, d_in, n_ids, 1.0, 21)
    cams = np.random.default_rng(21).integers(0, 6, N)
    names = ["img%05d.jpg" % i for i in range(N)]
    order = np.random.default_rng(22).permutation(N)           # the loader visits the files in another order
    loader = _loader(x[order], [names[i] for i in order], [int(ids[i]) for i in order], [int(cams[i]) for i in order])
    query = [(names[i], int(ids[i]), int(cams[i])) for i in range(Q)]
    gallery = [(names[i], int(ids[i]), int(cams[i])) for i in range(Q, N)]
    return _Model(d_in, d_out).cuda(), loader, query, gallery


def test_evaluator_without_rerank_is_the_composition_of_the_drop_ins(capsys):
    import reid_gan_b200 as rg
    from reid_gan_b200 import evaluation as ev
    model, loader, query, gallery = _eval_fixture()
    cmc_scores, mAP = rg.Evaluator(model).evaluate(loader, query, gallery, cmc_flag=True)
    printed = capsys.readouterr().out
    features, _ = rg.extract_features(model, loader)
    dm, _, _ = ev.pairwise_distance(features, query, gallery)
    args = (dm.numpy(), [p for _, p, _ in query], [p for _, p, _ in gallery], [c for _, _, c in query], [c for _, _, c in gallery])
    ref_map = ev.mean_ap(*args)
    ref_cmc = ev.cmc(*args, separate_camera_set=False, single_gallery_shot=False, first_match_break=True)
    assert abs(mAP - ref_map) <= 1e-12 and np.abs(cmc_scores - ref_cmc).max() <= 1e-12
    expect = ['Mean AP: {:4.1%}'.format(mAP), 'CMC Scores:'] + ['  top-{:<4}{:12.1%}'.format(k, cmc_scores[k - 1]) for k in (1, 5, 10)]
    lines = printed.splitlines()
    assert lines[-5:] == expect
    assert rg.Evaluator(model).evaluate(loader, query, gallery) == pytest.approx(mAP, abs=1e-12)


def test_evaluator_rerank_matches_the_dense_re_ranking(capsys):
    import reid_gan_b200 as rg
    from reid_gan_b200 import evaluation as ev
    model, loader, query, gallery = _eval_fixture()
    cmc_scores, mAP = rg.Evaluator(model).evaluate(loader, query, gallery, cmc_flag=True, rerank=True)
    lines = capsys.readouterr().out.splitlines()
    assert 'Applying person re-ranking ...' in lines
    assert lines[-5] == 'Mean AP: {:4.1%}'.format(mAP)
    features, _ = rg.extract_features(model, loader)
    q = features.matrix([f for f, _, _ in query])
    g = features.matrix([f for f, _, _ in gallery])
    pd = ev.pairwise_distance_device
    dense = rg.re_ranking(pd(q, g), pd(q, q), pd(g, g))
    ids = ([p for _, p, _ in query], [p for _, p, _ in gallery], [c for _, _, c in query], [c for _, _, c in gallery])
    assert abs(mAP - ev.mean_ap(dense, *ids)) <= 1e-4
    assert np.abs(cmc_scores - ev.cmc(dense, *ids, first_match_break=True)).max() <= 1e-4


def test_golden_ranking_through_the_evaluator(capsys):
    import reid_gan_b200 as rg
    from reid_gan_b200.evaluation import pairwise_distance_device
    gz = np.load(os.path.join(GOLD, "ranking_q120_g380.npz"))
    qf, gf = torch.from_numpy(gz["q"]), torch.from_numpy(gz["g"])
    d = pairwise_distance_device(qf.cuda(), gf.cuda())
    stored = gz["distmat"]
    # the device distances order every row like the stored matrix, up to the fp32 rounding of near-equal distances
    along = np.take_along_axis(stored, np.argsort(d.cpu().numpy(), axis=1, kind="stable"), axis=1)
    assert np.diff(along, axis=1).min() >= -1e-5
    Q, G = qf.shape[0], gf.shape[0]
    names = ["q%d" % i for i in range(Q)] + ["g%d" % i for i in range(G)]
    pids = [int(v) for v in gz["q_ids"]] + [int(v) for v in gz["g_ids"]]
    cams = [int(v) for v in gz["q_cams"]] + [int(v) for v in gz["g_cams"]]
    query = [(names[i], pids[i], cams[i]) for i in range(Q)]
    gallery = [(names[Q + i], pids[Q + i], cams[Q + i]) for i in range(G)]
    loader = _loader(torch.cat([qf, gf]), names, pids, cams, batch=100)
    cmc_scores, mAP = rg.Evaluator(torch.nn.Identity()).evaluate(loader, query, gallery, cmc_flag=True)
    ref = gz["cmc_market"]
    assert abs(mAP - float(gz["mAP"])) <= 1e-12, (mAP, float(gz["mAP"]))
    assert np.abs(cmc_scores[:len(ref)] - ref).max() <= 1e-12, np.abs(cmc_scores[:len(ref)] - ref).max()
    cmc2, mAP2 = rg.evaluate_all(None, None, torch.from_numpy(stored).cuda(), query=query, gallery=gallery, cmc_flag=True)
    assert abs(mAP2 - float(gz["mAP"])) <= 1e-12 and np.abs(cmc2[:len(ref)] - ref).max() <= 1e-12
