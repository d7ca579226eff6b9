"""CPU: pin the oracle (oracle/*.py) against the golden vectors produced by the UNMODIFIED
reference (oracle/make_golden.py), and the vectorised flavours against the loop flavours."""
import glob
import os

import numpy as np
import pytest

from oracle import rerank as orr, cluster as ocl, memory as omem

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
RERANK = sorted(glob.glob(os.path.join(GOLD, "rerank_*.npz")))
CM = sorted(glob.glob(os.path.join(GOLD, "cm_*.npz")))


def golden_J(g):
    N = g["x"].shape[0]
    J = np.ones((N, N), dtype=np.float32)
    J[g["J_rows"], g["J_cols"]] = g["J_vals"]
    return J


def test_fixtures_present():
    assert len(RERANK) >= 5 and len(CM) >= 3


@pytest.mark.parametrize("path", RERANK, ids=[os.path.basename(p)[:-4] for p in RERANK])
def test_rerank_oracle_matches_reference(path):
    g = np.load(path)
    x, k1, k2 = g["x"], int(g["k1"]), int(g["k2"])
    J_ref = golden_J(g)
    J = orr.compute_jaccard_distance_oracle(x, k1, k2)
    assert J.dtype == np.float32 and J.shape == J_ref.shape
    # same sparsity structure (integer logic: neighbour lists, reciprocal sets, expansion) ...
    assert np.array_equal(J == 1.0, J_ref == 1.0)
    # ... and values within fp32 summation noise of the reference (bar for the product: 1e-5)
    assert np.abs(J - J_ref).max() <= 2e-6
    assert np.array_equal(J, J.T)
    for eps in g["eps_list"]:
        tag = "eps%02d" % round(float(eps) * 100)
        lab_ref = g["labels_" + tag]
        if not bool(g["admissible_" + tag]):
            continue
        assert np.array_equal(ocl.dbscan_dense(J, float(eps), 4), lab_ref)
        assert np.array_equal(ocl.dbscan_dense(J_ref, float(eps), 4), lab_ref)
        jp, jj, jv = orr.jaccard_sparse(*_vq(x, k1, k2), x.shape[0])
        assert np.array_equal(ocl.dbscan_sparse_J(jp, jj, jv, float(eps), 4), lab_ref)
        if "centroids_" + tag in g.files:
            cen = ocl.cluster_centroids(x, lab_ref)
            np.testing.assert_allclose(cen, g["centroids_" + tag], rtol=1e-5, atol=1e-7)
        break  # one eps exercises the sparse path; the loop above covers the rest cheaply


def _vq(x, k1, k2):
    st = orr.sparse_pipeline(x, k1, k2)
    return st["Vq_ptr"], st["Vq_idx"], st["Vq_val"]


@pytest.mark.parametrize("path", RERANK, ids=[os.path.basename(p)[:-4] for p in RERANK])
def test_dbscan_restatement_all_eps(path):
    g = np.load(path)
    J_ref = golden_J(g)
    for eps in g["eps_list"]:
        tag = "eps%02d" % round(float(eps) * 100)
        assert np.array_equal(ocl.dbscan_dense(J_ref, float(eps), 4), g["labels_" + tag])


def test_loop_and_vectorised_flavours_agree():
    rng = np.random.default_rng(5)
    c = rng.standard_normal((12, 32)).astype(np.float32)
    x = c[rng.integers(0, 12, 300)] + 0.5 * rng.standard_normal((300, 32)).astype(np.float32)
    x /= np.linalg.norm(x, axis=1, keepdims=True)
    for k1, k2 in ((10, 3), (15, 6), (7, 1)):
        rank = orr.exact_knn(x, k1)
        R = orr.reciprocal_lists(rank, k1)
        Rh = orr.reciprocal_lists(rank, orr.half_k(k1))
        # faiss_rerank.py:23-27 restated literally
        for i in (0, 17, 299):
            fwd = rank[i, :k1 + 1]
            bwd = rank[fwd, :k1 + 1]
            assert np.array_equal(R[i], fwd[np.where(bwd == i)[0]])
        E = orr.expand_loops(R, Rh)
        ep, ei = orr.expand(rank, k1)
        for i in range(300):
            assert np.array_equal(E[i], ei[ep[i]:ep[i + 1]])
        st = orr.sparse_pipeline(x, k1, k2, rank=rank)
        N = 300
        Vq = np.zeros((N, N), np.float32)
        rows = np.repeat(np.arange(N), np.diff(st["Vq_ptr"]))
        Vq[rows, st["Vq_idx"]] = st["Vq_val"]
        np.testing.assert_allclose(Vq.sum(1), 1.0, atol=1e-5)
        Jd = orr.jaccard_dense_loops(Vq)
        jp, jj, jv = orr.jaccard_sparse(st["Vq_ptr"], st["Vq_idx"], st["Vq_val"], N)
        assert np.array_equal(orr.jaccard_dense_from_sparse(jp, jj, jv, N), Jd)   # bit-exact: same add order


def test_exact_knn_ties_and_duplicates():
    rng = np.random.default_rng(0)
    x = rng.standard_normal((64, 16)).astype(np.float32)
    x /= np.linalg.norm(x, axis=1, keepdims=True)
    x[10] = x[3]
    x[40] = x[3]
    idx, key = orr.exact_knn(x, 5, return_keys=True)
    assert list(idx[40][:3]) == [3, 10, 40]          # equal keys -> ascending index
    assert np.all(np.diff(key, axis=1) <= 0)
    sub = orr.exact_knn(x, 5, rows=[40, 3])
    assert np.array_equal(sub[0], idx[40]) and np.array_equal(sub[1], idx[3])


def test_half_k_is_round_half_to_even():
    assert [orr.half_k(k) for k in (15, 20, 25, 30, 5, 7)] == [8, 10, 12, 15, 2, 4]


@pytest.mark.parametrize("path", CM, ids=[os.path.basename(p)[:-4] for p in CM])
def test_cluster_memory_oracle_matches_reference(path):
    g = np.load(path)
    temp, mom = float(g["temp"]), float(g["momentum"])
    loss, z, xhat, nrm = omem.cm_forward(g["inputs"], g["targets"], g["features"], temp)
    np.testing.assert_allclose(loss, g["loss_cm"], rtol=1e-4, atol=1e-6)
    np.testing.assert_allclose(loss, g["loss_hard"], rtol=1e-4, atol=1e-6)
    gx = omem.cm_backward(g["grad_loss"], z, g["targets"], g["features"], xhat, nrm, temp)
    np.testing.assert_allclose(gx, g["grad_cm"], rtol=1e-4, atol=1e-6)
    np.testing.assert_allclose(omem.cm_update(g["features"], xhat, g["targets"], mom), g["features_after_cm"],
                               rtol=1e-4, atol=1e-6)
    f_hard, _ = omem.cm_hard_update(g["features"], xhat, g["targets"], mom)
    np.testing.assert_allclose(f_hard, g["features_after_hard"], rtol=1e-4, atol=1e-6)


# ---- golden vectors of the "next" rows (generated by oracle/make_golden.py from the unmodified reference) ----
def _gold(name):
    return np.load(os.path.join(GOLD, name))


def _links_from_gold(g, tag):
    return ({(int(a), int(b)): float(w) for (a, b), w in zip(g["links_ij_" + tag], g["links_w_" + tag])},
            [int(v) for v in g["single_" + tag]])


def test_golden_infomap_front_end():
    from oracle import infomap as oi
    g = _gold("infomap_n400_k15.npz")
    d, n = oi.get_dist_nbr(g["x"], int(g["k"]))
    assert d.dtype == g["dists"].dtype and n.dtype == g["nbrs"].dtype
    assert np.array_equal(n, g["nbrs"]) and np.array_equal(d, g["dists"])
    for min_sim, tag in ((0.3, "ms30"), (0.5, "ms50")):
        links_ref, single_ref = _links_from_gold(g, tag)
        single, links = oi.get_links(n, d, min_sim)
        assert links == links_ref and single == single_ref


def test_golden_eval_rerank():
    from oracle import eval_rerank as oe
    g = _gold("evalrerank_q100_g260.npz")
    for k1, k2 in ((20, 6), (7, 1)):
        ref = g["final_k%d_%d" % (k1, k2)]
        got = oe.re_ranking(g["q_g"], g["q_q"], g["g_g"], k1, k2, float(g["lambda_k%d_%d" % (k1, k2)]))
        assert got.dtype == ref.dtype and np.abs(got - ref).max() <= 1e-6


def test_golden_ranking_metrics():
    from oracle import ranking as orank
    g = _gold("ranking_q120_g380.npz")
    assert np.abs(orank.pairwise_distance(g["q"], g["g"]) - g["distmat"]).max() <= 2e-6
    args = (g["distmat"], g["q_ids"], g["g_ids"], g["q_cams"], g["g_cams"])
    assert abs(orank.mean_ap(*args) - float(g["mAP"])) <= 1e-12
    assert np.abs(orank.cmc(*args, topk=50, first_match_break=True) - g["cmc_market"]).max() <= 1e-12
    assert np.abs(orank.cmc(*args, topk=50) - g["cmc_allshots"]).max() <= 1e-12
    assert np.abs(orank.cmc(*args, topk=50, separate_camera_set=True, first_match_break=True) - g["cmc_sepcam"]).max() <= 1e-12


HALF = sorted(glob.glob(os.path.join(GOLD, "halfrerank_*.npz")))
HALF_ATOL = 2e-3          # a few float16 ulps: one V entry rounded the other way moves a sum by an ulp


@pytest.mark.parametrize("path", HALF, ids=[os.path.basename(p)[:-4] for p in HALF])
def test_oracle_use_float16_against_reference(path):
    """use_float16=True (faiss_rerank.py:37,82-83,102-104): the oracle's float16 restatement against the unmodified
    reference's float16 matrix.  The fp32 softmax feeding V differs in the last bit between implementations, so a
    handful of float16 roundings fall the other way: identical sparsity, >= 99.9 % identical entries, the rest within
    a few float16 ulps."""
    from oracle import rerank as orr
    g = np.load(path)
    x, k1, k2 = g["x"], int(g["k1"]), int(g["k2"])
    N = x.shape[0]
    J_ref = np.ones((N, N), dtype=np.float16)
    J_ref[g["J_rows"], g["J_cols"]] = g["J_vals"]
    J = orr.compute_jaccard_distance_oracle(x, k1, k2, use_float16=True)
    assert J.dtype == np.float16
    assert np.array_equal(J == 1.0, J_ref == 1.0)
    assert (J != J_ref).mean() <= 1e-3
    assert np.abs(J.astype(np.float32) - J_ref.astype(np.float32)).max() <= HALF_ATOL
