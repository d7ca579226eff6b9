"""GPU (-m gpu): DistributedEvaluator's stages against the single-process Evaluator, byte for byte.

One device: W "virtual ranks".  reid_peer_scatter_rows only STORES to the addresses in peer_base, so W plain device
buffers stand in for the W ranks' (M, D) matrices; every rank extracts its eval_shard share through the model and
scatters it in turn, then every rank's stages run on its own buffer.  Compared with Evaluator.evaluate /
_re_ranking_features on the same features: every rank's x, the concatenated (Q_r, G) distance blocks, colmax and the
neighbour lists, the concatenated re-ranked rows, and mAP / CMC with and without re-ranking.  Processes: two gloo ranks
sharing cuda:0 run the collective fallback through DistributedEvaluator; two NCCL ranks run both exchanges when the
box has two devices."""
import os
import socket

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


class _Model(torch.nn.Module):
    """A fixed, seeded backbone stand-in: linear + L2 normalisation."""

    def __init__(self, d_in, d_out, seed=11):
        super().__init__()
        self.fc = torch.nn.Linear(d_in, d_out, bias=False)
        with torch.no_grad():
            self.fc.weight.copy_(torch.randn(d_out, d_in, generator=torch.Generator().manual_seed(seed)) / d_in ** 0.5)

    def forward(self, x):
        return torch.nn.functional.normalize(self.fc(x), dim=1)


class _Scale(torch.nn.Module):
    """Rows of different norms: the L2-key neighbour search and the exact farthest-row scan."""

    def forward(self, x):
        return x * (0.7 + 0.8 * (x[:, :1].abs() * 1000 % 1))


def _loader(items, imgs_of, batch=1):
    """List loader over (fname, pid, cam) items, in the order given.  One image per batch by default: the backbone's
    GEMM may pick another kernel for another batch size (the rank shares end in batches of other sizes than the
    single-process loader), which changes the last bits of a feature row before any code under test runs."""
    out = []
    for i in range(0, len(items), batch):
        chunk = items[i:i + batch]
        out.append((torch.stack([imgs_of[f] for f, _, _ in chunk]), [f for f, _, _ in chunk], [p for _, p, _ in chunk],
                    [c for _, _, c in chunk], 0))
    return out


def _case_ranking():
    gz = np.load(os.path.join(GOLD, "ranking_q120_g380.npz"))
    feats = np.concatenate([gz["q"], gz["g"]])
    pids = np.concatenate([gz["q_ids"], gz["g_ids"]])
    cams = np.concatenate([gz["q_cams"], gz["g_cams"]])
    Q = gz["q"].shape[0]
    names = ["q%04d" % i for i in range(Q)] + ["g%04d" % i for i in range(feats.shape[0] - Q)]
    return torch.nn.Identity(), feats, names, pids, cams, Q, gz


def _case_evalrerank():
    """Features recovered from the stored distance matrices (classical MDS: they are squared distances of rank-64
    features), ids and cameras seeded."""
    gz = np.load(os.path.join(GOLD, "evalrerank_q100_g260.npz"))
    D2 = np.block([[gz["q_q"], gz["q_g"]], [gz["q_g"].T, gz["g_g"]]]).astype(np.float64)
    M = D2.shape[0]
    J = np.eye(M) - 1.0 / M
    w, v = np.linalg.eigh(-0.5 * J @ D2 @ J)
    top = np.argsort(w)[::-1][:64]
    feats = (v[:, top] * np.sqrt(np.maximum(w[top], 0))).astype(np.float32)
    rng = np.random.default_rng(3)
    names = ["x%04d" % i for i in range(M)]
    return torch.nn.Identity(), feats, names, rng.integers(0, 25, M), rng.integers(0, 4, M), 100, gz


def _case_synth(M, Q, d_in, d_out, n_ids, seed, model=None):
    import reid_gan_b200 as rg
    x, ids = rg.synth(M, d_in, n_ids, 1.0, seed)
    cams = np.random.default_rng(seed).integers(0, 6, M)
    names = ["s%06d.jpg" % i for i in range(M)]
    perm = np.random.default_rng(seed + 1).permutation(M)         # names are not in query/gallery order
    names = [names[i] for i in perm]
    return model or _Model(d_in, d_out), x.numpy(), names, ids.numpy(), cams, Q, None


def _lists(feats, names, pids, cams, Q, both=0):
    """query / gallery items and the image of every file; `both` query names are also gallery items."""
    items = [(names[i], int(pids[i]), int(cams[i])) for i in range(len(names))]
    query, gallery = items[:Q], items[Q:]
    if both:
        gallery = gallery + query[:both]
    imgs = {names[i]: torch.from_numpy(np.ascontiguousarray(feats[i])) for i in range(len(names))}
    return query, gallery, imgs


def _bytes_equal(a, b):
    return a.shape == b.shape and a.dtype == b.dtype and torch.equal(a.contiguous().view(torch.uint8),
                                                                     b.contiguous().view(torch.uint8))


def _reference(model, query, gallery, imgs, rerank_parts, batch=1):
    import reid_gan_b200 as rg
    from reid_gan_b200.evaluation import pairwise_distance_device
    from reid_gan_b200.rerank import _re_ranking_features
    loader = _loader(sorted(query + gallery, key=lambda it: it[0])[::-1], imgs, batch)
    ev = rg.Evaluator(model)
    plain = ev.evaluate(loader, query, gallery, cmc_flag=True)
    rr = ev.evaluate(loader, query, gallery, cmc_flag=True, rerank=True)
    mAP_only = ev.evaluate(loader, query, gallery)
    features, _ = rg.extract_features(model, loader)
    q = features.matrix([f for f, _, _ in query])
    g = features.matrix([f for f, _, _ in gallery])
    ref = dict(plain=plain, rerank=rr, mAP=mAP_only, x=torch.cat([q, g]), qg=pairwise_distance_device(q, g))
    if rerank_parts:
        out, parts = _re_ranking_features(q, g, q_g_dist=ref["qg"])
        ref.update(out=out, colmax=parts["colmax"], rank=parts["rank"], knn_mode=parts["knn_info"]["mode"],
                   metric=parts["knn_info"]["metric"], far_mode=parts["farthest_info"]["mode"])
    return ref


def _virtual_ranks(model, query, gallery, imgs, W, batch=1):
    """Every stage of DistributedEvaluator for W ranks on one device, the exchanges replaced by W local buffers."""
    import reid_gan_b200 as rg
    from reid_gan_b200 import eval_dist as ed
    from reid_gan_b200._lib import call, ptr
    from reid_gan_b200.evaluation import pairwise_distance_device
    from reid_gan_b200.rerank import _check_k, _rr_blend, _rr_sparse
    from reid_gan_b200.sharded import partition
    Q, G = len(query), len(gallery)
    M = Q + G
    qpos, gpos = ed._positions(query, gallery)
    bufs, D = None, None
    bad = torch.zeros(1, dtype=torch.int64, device="cuda")
    for r in range(W):
        share = rg.eval_shard(query, gallery, world=W, rank=r)
        features, _ = rg.extract_features(model, _loader(share[::-1], imgs, batch))
        names = list(features.keys())
        if bufs is None:
            D = features._buf.shape[1]
            bufs = [torch.full((M, D), float("nan"), device="cuda") for _ in range(W)]
            base = torch.tensor([b.data_ptr() for b in bufs], dtype=torch.int64, device="cuda")
        table = ed.dst_table(names, qpos, gpos, "cuda")
        call("reid_peer_scatter_rows", ptr(features._buf), len(names), D, ptr(table), M, W, ptr(base), 0, ptr(bad), None)
    torch.cuda.synchronize()
    assert int(bad) == 0
    ids = ed.device_ids(query, gallery, "cuda")
    Bq = -(-Q // W)
    res = dict(x=bufs, qg=[], rows=[], rows_rr=[], colmax=[], rank=[], out=[])
    cols = _check_k(20, 6, M)
    blocks = []
    for r in range(W):
        x = bufs[r]
        q0, q1 = partition(Q, W, r)
        qg = pairwise_distance_device(x[q0:q1], x[Q:]) if q1 > q0 else None
        blocks.append((q0, q1, qg))
        if qg is not None:
            res["qg"].append(qg)
        res["rows"].append(ed.block_metrics(qg, q0, ids, ed.CMC_TOPK, Bq)[:q1 - q0])
        sqnorm = torch.empty(M, dtype=torch.float64, device="cuda")
        call("reid_rr_row_sqnorm64", ptr(x), M, D, ptr(sqnorm), None)
        r0, r1 = partition(M, W, r)
        c, k = ed.rerank_rows(x, sqnorm, cols, r0, r1)
        res["colmax"].append(c)
        res["rank"].append(k)
    colmax, rank = torch.cat(res["colmax"]), torch.cat(res["rank"])
    for r in range(W):
        x = bufs[r]
        q0, q1, qg = blocks[r]
        sqnorm = torch.empty(M, dtype=torch.float64, device="cuda")
        call("reid_rr_row_sqnorm64", ptr(x), M, D, ptr(sqnorm), None)
        out = _rr_blend(x, _rr_sparse(x, sqnorm, colmax, rank, 20, 6), colmax, Q, 0.3, qg, q0, q1) if q1 > q0 else None
        if out is not None:
            res["out"].append(out)
        res["rows_rr"].append(ed.block_metrics(out, q0, ids, ed.CMC_TOPK, Bq)[:q1 - q0])
    res["plain"] = ed.metrics_from_rows(torch.cat(res["rows"]), ed.CMC_TOPK)
    res["rerank"] = ed.metrics_from_rows(torch.cat(res["rows_rr"]), ed.CMC_TOPK)
    res["mAP"] = ed.metrics_from_rows(torch.cat(res["rows"])[:, :2].contiguous(), 0)[0]
    res["colmax"], res["rank"] = colmax, rank
    return res


def _check(model, feats, names, pids, cams, Q, W_list=(2, 4, 8), both=0, batch=1):
    model = model.cuda()
    query, gallery, imgs = _lists(feats, names, pids, cams, Q, both)
    ref = _reference(model, query, gallery, imgs, True, batch)
    for W in W_list:
        got = _virtual_ranks(model, query, gallery, imgs, W, batch)
        for r, x in enumerate(got["x"]):
            assert _bytes_equal(x, ref["x"]), "W=%d: rank %d's x differs" % (W, r)
        assert _bytes_equal(torch.cat(got["qg"]), ref["qg"]), "W=%d: distance blocks" % W
        assert _bytes_equal(got["colmax"], ref["colmax"]), "W=%d: colmax" % W
        assert _bytes_equal(got["rank"], ref["rank"]), "W=%d: neighbour lists" % W
        assert _bytes_equal(torch.cat(got["out"]), ref["out"]), "W=%d: re-ranked rows" % W
        for key in ("plain", "rerank"):
            (cmc_ref, map_ref), (map_got, cmc_got) = ref[key], got[key]
            assert map_got == map_ref and np.array_equal(cmc_got, cmc_ref), (W, key, map_got, map_ref)
        assert got["mAP"] == ref["mAP"]
    return ref


def test_golden_ranking_set():
    model, feats, names, pids, cams, Q, gz = _case_ranking()
    ref = _check(model, feats, names, pids, cams, Q, batch=64)           # Identity: any batch gives the same rows
    cmc_scores, mAP = ref["plain"]
    assert abs(mAP - float(gz["mAP"])) <= 1e-12                      # the existing bar against the reference
    assert np.abs(cmc_scores[:50] - gz["cmc_market"]).max() <= 1e-12


def test_golden_eval_rerank_set():
    model, feats, names, pids, cams, Q, gz = _case_evalrerank()
    ref = _check(model, feats, names, pids, cams, Q, batch=64)
    # the recovered features reproduce the stored re-ranking (test_golden_eval_rerank_cuda's bar is 1e-5 on the
    # stored distances; the features add the fp32 rounding of the reconstruction)
    assert np.abs(ref["out"].cpu().numpy() - gz["final_k20_6"]).max() <= 1e-4


def test_large_set_uses_the_tensor_core_searches():
    """M = 9000 >= 8192, D = 128: tensor-core kNN and farthest-row search; Q = 1001 is not divisible by 2, 4 or 8."""
    ref = _check(*_case_synth(9000, 1001, 96, 128, 300, 5)[:6])
    assert ref["knn_mode"].startswith("tc") and ref["far_mode"] == "tc" and ref["metric"] == "ip"


def test_rows_of_different_norms_use_the_l2_key():
    model = torch.nn.Sequential(_Model(48, 64, seed=4), _Scale())
    ref = _check(*_case_synth(1300, 203, 48, 64, 60, 8, model=model)[:6])
    assert ref["metric"] == "l2" and ref["far_mode"] == "exact"


def test_file_in_both_lists_and_uneven_split():
    """Three query images are gallery items too: their rows are written twice; Q = 77 over 2, 4, 8 ranks."""
    ref = _check(*_case_synth(700, 77, 40, 64, 40, 9)[:6], both=3)
    assert ref["x"].shape[0] == 700 + 3


def test_scatter_guard_counts_and_skips_out_of_range_rows():
    from reid_gan_b200._lib import call, ptr
    src = torch.arange(3 * 8, dtype=torch.float32, device="cuda").view(3, 8)
    dst = torch.tensor([[0, 5], [-1, 2], [9, -1]], dtype=torch.int32, device="cuda")       # 5 and 9 are >= M = 4
    bufs = [torch.full((4, 8), -1.0, device="cuda") for _ in range(2)]
    base = torch.tensor([b.data_ptr() for b in bufs], dtype=torch.int64, device="cuda")
    bad = torch.zeros(1, dtype=torch.int64, device="cuda")
    call("reid_peer_scatter_rows", ptr(src), 3, 8, ptr(dst), 4, 2, ptr(base), 0, ptr(bad), None)
    torch.cuda.synchronize()
    assert int(bad) == 2
    for b in bufs:
        assert torch.equal(b[0], src[0]) and torch.equal(b[2], src[1])
        assert (b[1] == -1).all() and (b[3] == -1).all()


# ---- processes -----------------------------------------------------------------------------------------------------

def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, result_dir, peer, backend):
    import datetime
    import sys
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    dev = torch.device("cuda", rank if backend == "nccl" else 0)
    torch.cuda.set_device(dev)
    kw = dict(device_id=dev) if backend == "nccl" else {}
    dist.init_process_group(backend, rank=rank, world_size=world, timeout=datetime.timedelta(seconds=300), **kw)
    import reid_gan_b200 as rg
    from reid_gan_b200 import sharded
    sharded.PEER_EXCHANGE = peer
    model, feats, names, pids, cams, Q, _ = _case_synth(1500, 301, 48, 64, 60, 12)
    model = model.to(dev)
    query, gallery, imgs = _lists(feats, names, pids, cams, Q, both=2)
    ref = _reference(model, query, gallery, imgs, False)
    ev = rg.DistributedEvaluator(model)
    log = []
    for step in range(2):                                       # the second evaluation reuses the cached buffers
        loader = _loader(rg.eval_shard(query, gallery)[::-1], imgs)
        plain = ev.evaluate(loader, query, gallery, cmc_flag=True)
        rr = ev.evaluate(loader, query, gallery, cmc_flag=True, rerank=True)
        m = ev.evaluate(loader, query, gallery)
        ok = (plain[1] == ref["plain"][1] and np.array_equal(plain[0], ref["plain"][0]) and rr[1] == ref["rerank"][1]
              and np.array_equal(rr[0], ref["rerank"][0]) and m == ref["mAP"])
        log.append("step=%d ok=%s" % (step, ok))
    bad_loader = _loader(rg.eval_shard(query, gallery)[1:], imgs)           # every rank misses one file
    try:
        ev.evaluate(bad_loader, query, gallery)
        log.append("mismatch ok=False")
    except ValueError:
        log.append("mismatch ok=True")
    torch.cuda.synchronize()
    dist.barrier()
    open(os.path.join(result_dir, "r%d.txt" % rank), "w").write("\n".join(log))
    os._exit(0)                      # without tearing down the peer mappings one by one (as scripts/dist_check.py)


def _spawn(tmp_path, peer, backend):
    import torch.multiprocessing as mp
    mp.spawn(_worker, args=(2, _free_port(), str(tmp_path), peer, backend), nprocs=2, join=True)
    for r in range(2):
        log = (tmp_path / ("r%d.txt" % r)).read_text().splitlines()
        assert len(log) == 3
        bad = [line for line in log if not line.endswith("ok=True")]
        assert not bad, "rank %d: %s" % (r, bad)


def test_two_ranks_on_one_device_gloo(tmp_path):
    """DistributedEvaluator with the collective fallback: two gloo ranks share cuda:0."""
    _spawn(tmp_path, False, "gloo")


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
@pytest.mark.parametrize("peer", [True, False], ids=["peer-stores", "nccl"])
def test_two_devices(peer, tmp_path):
    _spawn(tmp_path, peer, "nccl")
