"""Check of DistributedEvaluator at MSMT17's test shape (Q = 11,659, G = 82,161, D = 2048; synthetic features, seeded):
every rank's mAP / CMC, with and without re-ranking, and a sha256 of the gathered re-ranked (Q, G) matrix must equal
the single-process Evaluator's; the stages are timed with CUDA events (max over ranks).  One JSON line per run.

    python -m torch.distributed.run --nproc-per-node W --master-addr 127.0.0.1 scripts/eval_dist_check.py [--json OUT]
    python scripts/eval_dist_check.py --virtual W [--json OUT]      # one GPU: W virtual ranks, stages run in turn

With --virtual the exchanges are replaced by W local buffers (reid_peer_scatter_rows only stores to the addresses it
is given); each stage is timed per virtual rank and the maximum is reported."""
import argparse
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import reid_gan_b200 as rg  # noqa: E402
from reid_gan_b200 import eval_dist as ed  # noqa: E402
from reid_gan_b200._lib import call, ptr  # noqa: E402
from reid_gan_b200.evaluation import pairwise_distance_device  # noqa: E402
from reid_gan_b200.rerank import _check_k, _re_ranking_features, _rr_blend, _rr_sparse  # noqa: E402
from reid_gan_b200.sharded import partition  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--virtual", type=int, default=0, help="W virtual ranks on one GPU (no torchrun)")
ap.add_argument("--Q", type=int, default=11659)
ap.add_argument("--G", type=int, default=82161)
ap.add_argument("--D", type=int, default=2048)
ap.add_argument("--json", default=None, help="append one JSON object (rank 0)")
args = ap.parse_args()

if args.virtual:
    rank, world, lr = 0, args.virtual, 0
else:
    rank, world, lr = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(lr)
dev = torch.device("cuda", lr)
if not args.virtual:
    dist.init_process_group("nccl", device_id=dev)
Q, G, D = args.Q, args.G, args.D
M = Q + G


def sha(t):
    return hashlib.sha256(np.ascontiguousarray(t.cpu().numpy()).tobytes()).hexdigest()[:16]


card = ""
if rank == 0:
    try:
        card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(lr)],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        card = "unknown (%r)" % (e,)
    print("card: %s; world %d%s" % (card, world, " (virtual)" if args.virtual else ""), flush=True)

x_host, ids = rg.synth(M, D, 3060, 0.8, 17)
cams = np.random.default_rng(17).integers(0, 15, M)
names = ["%07d.jpg" % i for i in np.random.default_rng(18).permutation(M)]
items = [(names[i], int(ids[i]), int(cams[i])) for i in range(M)]
query, gallery = items[:Q], items[Q:]
row_of = {names[i]: i for i in range(M)}


def loader(share, batch=512):
    out = []
    for i in range(0, len(share), batch):
        chunk = share[i:i + batch]
        rows = torch.tensor([row_of[f] for f, _, _ in chunk])
        out.append((x_host[rows], [f for f, _, _ in chunk], [p for _, p, _ in chunk], [c for _, _, c in chunk], 0))
    return out


class Timer:
    def __init__(self):
        self.ms = {}

    def __call__(self, name, fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        torch.cuda.synchronize()
        self.ms[name] = max(self.ms.get(name, 0.0), e0.elapsed_time(e1))
        return out


# single-process reference (every rank computes it; it is deterministic)
model = torch.nn.Identity()
full = loader(sorted(items))
ev = rg.Evaluator(model)
ref_plain = ev.evaluate(full, query, gallery, cmc_flag=True)
ref_rr = ev.evaluate(full, query, gallery, cmc_flag=True, rerank=True)
feats, _ = rg.extract_features(model, full)
q, g = feats.matrix([f for f, _, _ in query]), feats.matrix([f for f, _, _ in gallery])
ref_out, _ = _re_ranking_features(q, g, q_g_dist=pairwise_distance_device(q, g))
ref_sha = sha(ref_out)
del feats, q, g, ref_out
torch.cuda.empty_cache()

t = Timer()
if args.virtual:
    qpos, gpos = ed._positions(query, gallery)
    bufs = [torch.empty((M, D), device=dev) for _ in range(world)]
    base = torch.tensor([b.data_ptr() for b in bufs], dtype=torch.int64, device=dev)
    for r in range(world):
        f, _ = rg.extract_features(model, loader(rg.eval_shard(query, gallery, world=world, rank=r)))
        nm = list(f.keys())
        table = ed.dst_table(nm, qpos, gpos, dev)
        t("scatter", lambda: call("reid_peer_scatter_rows", ptr(f._buf), len(nm), D, ptr(table), M, world, ptr(base), 0,
                                  None, None))
        del f
    ids_d = ed.device_ids(query, gallery, dev)
    Bq = -(-Q // world)
    cols = _check_k(20, 6, M)
    rows, rows_rr, outs, colmax, rank_l, qgs = [], [], [], [], [], []
    for r in range(world):
        x = bufs[r]
        q0, q1 = partition(Q, world, r)
        qgs.append(pairwise_distance_device(x[q0:q1], x[Q:]))
        rows.append(t("distance_metrics", lambda: ed.block_metrics(pairwise_distance_device(x[q0:q1], x[Q:]), q0, ids_d,
                                                                    ed.CMC_TOPK, Bq))[:q1 - q0])
        sqn = torch.empty(M, dtype=torch.float64, device=dev)
        call("reid_rr_row_sqnorm64", ptr(x), M, D, ptr(sqn), None)
        r0, r1 = partition(M, world, r)
        c, k = t("rerank_search", lambda: ed.rerank_rows(x, sqn, cols, r0, r1))
        colmax.append(c)
        rank_l.append(k)
    colmax, rank_all = torch.cat(colmax), torch.cat(rank_l)
    for r in range(world):
        x = bufs[r]
        q0, q1 = partition(Q, world, r)
        sqn = torch.empty(M, dtype=torch.float64, device=dev)
        call("reid_rr_row_sqnorm64", ptr(x), M, D, ptr(sqn), None)
        sp = t("sparse_stages", lambda: _rr_sparse(x, sqn, colmax, rank_all, 20, 6))
        out = t("rerank_blend_metrics", lambda: _rr_blend(x, sp, colmax, Q, 0.3, qgs[r], q0, q1))
        del sp
        outs.append(out)
        rows_rr.append(ed.block_metrics(out, q0, ids_d, ed.CMC_TOPK, Bq)[:q1 - q0])
    same_x = all(torch.equal(b, bufs[0]) for b in bufs)
    m_plain, c_plain = ed.metrics_from_rows(torch.cat(rows), ed.CMC_TOPK)
    m_rr, c_rr = ed.metrics_from_rows(torch.cat(rows_rr), ed.CMC_TOPK)
    got_sha = sha(torch.cat(outs))
    results = [(m_plain, c_plain, m_rr, c_rr, got_sha, same_x)]
else:
    ed.TRACE_STEPS = True
    dev_ev = rg.DistributedEvaluator(model)
    share_loader = loader(rg.eval_shard(query, gallery))
    c_plain, m_plain = dev_ev.evaluate(share_loader, query, gallery, cmc_flag=True)
    steps = dict(dev_ev.steps_ms)
    c_rr, m_rr = dev_ev.evaluate(share_loader, query, gallery, cmc_flag=True, rerank=True)
    steps.update({k: v for k, v in dev_ev.steps_ms.items() if k != "scatter" and k != "distance_metrics"})
    for k in sorted(steps):
        v = torch.tensor([steps[k]], device=dev)
        dist.all_reduce(v, op=dist.ReduceOp.MAX)
        t.ms[k] = float(v.item())
    mine = (m_plain, c_plain, m_rr, c_rr, None, True)
    results = [None] * world
    dist.all_gather_object(results, mine)

ok = all(r[0] == ref_plain[1] and np.array_equal(r[1], ref_plain[0]) and r[2] == ref_rr[1]
         and np.array_equal(r[3], ref_rr[0]) and r[5] for r in results)
if args.virtual:
    ok = ok and results[0][4] == ref_sha
if rank == 0:
    rec = dict(world=world, virtual=bool(args.virtual), Q=Q, G=G, D=D, identical=bool(ok), ref_sha=ref_sha,
               rerank_sha=results[0][4], mAP=float(ref_plain[1]), mAP_rerank=float(ref_rr[1]),
               stage_ms={k: round(v, 3) for k, v in t.ms.items()}, card=card)
    print(json.dumps(rec), flush=True)
    print("EVAL DIST OK" if ok else "EVAL DIST MISMATCH", flush=True)
    if args.json:
        with open(args.json, "a") as f:
            f.write(json.dumps(rec) + "\n")
if not args.virtual:
    torch.cuda.synchronize()
    dist.barrier()
    os._exit(0 if ok else 1)
sys.exit(0 if ok else 1)
