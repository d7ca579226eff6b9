"""Evaluation re-ranking from features (re_ranking_features) against the dense re_ranking on synthetic, seeded features.
    Market-1501 shape (Q = 3,368, G = 15,913, D = 2048): both paths -- max |difference|, mAP / CMC of each, median call
        time over warmed repeats (CUDA events), peak device memory of the call.
    MSMT17 shape (Q = 11,659, G = 82,161): the feature path only -- time per C entry (grouped into stages), peak memory,
        uncertified rows of the kNN and of the farthest-neighbour search.
One JSON line per result; the card name and power limit are read in the same run.
    python scripts/eval_rerank_check.py [--repeats R] [--skip-msmt] [--json OUT]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import reid_gan_b200 as rg  # noqa: E402
from reid_gan_b200 import _lib, evaluation as ev  # noqa: E402
from reid_gan_b200.rerank import _re_ranking_features  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--repeats", type=int, default=5)
ap.add_argument("--skip-msmt", action="store_true")
ap.add_argument("--json", default=None)
args = ap.parse_args()
if not torch.cuda.is_available():
    raise SystemExit("needs a CUDA device")
dev = torch.device("cuda", 0)
torch.cuda.set_device(dev)


def emit(obj):
    line = json.dumps(obj)
    print(line, flush=True)
    if args.json:
        with open(args.json, "a") as f:
            f.write(line + "\n")


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def fixture(Q, G, D, seed):
    x, ids = rg.synth_device(Q + G, D, max(1, (Q + G) // 16), 0.8, seed)
    cams = torch.randint(0, 6, (Q + G,), generator=torch.Generator().manual_seed(seed))
    ids = ids.cpu().numpy()
    return x[:Q].contiguous(), x[Q:].contiguous(), (ids[:Q], ids[Q:], cams[:Q].numpy(), cams[Q:].numpy())


def timed(fn, repeats):
    out = fn()                                                 # warm-up: module loads, allocator
    times, peaks = [], []
    for _ in range(repeats):
        del out
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
        peaks.append(torch.cuda.max_memory_allocated() - base)
    return out, float(np.median(times)), max(peaks)


def metrics(d, ids):
    return float(ev.mean_ap(d, *ids)), [float(v) for v in ev.cmc(d, *ids, first_match_break=True)[[0, 4, 9]]]


gpu = card()
# ---- Market-1501 shape: both paths ----------------------------------------------------------------------------------
Q, G, D = 3368, 15913, 2048
q, g, ids = fixture(Q, G, D, 1)
pd = ev.pairwise_distance_device
feat = lambda: _re_ranking_features(q, g)[0]                   # noqa: E731
dense = lambda: rg.re_ranking(pd(q, g), pd(q, q), pd(g, g), return_device=True)   # noqa: E731
out_f, t_f, m_f = timed(feat, args.repeats)
out_d, t_d, m_d = timed(dense, args.repeats)
_, parts = _re_ranking_features(q, g)
map_f, cmc_f = metrics(out_f, ids)
map_d, cmc_d = metrics(out_d, ids)
diff = (out_f - out_d).abs()
emit(dict(shape="market", Q=Q, G=G, D=D, gpu=gpu, max_abs_diff=float(diff.max()),
          rows_over_1e5=int((diff.max(dim=1).values > 1e-5).sum()), entries_over_1e5=int((diff > 1e-5).sum()),
          features=dict(ms=t_f, peak_mb=m_f / 2**20, mAP=map_f, cmc_1_5_10=cmc_f,
                        knn_mode=parts["knn_info"]["mode"], farthest_mode=parts["farthest_info"]["mode"],
                        knn_uncertified=int(parts["knn_info"]["uncertified_rows"]),
                        farthest_uncertified=int(parts["farthest_info"]["uncertified_rows"])),
          dense=dict(ms=t_d, peak_mb=m_d / 2**20, mAP=map_d, cmc_1_5_10=cmc_d), repeats=args.repeats))
del out_f, out_d, q, g, parts
torch.cuda.empty_cache()

# ---- MSMT17 shape: the feature path, per stage ----------------------------------------------------------------------
STAGES = {"reid_rr_row_sqnorm64": "norms", "reid_features_to_half": "farthest", "reid_knn_tc_plan": "farthest",
          "reid_knn_candidates_tc_ab": "farthest", "reid_rr_farthest_certify": "farthest", "reid_rr_farthest_exact": "farthest",
          "reid_rr_weights_features": "weights", "reid_pairwise_distance": "qg_distance", "reid_jaccard_dense": "jaccard_blend",
          "reid_rr_final_qg": "jaccard_blend", "reid_rank_metrics": "metrics"}
SPARSE = ("reid_reciprocal_masks", "reid_expand", "reid_query_expand", "reid_csr_compact", "reid_transpose_count",
          "reid_transpose_fill", "reid_scan_counts")
if not args.skip_msmt:
    Q, G = 11659, 82161
    q, g, ids = fixture(Q, G, D, 2)
    _re_ranking_features(q, g)                                 # warm-up
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    _lib.profiler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out, parts = _re_ranking_features(q, g)
    e1.record()
    mAP, cmc1 = metrics(out, ids)
    torch.cuda.synchronize()
    _lib.profiler.stop()
    peak = torch.cuda.max_memory_allocated() - base
    stages = {}
    for name, (calls, ms) in _lib.profiler.summary().items():
        key = STAGES.get(name, "sparse" if name in SPARSE else "knn")
        stages[key] = stages.get(key, 0.0) + ms
    emit(dict(shape="msmt17", Q=Q, G=G, D=D, gpu=gpu, call_ms=e0.elapsed_time(e1), stage_ms=stages, peak_mb=peak / 2**20,
              knn_mode=parts["knn_info"]["mode"], knn_uncertified=int(parts["knn_info"]["uncertified_rows"]),
              farthest_mode=parts["farthest_info"]["mode"], farthest_uncertified=int(parts["farthest_info"]["uncertified_rows"]),
              mAP=mAP, cmc_1_5_10=cmc1, note="stage_ms: CUDA events around each C entry during one profiled call"))
