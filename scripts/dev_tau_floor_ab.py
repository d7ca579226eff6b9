"""Phase B of the sample-first search (the other rows against the sample) on the symmetric kernel with a provisional
threshold tau', against the tree of another commit.

  python scripts/dev_tau_floor_ab.py stats [--workloads market,rerank,hard,scale100k]
      one JSON line per workload: list lengths (mean / min / max of the candidate counts), rows whose
      threshold stayed tau', uncertified rows, per-entry-point CUDA-event ms of the search, sha256 of neighbours + keys;
  python scripts/dev_tau_floor_ab.py bench --other TREE [--reps 5] [--steps 200] [--workloads rerank,market,hard]
      the card's name and power limit, then bench.py of this tree and of TREE alternately, --reps times each per
      workload; one JSON line per run and a summary (median, spread) per tree and workload.

`stats` runs in whichever tree it is started from; running it from both trees compares the lists."""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def stats(args):
    sys.path.insert(0, ROOT)
    import numpy as np
    import torch
    import bench
    import reid_gan_b200 as rg
    from reid_gan_b200 import _lib, knn_tc as kt, faiss_rerank as fr
    has_floor = hasattr(kt, "_tau_floor")
    for wl in args.workloads.split(","):
        W = bench.WORKLOADS[wl]
        if W["gen"] == "synth_device":
            x = rg.synth_device(W["N"], W["D"], W["n_ids"], W["noise"], W["seed"], device="cuda")[0]
        else:
            import importlib
            x = getattr(importlib.import_module("reid_gan_b200.synth"), W["gen"])(**bench.synth_args(W))[0].cuda()
        N, D, k = W["N"], W["D"], W["k1"]
        m = kt.sample_size(N, k)
        for _ in range(2):
            idx, key, info = fr.knn_search(x, k, "tc")
        torch.cuda.synchronize()
        steps = 5
        _lib.profiler.start()
        for _ in range(steps):
            idx, key, info = fr.knn_search(x, k, "tc")
        torch.cuda.synchronize()
        _lib.profiler.stop()
        prof = {n: round(v[1] / steps, 4) for n, v in _lib.profiler.summary().items()}
        cnt = info["cand_cnt"]
        h = hashlib.sha256(idx.cpu().numpy().tobytes() + key.cpu().numpy().tobytes()).hexdigest()[:16]
        line = dict(tree=ROOT, workload=wl, N=N, sample=m, uncertified=int(info["uncertified_rows"]),
                    list_mean=round(float(cnt.float().mean()), 1), list_min=int(cnt.min()), list_max=int(cnt.max()),
                    lists_over_cap=int((cnt > kt.SYM_CAP).sum()), stage_ms=prof, knn_sha=h)
        if has_floor:                        # rows that kept tau': their threshold equals tau'
            msq = torch.zeros(2, dtype=torch.float32, device=x.device)
            _, cnt2, tau_o, _, _, _, _ = kt._candidates_sym_sf(x, N, D, _lib.stream_ptr(), x.device, k, msq)
            t = tau_o.cpu().numpy().view(np.uint32)
            floor = t[:m].min()
            line.update(tau_floor_rows=int((t[m:] == floor).sum()), other_rows=N - m,
                        list_mean_other=round(float(cnt2[m:].float().mean()), 1))
        print(json.dumps(line), flush=True)
        del x
        torch.cuda.empty_cache()


def bench_ab(args):
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                         text=True).stdout, flush=True)
    trees = [("this", ROOT), ("other", os.path.abspath(args.other))]
    runs = {}
    for wl in args.workloads.split(","):
        for rep in range(args.reps):
            for name, tree in (trees if rep % 2 == 0 else trees[::-1]):
                cmd = [sys.executable, "bench.py", "--gpus", "1", "--steps", str(args.steps), "--warmup", "20",
                       "--no-cpu-baseline", "--workload", wl]
                p = subprocess.run(cmd, cwd=tree, capture_output=True, text=True)
                js = [l for l in p.stdout.splitlines() if l.startswith("{")]
                if p.returncode or not js:
                    print(json.dumps(dict(tree=name, workload=wl, error=p.stderr[-2000:])), flush=True)
                    continue
                r = json.loads(js[-1])
                c = r["config"]
                line = dict(tree=name, workload=wl, rep=rep, ms_per_step=round(r["ms_per_step"], 4),
                            labels_sha256=c["labels_sha256"][:16], rank_sha256=c["rank_sha256"][:16],
                            e2e_labels_sha256=c.get("e2e_labels_sha256", "")[:16],
                            uncertified_rows=c["uncertified_rows"], stage_ms=r["stage_ms"])
                print(json.dumps(line), flush=True)
                runs.setdefault((wl, name), []).append(r["ms_per_step"])
    for (wl, name), v in sorted(runs.items()):
        print(json.dumps(dict(summary=True, workload=wl, tree=name, n=len(v), median=round(statistics.median(v), 4),
                              min=round(min(v), 4), max=round(max(v), 4), spread=round(max(v) - min(v), 4))), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("mode", choices=["stats", "bench"])
    ap.add_argument("--workloads", default=None)
    ap.add_argument("--other", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--steps", type=int, default=200)
    args = ap.parse_args()
    if args.mode == "stats":
        args.workloads = args.workloads or "market,rerank,hard,scale100k"
        stats(args)
    else:
        if not args.other:
            ap.error("bench needs --other TREE")
        args.workloads = args.workloads or "rerank,market,hard"
        bench_ab(args)


if __name__ == "__main__":
    main()
