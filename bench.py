#!/usr/bin/env python
"""Benchmark of the pseudo-label hot path (BASELINE.json: "k-reciprocal Jaccard+DBSCAN sec at N=32,621").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload rerank|cm|pass|market|scale100k|scale250k|hard]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

--dump-outputs DIR writes what the last timed step computed as DIR/<name>.npy (see dump_outputs); the inputs are seeded,
so two builds run with the same arguments can be compared output for output.

A step = one full pass: kNN (tcgen05 GEMM + fused top-K + exact re-score) -> k-reciprocal sets ->
expansion -> Gaussian weights -> k2 query expansion -> inverted index -> sparse Jaccard eps-graph ->
DBSCAN labels, on synthetic L2-normalised 2048-d features (BASELINE configs[1]: N=32,621, k1=30,
k2=6, eps=0.6, min_samples=4).  `value` = seconds per pass with the features resident in HBM;
`e2e` = the same pass through the drop-in API (compute_jaccard_distance + DBSCAN.fit_predict)
from pinned HOST features to HOST labels.  With --gpus N the rows are partitioned across N ranks
(strong scaling: the job is one N=32,621 pass).  `--workload cm` times BASELINE configs[2] instead (ClusterMemory
CM_Hard forward + backward + momentum update, latency bound: reported as seconds per step with the launch count).  `--impl reference` times the CPU restatement of the
reference on the host cores instead, at the FULL size of the workload (no sample, no scaling): the reference's own
unmodified faiss_rerank.py (byte-identical copy under the git-ignored oracle/_ref, placed there by
oracle/build_ref.py; faiss itself is not in this image and is replaced by an exact search that is timed
separately) + sklearn DBSCAN on the dense matrix, or the oracle's numpy port when that copy / the memory for
three dense N x N matrices is missing.  Every line carries config.labels_sha256 / rank_sha256: the same digest on the
reference arm and on 1, 2, 4 and 8 GPUs is the parity statement of the run.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "k-reciprocal Jaccard+DBSCAN sec at N=32,621"
_BASE = dict(D=2048, noise=0.8, seed=0, k1=30, k2=6, eps=0.6, min_samples=4, gen="synth", centroids=False)
# BASELINE.json configs[0..4]; "rerank" (configs[1]) is the headline the metric is quoted on
WORKLOADS = {
    "market": dict(_BASE, N=12936, n_ids=751, metric="k-reciprocal Jaccard+DBSCAN sec at N=12,936",
                   name="configs[0]: compute_jaccard_distance k1=30 k2=6 (+DBSCAN eps=0.6) on synthetic N=12936x2048 (Market-1501 train shape)"),
    "rerank": dict(_BASE, N=32621, n_ids=1041, metric=METRIC,
                   name="configs[1]: Jaccard re-rank + DBSCAN eps=0.6 min_samples=4 at N=32621x2048 (MSMT17 shape), k1=30 k2=6"),
    "pass": dict(_BASE, N=32621, n_ids=1041, centroids=True, metric="full pseudo-label pass (re-rank+DBSCAN+centroid init) sec at N=32,621",
                 name="configs[3]: full pseudo-label pass (re-rank + DBSCAN + centroid init) N=32621x2048, row-sharded over the ranks"),
    "scale100k": dict(_BASE, N=100000, n_ids=3200, gen="synth_device", metric="k-reciprocal Jaccard+DBSCAN sec at N=100,000",
                      name="configs[4]: scale sweep N=100000x2048 synthetic, row-partitioned"),
    "scale250k": dict(_BASE, N=250000, n_ids=8000, gen="synth_device", metric="k-reciprocal Jaccard+DBSCAN sec at N=250,000",
                      name="configs[4]: scale sweep N=250000x2048 synthetic, row-partitioned"),
    "hard": dict(_BASE, N=20480, n_ids=None, gen="synth_hard", metric="k-reciprocal Jaccard+DBSCAN sec at N=20,480 (hard set)",
                 name="parity set: heavy-tailed identities, hubs, duplicates, noise points, N=20480x2048"),
}
WORKLOAD = WORKLOADS["rerank"]


def workload(args):
    W = dict(WORKLOADS[args.workload])
    if getattr(args, "n", None):
        W["n_ids"] = max(1, round(W["n_ids"] * args.n / W["N"])) if W.get("n_ids") else None
        W["N"] = args.n
        W["name"] += " [N overridden to %d: development only]" % args.n
    return W


def synth_args(W):
    if W["gen"] == "synth_hard":
        return dict(N=W["N"], D=W["D"], seed=W["seed"])
    return dict(N=W["N"], D=W["D"], n_ids=W["n_ids"], noise=W["noise"], seed=W["seed"])


# ------------------------------------------------------------------ clocks -------------------
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
        sm, mx, pw, reasons = [], [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for r in self.rows:
            f = [c.strip() for c in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            try:
                pw.append(float(f[3]))
            except ValueError:
                pass
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm.sort()
        pw.sort()
        # power_w: board power during the timed region -- the symmetric candidate kernel runs into the board's power limit
        # (sw_power_cap; DESIGN.md 4, profiles/r02_k1_power.txt), which is what `reasons` then reports
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm),
                "power_w_median": pw[len(pw) // 2] if pw else None, "power_w_max": pw[-1] if pw else None}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return {"bf16_tflops": d.get("bf16_tflops", 1590.0), "hbm_gbs": d.get("hbm_gbs", 6650.0), "source": "measured"}
    return {"bf16_tflops": 1590.0, "hbm_gbs": 6650.0, "source": "fallback"}


# ------------------------------------------------------------------ CPU reference ------------
def pin_host_threads():
    """The CPU legs use every host core whatever the launcher exported (torchrun sets OMP_NUM_THREADS=1, which made
    the N=1 and N>1 reference arms differ 2.4x in round 1).  Must run before numpy / torch are imported."""
    n = os.cpu_count() or 1
    for k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS", "NUMEXPR_NUM_THREADS"):
        os.environ[k] = str(n)
    return n


def labels_sha256(labels):
    import hashlib
    import numpy as np
    return hashlib.sha256(np.ascontiguousarray(np.asarray(labels).astype(np.int64)).tobytes()).hexdigest()


def rank_sha256(rank):
    import hashlib
    import numpy as np
    return hashlib.sha256(np.ascontiguousarray(np.asarray(rank).astype(np.int32)).tobytes()).hexdigest()


DUMP_BYTES = 64 << 20                  # --dump-outputs writes at most this much in all,
DUMP_ARRAY_BYTES = DUMP_BYTES // 8     # and at most this much per output (a step has at most six outputs)


def host_outputs(arrays):
    """Host copies of one step's outputs (None entries dropped), taken before later passes reuse their buffers."""
    return {name: a.detach().cpu().numpy() for name, a in arrays.items() if a is not None}


def dump_outputs(out_dir, arrays):
    """Write every output as out_dir/<name>.npy: float64 stays float64, other floats become float32, integers and flags
    float64 (exact below 2^53).  An output larger than DUMP_ARRAY_BYTES keeps a fixed, seeded sample of its rows, whose
    indices go to out_dir/<name>_rows.npy: the same rows for the same shape, whichever build wrote them."""
    import numpy as np
    files = {}
    for name, a in arrays.items():
        a = np.asarray(a)
        a = a.astype(np.float32 if a.dtype in (np.float16, np.float32) else np.float64).reshape(a.shape or (1,))
        if a.nbytes > DUMP_ARRAY_BYTES:
            m = DUMP_ARRAY_BYTES // (a.nbytes // a.shape[0] + 8)
            rows = np.sort(np.random.default_rng(0).choice(a.shape[0], m, replace=False))
            files[name + "_rows"] = rows.astype(np.float64)
            a = a[rows]
        files[name] = a
    total = sum(a.nbytes for a in files.values())
    if total > DUMP_BYTES:
        raise RuntimeError("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in files.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def pass_outputs(out):
    """What a caller of pipeline / sharded.pseudo_labels receives: labels, core-point flags, the number of clusters, the
    centroids when the workload asks for them, and the neighbour lists with their search keys (the rank's own rows)."""
    st = out["state"]
    return {"labels": out["labels"], "core": out["core"], "num_clusters": out["num_clusters"],
            "centroids": out.get("centroids"), "neighbors": st.rank, "neighbor_keys": st.rank_key}


def host_mem_gb():
    try:
        import psutil
        return psutil.virtual_memory().available / 2 ** 30
    except Exception:
        return 0.0


def cpu_reference_pass(W, kind="auto", x=None):
    """ONE full pass of the workload on the host cores -- the whole N, no sample, no scaling.

    kind "_ref": the reference itself -- the unmodified clustercontrast/utils/faiss_rerank.py compute_jaccard_distance
    (search_option=3, oracle/_ref copy loaded by oracle/ref_shim.py; faiss = exact stand-in, timed separately) followed
    by sklearn DBSCAN on the dense matrix, exactly the two calls of examples/cluster_contrast_train_usl.py:154-163 (and
    the centroid closure :169-191 when the workload asks for it).  Needs ~4 x N^2 x 4 bytes of host memory.
    kind "port": the oracle's sparse numpy restatement of the same lines + sklearn DBSCAN on the dense matrix.
    "auto": "_ref" when oracle/_ref is present and the host has the memory, else "port"."""
    import numpy as np
    import torch
    from oracle import rerank as orr, cluster as ocl, ref_shim
    import importlib
    sm = importlib.import_module("reid_gan_b200.synth")
    N = W["N"]
    need_gb = 4.5 * N * N * 4 / 2 ** 30
    if kind == "auto":
        kind = "_ref" if (ref_shim.available() and host_mem_gb() > need_gb + 4) else "port"
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    if x is None:
        x = getattr(sm, W.get("gen", "synth"))(**synth_args(W))[0]
    xn = x.numpy()
    ocl.sklearn_dbscan(np.zeros((8, 8), np.float32), 0.5, 2)          # one-time joblib/threadpool start-up, untimed
    t = {}
    t_all = time.perf_counter()
    t0 = time.perf_counter()
    rank = orr.exact_knn(xn, W["k1"])                                 # faiss IndexFlatL2 stand-in (BLAS, all cores)
    t["knn_stand_in"] = time.perf_counter() - t0
    if kind == "_ref":
        mod = ref_shim.load_faiss_rerank()
        import faiss as faiss_stub                                    # the stand-in registered by ref_shim
        faiss_stub.IndexFlatL2.precomputed = (xn, rank)               # the search above is not repeated inside the call
        torch.set_num_threads(1)                                      # per-row torch.mm (faiss_rerank.py:83) thrashes with more
        t0 = time.perf_counter()
        J = mod.compute_jaccard_distance(x, k1=W["k1"], k2=W["k2"], print_flag=False, search_option=3)
        t["compute_jaccard_distance_after_search"] = time.perf_counter() - t0
        torch.set_num_threads(cores)
        faiss_stub.IndexFlatL2.precomputed = None
    else:
        t0 = time.perf_counter()
        ep, ei = orr.expand(rank, W["k1"])
        t["reciprocal+expand"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        ev = orr.v_weights(xn, ep, ei)
        t["v_weights"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        qp, qi, qv = orr.query_expand(ep, ei, ev, rank, W["k2"])
        t["query_expand"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        jp, jj, jv = orr.jaccard_sparse(qp, qi, qv, N)
        t["jaccard"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        J = orr.jaccard_dense_from_sparse(jp, jj, jv, N)              # the reference hands DBSCAN the dense matrix
        t["densify"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    labels = ocl.sklearn_dbscan(J, W["eps"], W["min_samples"])        # the reference's own DBSCAN on the dense matrix
    t["dbscan_dense"] = time.perf_counter() - t0
    del J
    if W.get("centroids"):
        t0 = time.perf_counter()
        if kind == "_ref":
            ref_shim.ref_generate_cluster_features(labels, x)
        else:
            ocl.cluster_centroids(xn, labels)
        t["centroids"] = time.perf_counter() - t0
    total = time.perf_counter() - t_all
    return {"value": total, "unit": "s", "cores": cores, "kind": "reference" if kind == "_ref" else "port",
            "sample": "the whole workload (N=%d), one pass, no scaling" % N,
            "what": ("unmodified faiss_rerank.compute_jaccard_distance(search_option=3) from oracle/_ref + sklearn DBSCAN on the "
                     "dense N x N matrix; faiss (not in this image) replaced by an exact fp64-BLAS search, timed as knn_stand_in"
                     if kind == "_ref" else
                     "oracle port (sparse numpy/scipy restatement of faiss_rerank.py:58-123) + sklearn DBSCAN on the dense matrix"),
            "stages_s": {k: round(v, 3) for k, v in t.items()},
            "threads": {"blas": cores, "torch_in_reference_loop": 1 if kind == "_ref" else cores, "os_cpu_count": cores,
                        "OMP_NUM_THREADS": os.environ.get("OMP_NUM_THREADS")},
            "clusters": int(labels.max() + 1), "noise_points": int((labels < 0).sum()),
            "labels_sha256": labels_sha256(labels), "rank_sha256": rank_sha256(rank)}


def run_reference(args):
    """--impl reference: the reference's CPU path on the box's host cores, on OUR arm's config (the whole N).  A pass
    takes minutes, so the number of passes is capped by wall time (--ref-budget-s) and reported as steps_run."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    W = workload(args)
    vals, last = [], None
    t_start = time.perf_counter()
    want = max(1, args.steps)
    done_warm = 0
    while len(vals) < want:
        last = cpu_reference_pass(W, args.ref_kind)
        elapsed = time.perf_counter() - t_start
        per = elapsed / (len(vals) + done_warm + 1)
        if done_warm < args.warmup and elapsed + (want + args.warmup - done_warm) * per < args.ref_budget_s:
            done_warm += 1                                            # affordable: treat this pass as a warm-up
            continue
        vals.append(last["value"])
        if elapsed + per > args.ref_budget_s:
            break
    v = sum(vals) / len(vals)
    last["value"] = v
    out = {"impl": "reference", "metric": W["metric"], "value": v, "unit": "s", "n_gpus": args.gpus, "steps": args.steps,
           "steps_run": len(vals), "warmup": args.warmup, "warmup_run": done_warm,
           "ms_per_step": v * 1e3, "higher_is_better": False, "scaling": "strong",
           "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": W["name"], **{k: W[k] for k in W if k not in ("metric", "name")},
                      "labels_sha256": last["labels_sha256"], "rank_sha256": last["rank_sha256"],
                      "clusters": last["clusters"], "noise_points": last["noise_points"],
                      "note": "full-size pass on the host cores; passes capped by --ref-budget-s=%g s of wall time" % args.ref_budget_s},
           "cpu_baseline": last,
           "e2e": {"value": v, "unit": "s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


# ------------------------------------------------------------------ per-stage roofline -------
def stage_rooflines(out, W, prof, steps, peaks, world):
    """SURVEY.md 8(d): algorithmic bytes (or flops) of every stage, counted from THIS run's sparse structures,
    over the stage's CUDA-event time inside the timed region.  Stages that are not the dominant kernel are
    gather / scan / sparse work: the bound is HBM bandwidth; several work out of L2 at this N (flagged)."""
    import torch
    st = out["state"]
    N, D, k1, k2 = st.N, st.D, st.k1, st.k2
    n = st.row_end - st.row_begin
    from reid_gan_b200.faiss_rerank import half_k
    h = half_k(k1)
    dev = st.rank.device

    def popc(m):
        m = m.clone()
        c = torch.zeros_like(m)
        for _ in range(64):
            c += m & 1
            m >>= 1
        return c

    r_cnt, rh_cnt = popc(st.R_mask[:n]), popc(st.Rh_mask)
    sum_R, sum_Rh = int(r_cnt.sum()), int(rh_cnt[st.row_begin:st.row_end].sum())
    e_cnt = (st.E_ptr[1:] - st.E_ptr[:-1])
    sum_E = int(e_cnt[st.row_begin:st.row_end].sum()) if e_cnt.numel() == N else int(e_cnt.sum())
    rank_local = st.rank[st.row_begin:st.row_end].long()
    # sum_i sum_{c in R(i)} |R_half(c)|  (R(i) as bit positions into rank[i,:])
    bits = ((st.R_mask[:n].unsqueeze(1) >> torch.arange(k1, device=dev)) & 1).bool()
    sum_RRh = int((rh_cnt[rank_local] * bits).sum())
    e_all = e_cnt if e_cnt.numel() == N else None
    sum_qe_in = int(e_all[rank_local[:, :k2]].sum()) if (e_all is not None and k2 != 1) else 0
    nnz_q = int(st.q_total)
    q_cnt = st.Q_ptr[1:] - st.Q_ptr[:-1]
    nnz_q_local = int(q_cnt[st.row_begin:st.row_end].sum())
    col_cnt = st.C_ptr[1:] - st.C_ptr[:-1]
    qa, qb = int(st.Q_ptr[st.row_begin]), int(st.Q_ptr[st.row_end])
    T = int(col_cnt[st.Q_idx[qa:qb].long()].sum())
    edges = int(out["nbr_cnt"].sum()) if "nbr_cnt" in out else 0
    win = out["state"].knn_info.get("window_counts")
    win = int(win.sum()) if win is not None else n * k1
    hbm = peaks["hbm_gbs"]

    def ms(*names):
        return sum(prof[nm][1] for nm in names if nm in prof) / steps

    sym = st.knn_info.get("sym") or {}
    # members of E(i) that are NOT among the row's k1 neighbours: the only ones whose feature row a4 gathers
    e_rows = torch.repeat_interleave(torch.arange(n, device=dev), e_cnt[st.row_begin:st.row_end] if e_cnt.numel() == N else e_cnt)
    ea, eb = (int(st.E_ptr[st.row_begin]), int(st.E_ptr[st.row_end])) if e_cnt.numel() == N else (0, sum_E)
    gathered = 0
    for c0 in range(0, e_rows.numel(), 1 << 20):
        rr = e_rows[c0:c0 + (1 << 20)]
        ee = st.E_idx[ea + c0: ea + c0 + rr.numel()]
        gathered += int((~(rank_local[rr] == ee[:, None].long()).any(1)).sum())
    fp64_peak = 148 * 64 * 2 * 1.965e9 / 1e12        # nominal: 64 FP64 FMA / clk / SM x 148 SMs x 1965 MHz = 37.2 TFLOP/s
    rows = [
        ("features_to_half", ("reid_features_to_half", "reid_features_to_half_gather", "reid_sqnorm_range_reset"), "hbm", 6.0 * N * D, "4ND read + 2ND write"),
        ("K1 sample thresholds", ("reid_features_sample", "reid_knn_candidates_tc_ab", "reid_knn_sample_tau", "reid_knn_candidates_tc_abt",
                                  "reid_knn_sample_tau_emit"), "tensor",
         2.0 * (n if world == 1 else -(-N // world)) * sym.get("sample", 0) * D,
         "2 * rows * sample(%d) * D flops (tcgen05 prepass) + r-th best selection" % sym.get("sample", 0)),
        ("K2 re-score", ("reid_knn_rescore", "reid_knn_rescore_mapped"), "fp64", 2.0 * D * win,
         "exact keys: 2*D flops per window member in the FP64 pipe, window total %d (%.1f/row); peak = nominal 64 FMA/clk/SM; "
         "HBM side: every feature row is needed once (4ND = %.0f MB compulsory), the SURVEY gather formula 4D*(window+rows) = "
         "%.2f GB is served by L2 because rows are visited in cluster-locality order" % (win, win / max(n, 1), 4.0 * N * D / 1e6,
                                                                                      (4.0 * D * (win + n)) / 1e9)),
        ("K3 reciprocal+expand", ("reid_reciprocal_masks", "reid_expand", "reid_sets"), "hbm",
         4.0 * (n * k1 * k1 + N * (h + 1) * (h + 1) + sum_RRh + sum_R + sum_Rh + sum_E),
         "4*[rows*k1^2 + N*(h+1)^2 + sum|R_half(c)| over c in R(i) + sum|R| + sum|R_half| + sum|E|]; L2-resident"),
        ("K4 V weights", ("reid_v_weights",), "hbm", 4.0 * D * gathered + 4.0 * D * n + 8.0 * sum_E,
         "4D*(gathered members + rows) + 8*sum|E|: %d of the %d members are not among the row's k1 neighbours (the others "
         "re-use the search key); SURVEY's formula 4D*(rows + sum|E|) would be %.2f GB" % (gathered, sum_E, (4.0 * D * (n + sum_E)) / 1e9)),
        ("K5 query expansion", ("reid_query_expand", "reid_csr_compact"), "hbm", 8.0 * (sum_qe_in + nnz_q_local),
         "8*(sum_i sum_{r<k2}|E(rank[i,r])| + nnz(V_qe)); L2-resident"),
        ("K6 inverted index", ("reid_transpose_count", "reid_transpose_fill"), "hbm", 16.0 * nnz_q, "2*8*nnz(V_qe); L2-resident"),
        ("K7 Jaccard eps-graph", ("reid_jaccard_bounds", "reid_jaccard_eps_graph", "reid_jaccard_neighbors",
                                  "reid_jaccard_neighbors_heavy"), "hbm",
         8.0 * T + 8.0 * edges, "8*T + 8*edges, T=%d (%.0f/row), edges=%d; L2-resident" % (T, T / max(n, 1), edges)),
        ("K8 DBSCAN", ("reid_dbscan_labels",), "hbm", 8.0 * edges + 16.0 * N, "8*edges + 16N; L2-resident"),
        ("K12 centroids", ("reid_centroids",), "hbm", 4.0 * N * D, "4ND + 4CD"),
        ("scans", ("reid_scan_counts",), "hbm", 0.0, "count->pointer scans between count/fill passes (latency bound)"),
    ]
    table = []
    for name, entries, bound, work, note in rows:
        t = ms(*entries)
        if t <= 0:
            continue
        if bound in ("tensor", "fp64"):
            tf = work / (t * 1e-3) / 1e12
            pk = peaks["bf16_tflops"] if bound == "tensor" else fp64_peak
            table.append({"stage": name, "ms": round(t, 4), "bound": bound, "flops": int(work),
                          "achieved_tflops": round(tf, 2), "peak_tflops": round(pk, 1),
                          "frac": round(tf / pk, 4), "note": note})
            continue
        gbs = work / (t * 1e-3) / 1e9 if work else None
        table.append({"stage": name, "ms": round(t, 4), "bound": "hbm", "bytes": int(work),
                      "achieved_gbs": None if gbs is None else round(gbs, 1), "peak_gbs": hbm,
                      "frac": None if gbs is None else round(gbs / hbm, 4), "note": note})
    return table

# ------------------------------------------------------------------ ClusterMemory (configs[2]) ----
CM_METRIC = "ClusterMemory CM_Hard fwd+bwd+update sec/step"


def cm_setup():
    import torch
    import reid_gan_b200 as rg
    C, D, B = 700, 2048, 256
    x, ids = rg.synth(C * 24, D, C, 0.8, 0)
    cen = torch.nn.functional.normalize(torch.stack([x[ids == c].mean(0) if (ids == c).any() else x[0] for c in range(C)]), dim=1)
    batches = [rg.synth_cm_batch(x, None, ids.clone(), num_ids=16, num_instances=16, seed=s) for s in range(8)]
    return C, D, B, cen, batches


def run_cm(args):
    """BASELINE configs[2]: ClusterMemory CM_Hard forward + backward + momentum update, bs=256 (16 labels x 16),
    ~700 centroids x 2048-d, temp 0.05, momentum 0.2.  Latency bound (1.5 GFLOP, 16 MB): reported as seconds per step
    with the launch count.  --impl reference: the reference's own clustercontrast/models/cm.py (oracle/_ref copy)
    ClusterMemory(use_hard=True) on the GPU -- the arm SURVEY 8(d) names: 256 .cpu() syncs per backward (cm.py:66);
    without a GPU or without oracle/_ref, the oracle's numpy port on the host."""
    import numpy as np
    import torch
    import reid_gan_b200 as rg
    from reid_gan_b200 import _lib
    C, D, B, cen, batches = cm_setup()
    cfg = {"workload": "configs[2]: ClusterMemory CM_Hard fwd/bwd bs=256 temp=0.05 momentum=0.2, 700 clusters x 2048-d",
           "B": B, "C": C, "D": D, "l2": "working set 16 MB: L2 resident by nature (latency-bound stage)"}
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:                                   # ClusterMemory stays single-GPU (north_star)
        return
    if args.impl == "reference":
        from oracle import ref_shim
        on_gpu = torch.cuda.is_available() and ref_shim.available()
        ts = []
        if on_gpu:
            dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
            torch.cuda.set_device(dev)
            mem = ref_shim.load_cm().ClusterMemory(D, C, temp=0.05, momentum=0.2, use_hard=True).to(dev)
            mem.features = cen.to(dev).clone()
            dbat = [(a.to(dev), b.to(dev)) for a, b in batches]
            for i in range(args.warmup + args.steps):
                inp, tgt = dbat[i % 8]
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                loss = mem(inp.detach().requires_grad_(True), tgt).mean()
                loss.backward()
                torch.cuda.synchronize()
                if i >= args.warmup:
                    ts.append(time.perf_counter() - t0)
            kind, what = "reference", "unmodified clustercontrast/models/cm.py ClusterMemory(use_hard=True) on cuda:0 (torch ops + 256 .cpu() syncs per backward)"
        else:
            from oracle import memory as omem
            f = cen.numpy().copy()
            for i in range(args.warmup + args.steps):
                inp, tgt = batches[i % len(batches)]
                t0 = time.perf_counter()
                loss, z, xhat, nrm = omem.cm_forward(inp.numpy(), tgt.numpy(), f, 0.05)
                omem.cm_backward(np.full(B, 1.0 / B, np.float32), z, tgt.numpy(), f, xhat, nrm, 0.05)
                f, _ = omem.cm_hard_update(f, xhat, tgt.numpy(), 0.2)
                if i >= args.warmup:
                    ts.append(time.perf_counter() - t0)
            kind, what = "port", "numpy oracle of cm.py on the host cores"
        v = sum(ts) / len(ts)
        print(json.dumps({"impl": "reference", "metric": CM_METRIC, "value": v, "unit": "s",
                          "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": v * 1e3,
                          "higher_is_better": False, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                          "config": dict(cfg, reference=what),
                          "cpu_baseline": {"value": v, "unit": "s", "cores": os.cpu_count(), "kind": kind, "sample": "every step"},
                          "e2e": {"value": v, "unit": "s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    mem = rg.ClusterMemory(D, C, temp=0.05, momentum=0.2, use_hard=True).to(dev)
    mem.features = cen.to(dev).clone()
    dbat = [(a.to(dev), b.to(dev)) for a, b in batches]
    hbat = [(a.pin_memory(), b.pin_memory()) for a, b in batches]

    def step(inp, tgt):
        """One step; returns the mean loss, the per-sample losses and the inputs, whose .grad the backward filled."""
        inp = inp.requires_grad_(True)
        loss = mem(inp, tgt)
        mean = loss.mean()
        mean.backward()
        return mean, loss, inp

    sampler = ClockSampler(dev.index or 0)
    sampler.start()
    for i in range(max(args.warmup, 3)):
        step(*dbat[i % 8])
    torch.cuda.synchronize()
    steps = args.steps                               # a step lasts tens of microseconds: --steps in the hundreds times enough
    l0 = _lib.launch_count()
    _lib.profiler.start()
    for i in range(8):
        step(dbat[i % 8][0].detach(), dbat[i % 8][1])
    torch.cuda.synchronize()
    _lib.profiler.stop()
    prof = _lib.profiler.summary()
    launches = (_lib.launch_count() - l0) // 8
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        _, loss, inp = step(dbat[i % 8][0].detach(), dbat[i % 8][1])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    if args.dump_outputs:                            # before the end-to-end steps move the centroids on
        dumped = host_outputs({"loss": loss, "input_grad": inp.grad, "features": mem.features})
    t0 = time.perf_counter()
    for i in range(steps):
        a, b = hbat[i % 8]
        lv = float(step(a.to(dev, non_blocking=True), b.to(dev, non_blocking=True))[0].item())
    e2e_s = (time.perf_counter() - t0) / steps
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dumped)
    peaks = measured_peaks()
    nbytes = 4.0 * (2 * B * D + 2 * C * D + B * C)
    kernel_ms = {k: round(v[1] / 8, 5) for k, v in sorted(prof.items(), key=lambda kv: -kv[1][1])}
    dev_ms = sum(kernel_ms.values())
    # reference cm_hard on the same GPU, same batches (oracle/_ref): reported beside ours, not a gate
    ref_ms = None
    try:
        from oracle import ref_shim
        if ref_shim.available():
            rmem = ref_shim.load_cm().ClusterMemory(D, C, temp=0.05, momentum=0.2, use_hard=True).to(dev)
            rmem.features = cen.to(dev).clone()
            rts = []
            for i in range(3 + 10):
                inp, tgt = dbat[i % 8]
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                rmem(inp.detach().requires_grad_(True), tgt).mean().backward()
                torch.cuda.synchronize()
                if i >= 3:
                    rts.append(time.perf_counter() - t0)
            ref_ms = 1e3 * sum(rts) / len(rts)
    except Exception as e:                            # reporting only
        ref_ms = "unavailable: %r" % (e,)
    print(json.dumps({"metric": CM_METRIC, "value": ms * 1e-3, "unit": "s", "n_gpus": 1,
                      "steps": steps, "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": False,
                      "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg, "clocks": clocks,
                      "e2e": {"value": e2e_s, "unit": "s", "h2d_bytes_per_step": B * D * 4 + B * 8, "d2h_bytes_per_step": 4},
                      "gpu_launches": int(launches),
                      "roofline": {"kernel": "reid_cm_* (%d launches)" % launches, "bound": "hbm",
                                   "achieved": nbytes / (ms * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                   "frac": nbytes / (ms * 1e-3) / 1e9 / peaks["hbm_gbs"], "traffic": None,
                                   "device_ms_in_kernels": round(dev_ms, 5),
                                   "note": "latency bound: 16 MB and 1.5 GFLOP per step (roofline ~2-3 us); read ms_per_step (step through "
                                           "autograd, host-launch bound), device_ms_in_kernels (CUDA events around our launches) and gpu_launches"},
                      "kernel_ms": kernel_ms,
                      "reference_cm_hard_on_this_gpu_ms": ref_ms,
                      "loss": lv}))


# ------------------------------------------------------------------ GPU arm ------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", type=int, default=None, help="override N (development only; invalidates the metric)")
    ap.add_argument("--knn", default="auto")
    ap.add_argument("--ref-kind", default="auto", choices=["auto", "_ref", "port"],
                    help="reference arm: the reference's own files (oracle/_ref) or the oracle's numpy port")
    ap.add_argument("--ref-budget-s", type=float, default=240.0, help="wall-time cap of the reference arm's passes")
    ap.add_argument("--cpu-baseline", default="port", choices=["port", "_ref", "auto", "none"],
                    help="the cpu_baseline leg of OUR line (one full-size pass on the host cores, N=1 only)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="enqueue every pass eagerly instead of replaying a CUDA graph")
    ap.add_argument("--workload", default="rerank", choices=["cm"] + list(WORKLOADS),
                    help="rerank = BASELINE configs[1] (the headline); cm = configs[2]; pass = configs[3]; "
                         "market = configs[0]; scale100k / scale250k = configs[4]; hard = the parity set")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the outputs of the last one as DIR/<name>.npy (float32 / float64, "
                         "at most 64 MB in all; larger outputs as a fixed, seeded sample of rows)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path; it does not apply to --impl reference")
    args.warmup = max(args.warmup, 0)
    pin_host_threads()
    if args.workload == "cm":
        return run_cm(args)
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import reid_gan_b200 as rg
    from reid_gan_b200 import _lib, pipeline

    W = workload(args)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus %d needs torchrun with %d ranks (WORLD_SIZE=%d)" % (args.gpus, args.gpus, world))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
        from reid_gan_b200 import sharded

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # synthetic features: generated on the host (seeded; same bytes on every box), kept in pinned memory for the e2e
    # leg.  The scale workloads generate on the device (the host generator would take longer than the run).
    if W["gen"] == "synth_device":
        x_dev, _ = rg.synth_device(W["N"], W["D"], W["n_ids"], W["noise"], W["seed"], device=dev)
        x_host = torch.empty(x_dev.shape, dtype=torch.float32).pin_memory()
        x_host.copy_(x_dev)
    else:
        import importlib
        x_host = getattr(importlib.import_module("reid_gan_b200.synth"), W["gen"])(**synth_args(W))[0]
        x_host = x_host.pin_memory()
        x_dev = x_host.to(dev, non_blocking=True)
    torch.cuda.synchronize()

    use_graph = not args.no_graph

    def one_pass(timers=False, graph=None):
        graph = use_graph if graph is None else graph
        if world > 1:
            return sharded.pseudo_labels(x_dev, W["k1"], W["k2"], W["eps"], W["min_samples"], knn=args.knn,
                                         centroids=W["centroids"], graph=graph)
        return pipeline.pseudo_labels(x_dev, W["k1"], W["k2"], W["eps"], W["min_samples"], knn=args.knn, timers=timers,
                                      centroids=W["centroids"], graph=graph)

    sampler = ClockSampler(local_rank)
    if rank == 0:                       # nvidia-smi needs a few hundred ms to start: begin before the warm-up and
        sampler.start()                 # keep the GPU busy until the first sample has arrived
        t_wait = time.time()
        while world == 1 and not sampler.rows and time.time() - t_wait < 3.0:
            one_pass()
    for _ in range(max(args.warmup, 3) + (10 if world > 1 else 0)):
        out = one_pass()
    barrier()
    # ---- timed region: K passes, CUDA events on the launching stream, no profiling hooks --------------------
    barrier()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        out = one_pass()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1) / args.steps
    if dist is not None:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:                     # `out` is still the last timed pass
        dump_outputs(args.dump_outputs, host_outputs(pass_outputs(out)))
    # ---- per-entry-point CUDA-event times (separate passes: the event pairs cost a few microseconds per launch) ----
    p_steps = max(3, min(args.steps, 10))
    l0 = _lib.launch_count()
    _lib.profiler.start()
    barrier()
    for _ in range(p_steps):
        out = one_pass(graph=False)                          # eager: the event pairs bracket the individual entry points
    barrier()
    _lib.profiler.stop()
    # kernels of OUR library per pass, counted where they are launched one by one (the timed passes replay the same
    # sequence from a CUDA graph, which the host-side counter does not see)
    launches = (_lib.launch_count() - l0) // p_steps
    prof = _lib.profiler.summary()
    labels = out["labels"]
    ncl = int(out["num_clusters"].item())
    info = out["state"].knn_info if "state" in out else {}
    lab_np = labels.cpu().numpy()
    digests = {"labels_sha256": labels_sha256(lab_np), "rank_sha256": rank_sha256(out["state"].rank.cpu().numpy())}

    # ---- end to end through the drop-in API: pinned host features -> host labels ------------
    e2e = None
    if not args.no_e2e:
        def e2e_pass():
            if world > 1:
                return sharded.pseudo_labels_host(x_host, W["k1"], W["k2"], W["eps"], W["min_samples"], knn=args.knn)
            d = rg.compute_jaccard_distance(x_host, k1=W["k1"], k2=W["k2"], print_flag=False, search_option=3,
                                            knn=args.knn)
            e2e_pass.info = d.state.knn_info
            lab = rg.DBSCAN(eps=W["eps"], min_samples=W["min_samples"], metric="precomputed", n_jobs=-1).fit_predict(d)
            if W["centroids"]:
                e2e_pass.cen = rg.generate_cluster_features(lab, d.state.x if hasattr(d.state, "x") else x_dev, normalize=True)
            return lab
        for _ in range(2):
            lab_host = e2e_pass()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            lab_host = e2e_pass()
        barrier()
        e2e_s = (time.perf_counter() - t0) / args.steps
        if dist is not None:
            t = torch.tensor([e2e_s], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e_s = float(t.item())
        digests["e2e_labels_sha256"] = labels_sha256(lab_host)
        extra = 0
        if world == 1:                      # the streamed search uploads its threshold sample ahead of the bulk
            extra = int(((getattr(e2e_pass, "info", None) or {}).get("sym") or {}).get("sample", 0)) * W["D"] * 4
        e2e = {"value": e2e_s, "unit": "s", "h2d_bytes_per_step": int(W["N"] * W["D"] * 4 // world) + extra,
               "d2h_bytes_per_step": int(W["N"] * 9)}

    def shutdown():
        """Graphs that hold NCCL kernels must be released before the communicator (destroying it with live graphs can
        hang); a watchdog ends the process if the teardown still does not return."""
        if dist is None:
            return
        sys.stdout.flush()
        threading.Timer(20.0, lambda: os._exit(0)).start()
        pipeline.PassGraph._cache.clear()
        torch.cuda.synchronize()
        dist.barrier()
        dist.destroy_process_group()
        os._exit(0)

    if rank != 0:
        shutdown()
        return

    # ---- roofline of the dominant kernel (tcgen05 similarity GEMM + fused top-K) -------------
    peaks = measured_peaks()
    n_rows = W["N"] // world + (1 if W["N"] % world else 0)
    flops = 2.0 * n_rows * W["N"] * W["D"]               # algorithmic: 2*N^2*D, symmetry not credited (SURVEY 8d)
    roof = None
    sym_key = next((k_ for k_ in ("reid_knn_candidates_sym_wide", "reid_knn_candidates_sym") if k_ in prof), None)
    if sym_key:
        # symmetric search: the dominant kernel executes only the tiles (I <= J); `achieved` counts the flops it
        # really issues (tiles * 2*256*256*D, padding included), `algorithmic_tflops` credits the 2*N^2*D of SURVEY 8(d)
        # to the whole candidate stage (prepass + main pass).
        calls, tot_ms = prof[sym_key]
        k_ms = tot_ms / calls
        n_tiles = (info.get("sym") or {}).get("tiles", 0)
        exec_flops = 2.0 * 256 * 256 * W["D"] * n_tiles
        pre_ms = sum(prof[k_][1] for k_ in ("reid_knn_candidates_tc_ab", "reid_knn_candidates_tc_abt") if k_ in prof) / max(calls, 1)
        ach = exec_flops / (k_ms * 1e-3) / 1e12
        roof = {"kernel": "simsym_kernel<%d> (%s)" % (2 if sym_key.endswith("wide") else 1, sym_key), "bound": "tensor", "achieved": ach,
                "peak": peaks["bf16_tflops"], "unit": "TFLOP/s", "frac": ach / peaks["bf16_tflops"],
                # dram__bytes_read.sum + dram__bytes_write.sum of one launch, `ncu --set full` capture of this
                # workload on one GPU: sample-first layout, 7,260 tiles (profiles/r02_v4_summary.txt: 455 MB read + 57 MB
                # written); all 8,256 tiles (profiles/r02_v3_summary.txt): 523 + 65 MB; the fp16 operand alone is 134 MB
                "traffic": ((512.2e6 if (info.get("sym") or {}).get("layout") == "sample-first" else 587.6e6)
                            if (world == 1 and W["N"] == WORKLOAD["N"]) else None),
                "ms_per_launch": k_ms, "flops_per_launch": exec_flops,
                "algorithmic_flops": flops, "algorithmic_tflops": flops / ((k_ms + pre_ms) * 1e-3) / 1e12,
                "prepass_ms": pre_ms,
                "peak_source": peaks["source"] + " cuBLAS bf16 burst (kernel lasts a few ms)"}
    elif "reid_knn_candidates_tc" in prof:
        calls, tot_ms = prof["reid_knn_candidates_tc"]
        k_ms = tot_ms / calls
        ach = flops / (k_ms * 1e-3) / 1e12
        roof = {"kernel": "simtopk_kernel (reid_knn_candidates_tc)", "bound": "tensor", "achieved": ach,
                "peak": peaks["bf16_tflops"], "unit": "TFLOP/s", "frac": ach / peaks["bf16_tflops"],
                "traffic": None, "ms_per_launch": k_ms, "flops_per_launch": flops,
                "peak_source": peaks["source"] + " cuBLAS bf16 burst (kernel lasts a few ms)"}
    stage_ms = {k: round(v[1] / p_steps, 4) for k, v in sorted(prof.items(), key=lambda kv: -kv[1][1])}
    try:
        stages = stage_rooflines(out, W, prof, p_steps, peaks, world)
    except Exception as e:                                   # reporting only: never fail the bench line on it
        stages = [{"error": repr(e)}]

    cpu = None
    if not args.no_cpu_baseline and args.cpu_baseline != "none" and world == 1 and W["gen"] != "synth_device":
        # one FULL-size pass of the CPU path on this box's host cores (no sample, no scaling); its labels digest must
        # equal ours -- the parity statement of this very run
        cpu = cpu_reference_pass(W, args.cpu_baseline, x=x_host)
        cpu["labels_match_gpu"] = cpu["labels_sha256"] == digests["labels_sha256"]
        cpu["rank_match_gpu"] = cpu["rank_sha256"] == digests["rank_sha256"]

    line = {"metric": W["metric"], "value": ms * 1e-3, "unit": "s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": False, "scaling": "strong",
            "vs_baseline": None, "dtype": "f16 tensor-core candidates, f64-accumulated f32 keys, f32 weights",
            "data": "synthetic",
            "config": {"workload": W["name"], **{k: W[k] for k in W if k not in ("metric", "name")},
                       "parallelism": "rows partitioned over %d GPU(s)" % world,
                       "launch": "one CUDA graph per pass (captured once, replayed)" if use_graph else "eager launches",
                       "l2": "inputs (%.0f MB fp32 + %.0f MB fp16) exceed the 126 MB L2; no flush needed"
                             % (W["N"] * W["D"] * 4 / 1e6, W["N"] * W["D"] * 2 / 1e6),
                       "knn": info.get("mode"), "knn_splits": info.get("n_splits"), "knn_keep": info.get("keep"),
                       "uncertified_rows": info.get("uncertified_rows"), "clusters": ncl,
                       "noise_points": int((labels < 0).sum().item()), **digests},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roof, "cpu_baseline": cpu,
            "stage_ms": stage_ms, "stages": stages}
    print(json.dumps(line))
    shutdown()


if __name__ == "__main__":
    main()
