"""ctypes binding of libreid_b200.so (include/reid_b200.h).

The library is the product: if it is missing or a call fails there is NO fallback --
`lib()` raises and every wrapper turns a non-zero return code into an exception
(REID_ERR_INVALID_ARG -> ValueError, everything else -> RuntimeError), mirroring the
reference's assert/exception-only error convention (utils/faiss_utils.py:7-8,13-14,22-24).
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libreid_b200.so")

REID_OK = 0
REID_ERR_INVALID_ARG = -1
REID_ERR_CUDA = -2
REID_ERR_NCCL = -3
REID_ERR_CERTIFICATE = -4
REID_ERR_UNSUPPORTED = -5

_P = ctypes.c_void_p
_I = ctypes.c_int
_L = ctypes.c_int64
_F = ctypes.c_float
_Z = ctypes.c_size_t

# name -> (restype, argtypes); must list every symbol declared in include/reid_b200.h
SIGNATURES = {
    "reid_abi_version": (_I, []),
    "reid_last_error": (ctypes.c_char_p, []),
    "reid_launch_count": (ctypes.c_uint64, []),
    "reid_scan_counts": (_I, [_P, _L, _P, _P, _P]),
    "reid_knn_exact_scratch_bytes": (_Z, [_L, _L]),
    "reid_knn_exact": (_I, [_P, _L, _L, _P, _L, _L, _I, _P, _P, _P, _Z, _P]),
    "reid_sqnorm_range": (_I, [_P, _L, _L, _P, _P]),
    "reid_knn_exact_l2": (_I, [_P, _L, _L, _P, _L, _L, _I, _P, _P, _P, _Z, _P]),
    "reid_knn_tc_plan": (_I, [_L, _L, _I, _P]),
    "reid_knn_candidates_tc": (_I, [_P, _L, _L, _I, _L, _L, _I, _I, _I, _P, _P, _P, _P]),
    "reid_features_to_half": (_I, [_P, _L, _L, _I, _P, _P, _P]),
    "reid_sqnorm_range_reset": (_I, [_P, _P]),
    "reid_knn_rescore_workspace_bytes": (_Z, [_L, _L]),
    "reid_knn_rescore_window_counts_offset": (_Z, [_L, _L]),
    "reid_knn_rescore": (_I, [_P, _L, _L, _L, _L, _P, _P, _P, _I, _I, _L, _I, _F, _P, _I, _P, _P, _P, _P, _P, _P, _P]),
    "reid_knn_candidates_tc_ab": (_I, [_P, _L, _P, _L, _L, _I, _L, _L, _I, _I, _I, _P, _P, _P, _P]),
    "reid_knn_candidates_sym": (_I, [_P, _L, _L, _I, _P, _P, _L, _I, _P, _P, _I, _P]),
    "reid_knn_candidates_sym_wide": (_I, [_P, _L, _L, _I, _P, _P, _L, _I, _P, _P, _I, _P]),
    "reid_upload_rows_strided": (_I, [_P, _P, _Z, _Z, _L, _P]),
    "reid_features_to_half_acc": (_I, [_P, _L, _L, _I, _P, _P, _P]),
    "reid_features_sample": (_I, [_P, _L, _L, _L, _L, _P, _P]),
    "reid_knn_sample_tau": (_I, [_P, _P, _P, _I, _L, _I, _P, _P, _P]),
    "reid_knn_sample_tau_emit": (_I, [_P, _P, _P, _I, _L, _I, _P, _P, _P, _P, _I, _L, _P]),
    "reid_features_to_half_gather": (_I, [_P, _P, _L, _L, _I, _P, _P, _P]),
    "reid_knn_candidates_tc_abt": (_I, [_P, _L, _P, _L, _L, _I, _L, _L, _I, _I, _I, _P, _P, _P, _I, _P, _P, _P, _I, _P]),
    "reid_knn_candidates_sym_tiles": (_I, [_P, _L, _L, _I, _P, _P, _L, _I, _P, _P, _I, _P]),
    "reid_knn_tau_floor": (_I, [_P, _P, _L, _L, _P]),
    "reid_knn_list_tau": (_I, [_P, _P, _I, _L, _L, _I, _P, _P, _P]),
    "reid_knn_rescore_mapped": (_I, [_P, _L, _L, _L, _L, _P, _P, _P, _I, _I, _L, _I, _F, _P, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "reid_reciprocal_masks": (_I, [_P, _L, _I, _I, _L, _L, _P, _P]),
    "reid_reciprocal_masks2": (_I, [_P, _L, _I, _I, _I, _L, _L, _P, _P, _P]),
    "reid_expand": (_I, [_P, _L, _I, _I, _P, _P, _L, _L, _I, _P, _P, _P]),
    "reid_v_weights": (_I, [_P, _L, _L, _P, _I, _P, _L, _L, _P, _P, _I, _P, _P, _P, _I, _P]),
    "reid_knn_rescore_order_offset": (_Z, [_L, _L]),
    "reid_query_expand_stride": (_I, [_I, _I]),
    "reid_query_expand": (_I, [_P, _L, _I, _I, _P, _P, _P, _I, _L, _L, _P, _P, _P, _P, _I, _P]),
    "reid_csr_compact": (_I, [_P, _P, _L, _P, _P, _L, _P, _P, _P]),
    "reid_lists_compact": (_I, [_P, _P, _P, _P, _L, _P, _P]),
    "reid_rows_pack": (_I, [_P, _P, _P, _P, _L, _L, _I, _P, _P]),
    "reid_rows_unpack_counts": (_I, [_P, _I, _I, _I, _L, _P, _L, _P, _P, _P]),
    "reid_rows_unpack_fill": (_I, [_P, _I, _I, _L, _P, _L, _P, _P, _P, _P]),
    "reid_transpose_count": (_I, [_P, _L, _P, _L, _P, _P]),
    "reid_transpose_fill": (_I, [_P, _P, _P, _L, _L, _P, _P, _P, _P, _I, _P]),
    "reid_jaccard_bounds": (_I, [_P, _P, _P, _P, _L, _L, _F, _P, _P, _P, _P]),
    "reid_jaccard_neighbors": (_I, [_P, _P, _P, _P, _P, _P, _L, _L, _L, _P, _L, _F, _P, _P, _P, _P, _I, _P]),
    "reid_jaccard_neighbors_heavy": (_I, [_P, _P, _P, _P, _P, _P, _L, _L, _P, _L, _F, _P, _P, _P, _P, _P, _P]),
    "reid_jaccard_eps_graph_workspace_bytes": (ctypes.c_size_t, [_L, _L]),
    "reid_jaccard_eps_graph": (_I, [_P, _P, _P, _P, _P, _P, _L, _L, _L, _F, _P, _P, _P, _P, _P, _P, _L, _P, _I, _I, _P, _P, _P]),
    "reid_rr_normalised_distance": (_I, [_P, _P, _P, _L, _L, _P, _P, _P, _P]),
    "reid_rr_weights": (_I, [_P, _L, _P, _I, _P, _L, _P, _P, _P]),
    "reid_rr_final": (_I, [_P, _L, _P, _L, _L, _F, _F, _P, _P]),
    "reid_rr_row_sqnorm64": (_I, [_P, _L, _L, _P, _P]),
    "reid_rr_farthest_certify": (_I, [_P, _L, _L, _P, _P, _P, _P, _I, _I, _L, _L, _P, _P, _P, _P, _P]),
    "reid_rr_farthest_exact": (_I, [_P, _L, _L, _P, _P, _L, _L, _P, _P]),
    "reid_rr_weights_features": (_I, [_P, _L, _L, _P, _P, _P, _I, _P, _L, _P, _P, _P]),
    "reid_rr_final_qg": (_I, [_P, _L, _P, _P, _L, _L, _L, _L, _F, _F, _P, _P]),
    "reid_select_rows": (_I, [_P, _L, _L, _I, _I, _P, _P, _P]),
    "reid_pairwise_distance": (_I, [_P, _P, _L, _L, _L, _P, _P, _P]),
    "reid_rank_metrics_smem_bytes": (_Z, [_L]),
    "reid_rank_metrics": (_I, [_P, _L, _L, _L, _P, _P, _P, _P, _I, _I, _I, _P, _P, _P, _P, _P]),
    "reid_links_count": (_I, [_P, _P, _L, _I, ctypes.c_double, _P, _P]),
    "reid_links_fill": (_I, [_P, _P, _L, _I, ctypes.c_double, _P, _P, _P, _P]),
    "reid_jaccard_dense": (_I, [_P, _P, _P, _P, _P, _P, _L, _L, _L, _P, _L, _I, _P]),
    "reid_dbscan_dense_count": (_I, [_P, _L, _L, _F, _L, _L, _P, _P]),
    "reid_dbscan_dense_fill": (_I, [_P, _L, _L, _F, _L, _L, _P, _P, _P]),
    "reid_dbscan_workspace_bytes": (_Z, [_L]),
    "reid_dbscan_labels": (_I, [_L, _P, _P, _P, _I, _P, _P, _P, _P, _I, _P]),
    "reid_centroids_workspace_bytes": (_Z, [_L, _L]),
    "reid_centroids": (_I, [_P, _L, _L, _P, _L, _I, _P, _P, _P]),
    "reid_peer_push_lists": (_I, [_P, _P, _I, _L, _I, _I, _P, _L, _P]),
    "reid_peer_push_records": (_I, [_P, _P, _P, _P, _L, _L, _I, _I, _I, _P, _L, _P]),
    "reid_peer_allgather": (_I, [_P, _L, _I, _I, _P, _L, _P]),
    "reid_peer_scatter_rows": (_I, [_P, _L, _L, _P, _L, _I, _P, _L, _P, _P]),
    "reid_cmc_reduce": (_I, [_P, _L, _I, _P, _P]),
    "reid_gather_rows": (_I, [_P, _L, _P, _L, _L, _P, _P]),
    "reid_centroids_dev": (_I, [_P, _L, _L, _P, _P, _L, _I, _P, _P, _P]),
    "reid_cm_forward_scratch_bytes": (_Z, [_L, _L, _L]),
    "reid_cm_forward": (_I, [_P, _P, _P, _L, _L, _L, _F, _P, _P, _P, _P, _P, _P]),
    "reid_cm_backward": (_I, [_P, _P, _P, _P, _P, _P, _L, _L, _L, _F, _P, _P, _P]),
    "reid_cm_logits": (_I, [_P, _P, _L, _L, _L, _P, _P]),
    "reid_cm_grad_inputs": (_I, [_P, _P, _L, _L, _L, _P, _P]),
    "reid_cm_update": (_I, [_P, _P, _P, _L, _L, _L, _F, _I, _P, _P]),
    "reid_cm_forward_push": (_I, [_P, _P, _P, _L, _L, _L, _F, _L, _P, _P, _P, _P, _P, _I, _I, _L, _P, _P]),
}

_lib = None


def lib():
    """Load libreid_b200.so (once).  Raises if it has not been built -- there is no CPU path."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError(
                "libreid_b200.so not found at %s: build it with `python -c \"import __graft_entry__ as g; g.build()\"` "
                "(or reid-gan_b200/csrc/build.sh).  This package has no CPU fallback." % LIB_PATH)
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def last_error():
    msg = lib().reid_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def check(rc, what=""):
    if rc == REID_OK:
        return
    msg = "%s failed (%d): %s" % (what or "libreid_b200 call", rc, last_error())
    if rc == REID_ERR_INVALID_ARG:
        raise ValueError(msg)
    raise RuntimeError(msg)


class Profiler:
    """Optional per-entry-point device timing (CUDA events on the launching stream) and launch
    counting, used by bench.py for the roofline / gpu_launches fields.  Off by default."""

    def __init__(self):
        self.enabled = False
        self.records = []          # (name, start_event, end_event)

    def start(self):
        self.records = []
        self.enabled = True

    def stop(self):
        self.enabled = False

    def summary(self):
        """{name: (calls, total_ms)} -- call after a device synchronize."""
        out = {}
        for name, e0, e1 in self.records:
            c, t = out.get(name, (0, 0.0))
            out[name] = (c + 1, t + e0.elapsed_time(e1))
        return out


profiler = Profiler()


def call(name, *args):
    """Invoke one C-ABI entry point and raise on a non-zero return code."""
    fn = getattr(lib(), name)
    if profiler.enabled:
        import torch
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        rc = fn(*args)
        e1.record()
        profiler.records.append((name, e0, e1))
    else:
        rc = fn(*args)
    check(rc, name)


def launch_count():
    """Number of kernels libreid_b200.so has launched in this process."""
    return int(lib().reid_launch_count())


def ptr(t):
    """Device (or host) address of a torch tensor / None."""
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def stream_ptr():
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
