"""CPU: the C entries of the feature-based evaluation re-ranking validate their arguments before any CUDA call, the
public signatures follow the reference's evaluators.py, and nothing falls back to the CPU."""
import ctypes
import inspect

import numpy as np
import pytest
import torch


def _buf():
    b = (ctypes.c_int64 * 64)()
    return b, ctypes.addressof(b)


def _rejects(rc, what):
    from reid_gan_b200 import _lib
    assert rc == _lib.REID_ERR_INVALID_ARG
    assert what in _lib.last_error(), _lib.last_error()


def test_row_sqnorm64_argument_validation():
    from reid_gan_b200 import _lib
    L = _lib.lib()
    _b, a = _buf()
    _rejects(L.reid_rr_row_sqnorm64(None, 4, 8, a, None), "NULL")
    _rejects(L.reid_rr_row_sqnorm64(a, 4, 8, None, None), "NULL")
    _rejects(L.reid_rr_row_sqnorm64(a, 0, 8, a, None), "bad shape")
    _rejects(L.reid_rr_row_sqnorm64(a, 4, 0, a, None), "bad shape")


def test_farthest_certify_argument_validation():
    from reid_gan_b200 import _lib
    L = _lib.lib()
    _b, a = _buf()

    def certify(x=a, M=100, D=64, cand=a, n_lists=2, cap=512, r0=0, r1=100, colmax=a, flag=a):
        return L.reid_rr_farthest_certify(x, M, D, a, cand, a, a, n_lists, cap, r0, r1, a, colmax, flag, None, None)

    for kw, what in [(dict(x=None), "NULL"), (dict(cand=None), "NULL"), (dict(colmax=None), "NULL"), (dict(flag=None), "NULL"),
                     (dict(r1=101), "bad shape"), (dict(r0=5, r1=5), "bad shape"), (dict(r0=-1), "bad shape"),
                     (dict(D=0), "bad shape"), (dict(n_lists=0), "n_lists"), (dict(n_lists=9), "n_lists"),
                     (dict(cap=0), "list_cap")]:
        _rejects(certify(**kw), what)


def test_farthest_exact_argument_validation():
    from reid_gan_b200 import _lib
    L = _lib.lib()
    _b, a = _buf()
    _rejects(L.reid_rr_farthest_exact(None, 10, 8, a, None, 0, 10, a, None), "NULL")
    _rejects(L.reid_rr_farthest_exact(a, 10, 8, None, None, 0, 10, a, None), "NULL")
    _rejects(L.reid_rr_farthest_exact(a, 10, 8, a, None, 0, 10, None, None), "NULL")
    _rejects(L.reid_rr_farthest_exact(a, 10, 8, a, None, 5, 6, a, None), "bad shape")
    _rejects(L.reid_rr_farthest_exact(a, 10, 8, a, None, 0, -1, a, None), "bad shape")
    _rejects(L.reid_rr_farthest_exact(a, 10, 60000, a, a, 0, 10, a, None), "too large")
    assert L.reid_rr_farthest_exact(a, 10, 8, a, a, 0, 0, a, None) == _lib.REID_OK      # nothing to do, no CUDA call


def test_weights_features_argument_validation():
    from reid_gan_b200 import _lib
    L = _lib.lib()
    _b, a = _buf()

    def w(x=a, colmax=a, e_pad=a, stride=8, n=10, M=10):
        return L.reid_rr_weights_features(x, M, 16, a, colmax, e_pad, stride, a, n, a, a, None)

    for kw, what in [(dict(x=None), "NULL"), (dict(colmax=None), "NULL"), (dict(e_pad=None), "NULL"),
                     (dict(stride=0), "bad shape"), (dict(n=11), "bad shape"), (dict(n=-1), "bad shape")]:
        _rejects(w(**kw), what)


def test_final_qg_argument_validation():
    from reid_gan_b200 import _lib
    L = _lib.lib()
    _b, a = _buf()

    def f(J=a, ldJ=30, qg=a, colmax=a, Q=10, G=20, r0=0, r1=10, out=a):
        return L.reid_rr_final_qg(J, ldJ, qg, colmax, Q, G, r0, r1, 0.7, 0.3, out, None)

    for kw, what in [(dict(J=None), "NULL"), (dict(qg=None), "NULL"), (dict(colmax=None), "NULL"), (dict(out=None), "NULL"),
                     (dict(ldJ=29), "bad shape"), (dict(r1=11), "bad shape"), (dict(r0=4, r1=4), "bad shape"),
                     (dict(Q=0, r1=0), "bad shape")]:
        _rejects(f(**kw), what)


@pytest.mark.parametrize("k1,k2", [(64, 6), (0, 1), (20, 22), (20, 0)])
def test_re_ranking_features_rejects_k_before_any_device(k1, k2):
    import reid_gan_b200 as rg
    x = np.zeros((4, 8), np.float32)
    with pytest.raises(ValueError):
        rg.re_ranking_features(x, x, k1=k1, k2=k2)


def test_signatures():
    import reid_gan_b200 as rg
    from reid_gan_b200 import evaluators
    assert rg.evaluate_all is evaluators.evaluate_all and rg.Evaluator is evaluators.Evaluator
    p = inspect.signature(rg.re_ranking_features).parameters
    assert list(p) == ["query_features", "gallery_features", "k1", "k2", "lambda_value", "return_device"]
    assert [p[n].default for n in ("k1", "k2", "lambda_value", "return_device")] == [20, 6, 0.3, False]
    p = inspect.signature(rg.evaluate_all).parameters
    assert list(p) == ["query_features", "gallery_features", "distmat", "query", "gallery", "query_ids", "gallery_ids",
                       "query_cams", "gallery_cams", "cmc_topk", "cmc_flag"]
    assert p["cmc_topk"].default == (1, 5, 10) and p["cmc_flag"].default is False
    assert all(p[n].default is None for n in ("query", "gallery", "query_ids", "gallery_ids", "query_cams", "gallery_cams"))
    p = inspect.signature(rg.Evaluator.evaluate).parameters
    assert list(p) == ["self", "data_loader", "query", "gallery", "cmc_flag", "rerank"]
    assert p["cmc_flag"].default is False and p["rerank"].default is False
    assert list(inspect.signature(rg.Evaluator.__init__).parameters) == ["self", "model"]
    for name in ("re_ranking_features", "Evaluator", "evaluate_all"):
        assert name in rg.__all__


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_no_cpu_fallback():
    import reid_gan_b200 as rg
    from reid_gan_b200.rerank import farthest_colmax
    x = np.random.default_rng(0).standard_normal((40, 16)).astype(np.float32)
    with pytest.raises(RuntimeError):
        rg.re_ranking_features(x[:10], x[10:], k1=5, k2=2)
    with pytest.raises(RuntimeError):
        rg.re_ranking_features(torch.from_numpy(x[:10]), torch.from_numpy(x[10:]), k1=5, k2=2)
    ids = list(range(10))
    with pytest.raises(RuntimeError):
        rg.evaluate_all(None, None, x[:10, :10], query_ids=ids, gallery_ids=ids, query_cams=[0] * 10, gallery_cams=[1] * 10)
    with pytest.raises(RuntimeError):
        rg.Evaluator(torch.nn.Identity()).evaluate([(torch.from_numpy(x[:4]), ["a", "b", "c", "d"], [0, 1, 0, 1], [0] * 4, 0)],
                                                   [("a", 0, 0)], [("b", 1, 0)])
    with pytest.raises(RuntimeError):
        farthest_colmax(torch.from_numpy(x))
