"""CPU: the entry points of the sample block column in the sample-first symmetric search (reid_knn_tau_floor,
reid_knn_candidates_sym_tiles, reid_knn_list_tau) reject bad arguments before any CUDA call; the tile list covers the
block column exactly once."""
import ctypes

import pytest


@pytest.fixture
def lib_and_ptr():
    from reid_gan_b200 import _lib
    buf = (ctypes.c_int64 * 16)()
    return _lib, _lib.lib(), (ctypes.addressof(buf) + 15) & ~15


def test_tau_floor_arguments(lib_and_ptr):
    _lib, L, a = lib_and_ptr
    assert L.reid_knn_tau_floor(None, a, 1024, 8192, None) == _lib.REID_ERR_INVALID_ARG
    assert "NULL" in _lib.last_error()
    for m, N in ((0, 8192), (-5, 8192), (8193, 8192)):
        rc = L.reid_knn_tau_floor(a, a, m, N, None)
        assert rc == _lib.REID_ERR_INVALID_ARG and "m <= N" in _lib.last_error(), (m, N)
    assert L.reid_knn_tau_floor(a, a, 8192, 8192, None) == _lib.REID_OK        # no rows outside the sample: no launch


def test_list_tau_arguments(lib_and_ptr):
    _lib, L, a = lib_and_ptr
    assert L.reid_knn_list_tau(a, None, 1024, 1024, 10, 16, a, a, None) == _lib.REID_ERR_INVALID_ARG
    assert "NULL" in _lib.last_error()
    for cap, row0, n_rows, r in ((0, 1024, 10, 16), (1024, -1, 10, 16), (1024, 1024, -1, 16), (1024, 1024, 10, 0)):
        rc = L.reid_knn_list_tau(a, a, cap, row0, n_rows, r, a, a, None)
        assert rc == _lib.REID_ERR_INVALID_ARG and "bad arguments" in _lib.last_error(), (cap, row0, n_rows, r)
    assert L.reid_knn_list_tau(a, a, 1024, 1024, 0, 16, a, a, None) == _lib.REID_OK


def test_sym_tiles_arguments(lib_and_ptr):
    _lib, L, a = lib_and_ptr
    rc = L.reid_knn_candidates_sym_tiles(a, 8192, 128, 4, None, a, 4, 1024, a, a, 0, None)
    assert rc == _lib.REID_ERR_INVALID_ARG and "NULL" in _lib.last_error()
    rc = L.reid_knn_candidates_sym_tiles(a, 8192, 100, 4, a, a, 4, 1024, a, a, 0, None)
    assert rc == _lib.REID_ERR_INVALID_ARG and "D %" in _lib.last_error()
    rc = L.reid_knn_candidates_sym_tiles(a, 8192, 128, 4, a, a, 0, 1024, a, a, 0, None)
    assert rc == _lib.REID_ERR_INVALID_ARG and "tile list" in _lib.last_error()


@pytest.mark.parametrize("n_t,s_t", [(33, 4), (128, 8), (5, 4)])
def test_sample_block_tiles(n_t, s_t):
    """(I, J) with I < s_t <= J, each once, column block by column block."""
    from reid_gan_b200 import knn_tc
    t = knn_tc._sample_block_tiles(n_t, s_t, "cpu").tolist()
    assert sorted(map(tuple, t)) == [(i, j) for i in range(s_t) for j in range(s_t, n_t)]
    assert [j for _, j in t] == sorted(j for _, j in t)
