"""CPU: distributed evaluation's C entries (reid_peer_scatter_rows, reid_cmc_reduce) validate their arguments before any
CUDA call, eval_shard splits the test images, and DistributedEvaluator's host logic up to the first device call (two
gloo ranks)."""
import ctypes
import inspect
import os
import socket

import pytest
import torch
import torch.multiprocessing as mp


def test_abi_version_and_new_entries():
    """The two entries are additions: the ABI version of the existing entries stays 5."""
    from reid_gan_b200 import _lib
    L = _lib.lib()
    assert L.reid_abi_version() == 5
    assert hasattr(L, "reid_peer_scatter_rows") and hasattr(L, "reid_cmc_reduce")


def test_scatter_rows_argument_validation():
    from reid_gan_b200 import _lib
    L = _lib.lib()
    buf = (ctypes.c_int64 * 64)()
    a = (ctypes.addressof(buf) + 15) & ~15

    def scatter(src=a, n=4, D=8, dst=a, M=10, world=2, base=a, off=0):
        return L.reid_peer_scatter_rows(src, n, D, dst, M, world, base, off, None, None)

    for kw, what in [(dict(src=None), "NULL"), (dict(dst=None), "NULL"), (dict(base=None), "bad arguments"),
                     (dict(D=6), "D=6"), (dict(src=a + 4), "aligned"), (dict(off=8), "aligned"),
                     (dict(world=0), "bad arguments"), (dict(M=0), "bad arguments"), (dict(n=-1), "bad arguments")]:
        rc = scatter(**kw)
        assert rc == _lib.REID_ERR_INVALID_ARG, kw
        assert what in _lib.last_error(), (kw, _lib.last_error())
    assert scatter(n=0, src=None, dst=None) == _lib.REID_OK          # nothing to store: no launch


def test_cmc_reduce_argument_validation():
    from reid_gan_b200 import _lib
    L = _lib.lib()
    buf = (ctypes.c_double * 8)()
    a = ctypes.addressof(buf)
    for args in [(None, 2, 4, a), (a, 2, 4, None), (a, 0, 4, a), (a, 2, 0, a)]:
        assert L.reid_cmc_reduce(*args, None) == _lib.REID_ERR_INVALID_ARG
        assert "reid_cmc_reduce" in _lib.last_error()


def _items(n, offset=0):
    return [("img_%05d.jpg" % (offset + i), (offset + i) % 7, (offset + i) % 3) for i in range(n)]


@pytest.mark.parametrize("overlap", [0, 5])
def test_eval_shard_partitions_the_sorted_union(overlap):
    from reid_gan_b200.evaluators import eval_shard
    from reid_gan_b200.sharded import partition
    gallery = _items(40, 10)
    query = _items(13)[::-1] + gallery[:overlap]                   # unsorted; `overlap` names also in the gallery
    union = sorted({it[0]: it for it in query + gallery}.values())
    assert len(union) == 50
    for world in range(1, 9):
        seen = []
        for rank in range(world):
            share = eval_shard(query, gallery, world=world, rank=rank)
            r0, r1 = partition(len(union), world, rank)
            assert share == union[r0:r1]
            seen += share
        assert seen == union


def test_constructor_is_evaluator_plus_group():
    import reid_gan_b200 as rg
    base = list(inspect.signature(rg.Evaluator.__init__).parameters)
    sig = inspect.signature(rg.DistributedEvaluator.__init__)
    assert list(sig.parameters) == base + ["group"] and sig.parameters["group"].default is None
    assert (list(inspect.signature(rg.DistributedEvaluator.evaluate).parameters)
            == list(inspect.signature(rg.Evaluator.evaluate).parameters))
    assert issubclass(rg.DistributedEvaluator, rg.Evaluator)
    ev = rg.DistributedEvaluator(torch.nn.Identity())
    assert ev.group is None


def test_destination_table():
    from reid_gan_b200.eval_dist import _positions, dst_table
    query = [("a", 1, 0), ("b", 2, 0)]
    gallery = [("c", 1, 1), ("a", 1, 0), ("d", 3, 1)]
    qpos, gpos = _positions(query, gallery)
    t = dst_table(["d", "a", "b", "c"], qpos, gpos, "cpu")
    assert t.dtype == torch.int32 and t.tolist() == [[-1, 4], [0, 3], [1, -1], [-1, 2]]
    with pytest.raises(ValueError):
        _positions(query + [("a", 1, 0)], gallery)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


class _Features:
    """Stands in for extract_features' DeviceFeatures: the names a rank's loader yielded (host rows: the check runs on
    the CPU here)."""

    def __init__(self, names, D):
        self._rows = names
        self._buf = torch.zeros((max(1, len(names)), D))
        self.device = torch.device("cpu")

    def keys(self):
        return list(self._rows)


def _worker(rank, world, port, result_dir, case):
    import sys
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from reid_gan_b200 import eval_dist
        from reid_gan_b200.evaluators import eval_shard
        query, gallery = _items(7), _items(20, 5) + _items(2)                  # two names in both lists
        share = eval_shard(query, gallery)
        names = [f for f, _, _ in share][::-1]                                  # any loader order
        D = 8
        if case == "rank1_misses_a_file" and rank == 1:
            names = names[1:]
        if case == "rank0_has_an_extra_file" and rank == 0:
            names = names + ["img_99999.jpg"]
        if case == "widths_differ" and rank == 1:
            D = 12
        if case == "width_not_a_multiple_of_4":
            D = 10
        eval_dist.extract_features = lambda model, loader: (_Features(names, D), None)

        def first_device_call(*a, **k):
            raise RuntimeError("first device call")
        eval_dist.torch.cuda.device = first_device_call
        try:
            eval_dist.DistributedEvaluator(None).evaluate(None, query, gallery)
            msg = "returned"
        except (ValueError, RuntimeError) as e:
            msg = "%s: %s" % (type(e).__name__, e)
        open(os.path.join(result_dir, "r%d.txt" % rank), "w").write(msg)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("case,expect", [
    ("all_loaded", "RuntimeError: first device call"),
    ("rank1_misses_a_file", "ValueError: DistributedEvaluator: rank(s) [1] extracted other files"),
    ("rank0_has_an_extra_file", "ValueError: DistributedEvaluator: rank(s) [0] extracted other files"),
    ("widths_differ", "ValueError: DistributedEvaluator: the ranks extracted features of different widths [8, 12]"),
    ("width_not_a_multiple_of_4", "ValueError: DistributedEvaluator: feature width D=10")])
def test_two_gloo_ranks_check_their_shares(case, expect, tmp_path):
    """Two ranks: the evaluator reaches its first device call only when each rank's loader yielded exactly its
    eval_shard share at one feature width; otherwise EVERY rank raises the same ValueError (no rank is left waiting
    in a collective)."""
    mp.spawn(_worker, args=(2, _free_port(), str(tmp_path), case), nprocs=2, join=True)
    for r in range(2):
        msg = (tmp_path / ("r%d.txt" % r)).read_text()
        assert msg.startswith(expect), msg
