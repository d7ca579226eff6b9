"""GPU (-m gpu): DistributedClusterMemory and its C entry reid_cm_forward_push against the single-process ClusterMemory
on the concatenated batch (nn.DataParallel's gather order).

One device: W "virtual ranks".  The push kernel only STORES to the addresses in peer_base, so W plain device buffers
stand in for the W ranks' receive buffers; every rank's forward is issued in turn, then reid_cm_update runs on every
buffer.  Two or more devices: mp.spawn with NCCL, W = 2, ten training steps through the module."""
import os
import socket

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GOLDEN = ["cm_c300_d128", "cm_c40_d64", "cm_c33_d128_single"]


def _virtual_ranks(inp, tgt, cen, sizes, temp, momentum, hard, grad_loss):
    """Split (inp, tgt) over len(sizes) virtual ranks; returns (loss, z, grad) of the concatenated rows and the W
    updated centroid tensors."""
    from reid_gan_b200 import _lib
    from reid_gan_b200._lib import call, ptr
    from reid_gan_b200.cm import _update
    L = _lib.lib()
    W, cap = len(sizes), max(sizes)
    C, D = cen.shape
    n = W * cap
    bufs = [torch.full((n + (n * D + 1) // 2,), -7, dtype=torch.int64, device="cuda") for _ in range(W)]
    peer_base = torch.tensor([b.data_ptr() for b in bufs], dtype=torch.int64, device="cuda")
    scratch = torch.empty(L.reid_cm_forward_scratch_bytes(n, C, D), dtype=torch.uint8, device="cuda")
    losses, zs, grads = [], [], []
    o = 0
    for me, b in enumerate(sizes):
        x = inp[o:o + b].contiguous()
        t = tgt[o:o + b].contiguous()
        g = grad_loss[o:o + b].contiguous()
        o += b
        loss = torch.empty(b, device="cuda")
        xhat = torch.empty((b, D), device="cuda")
        inv = torch.empty(b, device="cuda")
        z = torch.empty((b, C), device="cuda")
        call("reid_cm_forward_push", ptr(x), ptr(t), ptr(cen), b, C, D, temp, n, ptr(loss), ptr(xhat), ptr(inv), ptr(z),
             ptr(scratch), me, W, cap, ptr(peer_base), None)
        gz = torch.empty((b, C), device="cuda")
        grad = torch.empty((b, D), device="cuda")
        call("reid_cm_backward", ptr(g), ptr(z), ptr(t), ptr(cen), ptr(xhat), ptr(inv), b, C, D, temp, ptr(gz), ptr(grad),
             None)
        losses.append(loss)
        zs.append(z)
        grads.append(grad)
    torch.cuda.synchronize()
    feats = []
    for buf in bufs:
        f = cen.clone()
        _update(buf.view(torch.float32)[2 * n: 2 * n + n * D].view(n, D), buf[:n], f, momentum, hard)
        feats.append(f)
    torch.cuda.synchronize()
    return torch.cat(losses), torch.cat(zs), torch.cat(grads), feats, bufs


def _single(inp, tgt, cen, temp, momentum, hard, grad_loss):
    """ClusterMemory on the whole batch: loss, z (same forward entry), input gradient, centroids after backward."""
    import reid_gan_b200 as rg
    from reid_gan_b200 import _lib
    from reid_gan_b200._lib import call, ptr
    B, D = inp.shape
    C = cen.shape[0]
    mem = rg.ClusterMemory(D, C, temp=temp, momentum=momentum, use_hard=hard).cuda()
    mem.features = cen.clone()
    x = inp.clone().requires_grad_(True)
    loss = mem(x, tgt)
    loss.backward(grad_loss)
    z = torch.empty((B, C), device="cuda")
    scratch = torch.empty(_lib.lib().reid_cm_forward_scratch_bytes(B, C, D), dtype=torch.uint8, device="cuda")
    tmp = [torch.empty(B, device="cuda"), torch.empty((B, D), device="cuda"), torch.empty(B, device="cuda")]
    call("reid_cm_forward", ptr(inp), ptr(tgt), ptr(cen), B, C, D, temp, ptr(tmp[0]), ptr(tmp[1]), ptr(tmp[2]), ptr(z),
         ptr(scratch), None)
    torch.cuda.synchronize()
    return loss.detach(), z, x.grad, mem.features


def _bytes_equal(a, b):
    return a.shape == b.shape and torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def _check(inp, tgt, cen, sizes, temp, momentum, hard, grad_loss, even):
    ref_loss, ref_z, ref_grad, ref_f = _single(inp, tgt, cen, temp, momentum, hard, grad_loss)
    loss, z, grad, feats, _ = _virtual_ranks(inp, tgt, cen, sizes, temp, momentum, hard, grad_loss)
    for f in feats:
        assert _bytes_equal(f, ref_f), "centroids differ from the single-process update"
    assert not torch.equal(ref_f, cen)
    if even:
        assert _bytes_equal(loss, ref_loss) and _bytes_equal(z, ref_z) and _bytes_equal(grad, ref_grad)
    else:
        # the logits may differ in the last bits (another split-K count), x 1 / temp in the softmax; the normalize-
        # backward then removes the radial part of the gradient, which leaves that error relative to a smaller
        # result (5.8e-5 measured at configs[2]): compare norms
        # the loss is a difference of logits: an ulp of |z| <= 1 / temp is its absolute error
        np.testing.assert_allclose(loss.cpu().numpy(), ref_loss.cpu().numpy(), rtol=1e-6,
                                   atol=1e-6 * float(ref_z.abs().max()))
        err = float((grad - ref_grad).norm() / ref_grad.norm())
        assert err <= 2e-4, "gradient differs by %g (relative Frobenius norm)" % err
    return ref_loss, ref_f


@pytest.mark.parametrize("hard", [False, True])
@pytest.mark.parametrize("W", [2, 4, 8])
@pytest.mark.parametrize("name", GOLDEN)
def test_virtual_ranks_golden(name, W, hard):
    g = np.load(os.path.join(GOLD, name + ".npz"))
    inp = torch.from_numpy(g["inputs"]).cuda()
    tgt = torch.from_numpy(g["targets"]).cuda()
    cen = torch.from_numpy(g["features"]).cuda()
    B = inp.shape[0]
    _check(inp, tgt, cen, [B // W] * W, float(g["temp"]), float(g["momentum"]), hard,
           torch.from_numpy(g["grad_loss"]).cuda(), even=True)


def _full_size():
    import reid_gan_b200 as rg
    x, ids = rg.synth(22000, 2048, 700, 0.8, 0)
    cen = torch.nn.functional.normalize(torch.stack([x[ids == k].mean(0) for k in range(700)]), dim=1)
    inp, tgt = rg.synth_cm_batch(x, ids, ids, 16, 16, seed=1)
    g = torch.Generator().manual_seed(5)
    grad_loss = torch.rand(256, generator=g) / 256
    return inp.cuda(), tgt.cuda(), cen.cuda(), grad_loss.cuda()


@pytest.fixture(scope="module")
def full_size():
    return _full_size()


@pytest.mark.parametrize("hard", [False, True])
@pytest.mark.parametrize("W", [2, 4, 8])
def test_virtual_ranks_full_size(full_size, W, hard):
    """BASELINE configs[2]: B = 256 (16 ids x 16), C = 700, D = 2048; every label occurs on several ranks."""
    inp, tgt, cen, grad_loss = full_size
    per_rank = [set(tgt[r * 256 // W:(r + 1) * 256 // W].tolist()) for r in range(W)]
    assert sum(len(a & b) for a in per_rank for b in per_rank if a is not b) > 0
    _check(inp, tgt, cen, [256 // W] * W, 0.05, 0.2, hard, grad_loss, even=True)


def test_hardest_member_on_a_later_rank(full_size):
    """CM_Hard: the hardest member of a label sits on the last rank, its first occurrence on rank 0."""
    inp, tgt, cen, grad_loss = (t.clone() for t in full_size)
    y = int(tgt[0])
    inp[250] = -3.0 * cen[y]
    tgt[250] = y
    xhat = torch.nn.functional.normalize(inp[tgt == y], dim=1)
    rows = torch.nonzero(tgt == y).flatten()
    assert int(rows[torch.argmin(xhat @ cen[y])]) == 250
    for W in (2, 4, 8):
        _check(inp, tgt, cen, [256 // W] * W, 0.05, 0.2, True, grad_loss, even=True)


@pytest.mark.parametrize("hard", [False, True])
def test_uneven_split(full_size, hard):
    """100 / 100 / 56 rows: centroids byte-identical; loss and gradients close (the split-K count of 3 x 100 rows may
    differ from that of 256)."""
    inp, tgt, cen, grad_loss = full_size
    _check(inp, tgt, cen, [100, 100, 56], 0.05, 0.2, hard, grad_loss, even=False)


@pytest.mark.parametrize("hard", [False, True])
def test_invalid_target_on_one_rank(full_size, hard):
    """Target -1 on rank 1: NaN loss for that row, no centroid row touched for it, everything else as on one GPU."""
    inp, tgt, cen, grad_loss = (t.clone() for t in full_size)
    tgt[70] = -1
    ref_loss, ref_f = _check(inp, tgt, cen, [64] * 4, 0.05, 0.2, hard, grad_loss, even=True)
    assert torch.isnan(ref_loss[70]) and not torch.isnan(ref_loss[torch.arange(256, device="cuda") != 70]).any()
    touched = set(torch.nonzero((ref_f != cen).any(dim=1)).flatten().tolist())
    assert touched == set(tgt[tgt >= 0].tolist())


def test_padding_slots_carry_target_minus_one(full_size):
    inp, tgt, cen, grad_loss = full_size
    _, _, _, _, bufs = _virtual_ranks(inp[:200], tgt[:200], cen, [100, 60, 40], 0.05, 0.2, False, grad_loss)
    for buf in bufs:
        t = buf[:300].view(3, 100)
        assert torch.equal(t[0], tgt[:100]) and torch.equal(t[1, :60], tgt[100:160]) and torch.equal(t[2, :40], tgt[160:200])
        assert (t[1, 60:] == -1).all() and (t[2, 40:] == -1).all()


def test_oversized_local_batch_raises_before_any_push():
    """Single process: a rank whose batch exceeds the agreed cap raises ValueError before anything is pushed."""
    from reid_gan_b200 import _lib
    from reid_gan_b200._lib import ptr
    L = _lib.lib()
    buf = torch.zeros(64, dtype=torch.int64, device="cuda")
    base = torch.tensor([buf.data_ptr()], dtype=torch.int64, device="cuda")
    x = torch.ones((5, 4), device="cuda")
    rc = L.reid_cm_forward_push(ptr(x), ptr(buf), ptr(x), 5, 3, 4, 0.05, 8, ptr(x), ptr(x), ptr(x), ptr(x), ptr(x), 0, 1, 4,
                                ptr(base), None)
    assert rc == _lib.REID_ERR_INVALID_ARG
    torch.cuda.synchronize()
    assert (buf == 0).all()


# ---- two devices ---------------------------------------------------------------------------------------------------

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
    x, ids = rg.synth(6000, 256, 120, 0.8, 3)
    cen = torch.nn.functional.normalize(torch.stack([x[ids == k].mean(0) for k in range(120)]), dim=1).to(dev)
    log = []
    for hard in (False, True):
        ref = rg.ClusterMemory(256, 120, temp=0.05, momentum=0.2, use_hard=hard).to(dev)
        ref.features = cen.clone()
        mem = rg.DistributedClusterMemory(256, 120, temp=0.05, momentum=0.2, use_hard=hard).to(dev)
        mem.features = cen.clone()
        for step in range(10):
            inp, tgt = rg.synth_cm_batch(x, ids, ids, 8, 8, seed=100 * step + int(hard))     # 64 rows
            inp, tgt = inp.to(dev), tgt.to(dev)
            g = torch.Generator().manual_seed(step)
            gl = (torch.rand(64, generator=g) / 64).to(dev)
            sizes = [32, 32] if step != 7 else [32, 20]                                      # step 7: uneven
            if step == 5:                                                                    # per-epoch re-creation
                f = mem.features.clone()
                mem = rg.DistributedClusterMemory(256, 120, temp=0.05, momentum=0.2, use_hard=hard).to(dev)
                mem.features = f
            rows = torch.cat([torch.arange(sum(sizes[:r]), sum(sizes[:r + 1])) for r in range(world)]).to(dev)
            a, b = sum(sizes[:rank]), sum(sizes[:rank + 1])
            xa, ta, ga = inp[rows], tgt[rows], gl[rows]
            xl = xa[a:b].clone()
            before = mem.features.clone()
            if step == 3:                                                   # evaluation: no exchange, no update
                with torch.no_grad():
                    loss = mem(xl, ta[a:b])
                    ref_loss = ref(xa, ta)
                ok = torch.equal(loss, ref_loss[a:b]) and torch.equal(mem.features, before)
            elif step == 4:                                                 # forward without backward: no update
                loss = mem(xl.requires_grad_(True), ta[a:b])
                ref_loss = ref(xa.clone().requires_grad_(True), ta)
                ok = torch.equal(loss.detach(), ref_loss.detach()[a:b]) and torch.equal(mem.features, before)
            else:
                xl.requires_grad_(True)
                loss = mem(xl, ta[a:b])
                loss.backward(ga[a:b])
                xr = xa.clone().requires_grad_(True)
                ref_loss = ref(xr, ta)
                ref_loss.backward(ga)
                if sizes[0] == sizes[1]:
                    ok = torch.equal(loss.detach(), ref_loss.detach()[a:b]) and torch.equal(xl.grad, xr.grad[a:b])
                else:
                    ok = bool(torch.allclose(loss.detach(), ref_loss.detach()[a:b], rtol=1e-6, atol=0))
                ok = ok and not torch.equal(mem.features, before)
            ok = ok and torch.equal(mem.features, ref.features)
            log.append("hard=%s step=%d ok=%s" % (hard, step, ok))
    torch.cuda.synchronize()
    dist.barrier()
    open(os.path.join(result_dir, "r%d.txt" % rank), "w").write("\n".join(log))
    os._exit(0)                      # without tearing down the peer mappings one by one (as scripts/dist_check.py)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
@pytest.mark.parametrize("peer", [True, False], ids=["peer-stores", "nccl"])
def test_two_devices(peer, tmp_path):
    _spawn(tmp_path, peer, "nccl")


def test_two_ranks_on_one_device_gloo(tmp_path):
    """The host layer with the collective fallback on a single GPU: two gloo ranks share cuda:0."""
    _spawn(tmp_path, False, "gloo")


def _spawn(tmp_path, peer, backend):
    import torch.multiprocessing as mp
    mp.spawn(_worker, args=(2, _free_port(), str(tmp_path), peer, backend), nprocs=2, join=True)
    for r in range(2):
        log = (tmp_path / ("r%d.txt" % r)).read_text().splitlines()
        assert len(log) == 20
        bad = [line for line in log if not line.endswith("ok=True")]
        assert not bad, "rank %d: %s" % (r, bad)
