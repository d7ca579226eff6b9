"""DistributedClusterMemory: one ClusterMemory shared by the ranks of a process group (one process per GPU).

The reference trains with nn.DataParallel: the backbone outputs of all GPUs are gathered onto GPU 0 in device order
and ONE ClusterMemory computes the loss and applies the momentum update over the concatenated batch (cm.py:110-137,
train_usl.py:189).  Here every rank keeps a replica of the centroids and computes the loss of its own rows; the rows
the update needs (xhat and target) travel as NVLink peer stores from the loss kernel itself (reid_cm_forward_push)
into a receive buffer on every rank, and in backward every rank applies the update of the whole batch, in rank order,
to its replica (reid_cm_update on W * cap rows, the padding rows carry target -1).  The split-K count of the logits
GEMM is that of the whole batch, so loss, gradients and centroids are those of the single-process module on the
concatenated batch -- byte for byte when all local batches have the same size (with different sizes the centroids
still are; loss and gradients may then use another split-K count and differ in the last bits).

Without an initialised process group, or with one rank, the module is a plain ClusterMemory.
"""
import torch
import torch.distributed as dist
from torch import autograd

from . import _lib, sharded
from ._lib import call, ptr, stream_ptr
from .cm import ClusterMemory, _need_cuda, _update


class _Exchange:
    """Receive-buffer bookkeeping of one (cap, D, W, device, group): the buffers themselves are symmetric memory
    (sharded._peer_buffer, one per step parity, cached there, so a module re-created every epoch does not rendezvous
    again).

    Why two buffers are enough.  Step s pushes into parity p = s mod 2, then every rank passes barrier s, then reads
    parity p in its update.  Rank A can push into parity p again only at step s + 2, and in A's stream order that
    push comes after barrier s + 1.  Every rank B reaches barrier s + 1, in ITS stream order, after its update of step
    s, the last reader of parity p.  So no rank overwrites a buffer another rank still reads -- provided every
    pushing forward is matched by exactly one barrier (in its backward, or, when no backward ran, at the start of the
    next pushing forward: `pending`) and the parity advances only on peer-store steps."""

    def __init__(self, cap, D, W):
        self.cap, self.D, self.W = cap, D, W
        self.nbytes = W * cap * 8 + W * cap * D * 4
        self.parity = 0
        self.pending = None        # (PeerBuffer, token) of a push whose barrier has not run yet

    def views(self, buf):
        """(targets (W * cap) int64, xhat (W * cap, D) fp32) of a receive buffer."""
        n = self.W * self.cap
        return buf[:n], buf.view(torch.float32)[2 * n: 2 * n + n * self.D].view(n, self.D)

    def settle(self):
        """Run the barrier of a push that no backward matched."""
        if self.pending is not None:
            self.pending[0].barrier()
            self.pending = None


_exchanges = {}


def _exchange(cap, D, W, dev, group):
    key_ = (cap, D, W, str(dev), id(group))
    if key_ not in _exchanges:
        _exchanges[key_] = _Exchange(cap, D, W)
    return _exchanges[key_]


def _local_slot(rows, D, dev):
    """A one-rank receive buffer (rows targets + rows x D xhat) and its address as a one-entry peer_base (filled on
    the device: no host-to-device copy)."""
    buf = torch.empty(rows + (rows * D + 1) // 2, dtype=torch.int64, device=dev)
    return buf, torch.full((1,), buf.data_ptr(), dtype=torch.int64, device=dev)


class _DistClusterLoss(autograd.Function):
    """_FusedClusterLoss with the batch exchange: forward pushes this rank's rows, backward applies the update of all
    ranks' rows."""

    @staticmethod
    def forward(ctx, inputs, targets, features, mem, push):
        _need_cuda(inputs, targets, features)
        L = _lib.lib()
        x = inputs.detach().to(torch.float32).contiguous()
        t = targets.to(torch.int64).contiguous()
        B, D = x.shape
        C = features.shape[0]
        W, me = mem._world()
        dev = x.device
        if B == 0:
            raise ValueError("DistributedClusterMemory: empty local batch")
        cap = mem._agree(B, C, D, dev) if push else max(mem._cap or 0, B)
        if B > cap:
            raise ValueError("DistributedClusterMemory: local batch of %d rows exceeds the %d agreed at the first "
                             "training step (the largest first batch of any rank)" % (B, cap))
        loss = torch.empty(B, dtype=torch.float32, device=dev)
        xhat = torch.empty((B, D), dtype=torch.float32, device=dev)
        inv_norm = torch.empty(B, dtype=torch.float32, device=dev)
        z = torch.empty((B, C), dtype=torch.float32, device=dev)
        scratch = torch.empty(max(1, L.reid_cm_forward_scratch_bytes(W * cap, C, D)), dtype=torch.uint8, device=dev)
        ctx.pb = ctx.slot = None
        with torch.cuda.device(dev):
            if push:
                ex = _exchange(cap, D, W, dev, mem.group)
                ex.settle()
                pb = sharded._peer_buffer("cm%d" % ex.parity, ex.nbytes, dev, mem.group)
                ctx.ex = ex
            else:
                pb = None
            if pb is not None:                          # peer stores into slot `me` of every rank's buffer
                ex.parity ^= 1
                token = object()
                ex.pending = (pb, token)
                ctx.pb, ctx.token = pb, token
                w_, me_, base = W, me, pb.peer_base
            else:                                       # no push / NCCL fallback: the slot stays local
                ctx.slot, base = _local_slot(cap, D, dev)
                w_, me_ = 1, 0
            call("reid_cm_forward_push", ptr(x), ptr(t), ptr(features), B, C, D, float(mem.temp), W * cap, ptr(loss),
                 ptr(xhat), ptr(inv_norm), ptr(z), ptr(scratch), me_, w_, cap, ptr(base), stream_ptr())
        ctx.features = features
        ctx.momentum = float(mem.momentum)
        ctx.temp = float(mem.temp)
        ctx.hard = bool(mem.use_hard)
        ctx.group = mem.group
        ctx.save_for_backward(t, xhat, inv_norm, z)
        return loss

    @staticmethod
    def backward(ctx, grad_loss):
        t, xhat, inv_norm, z = ctx.saved_tensors
        f = ctx.features
        B, D = xhat.shape
        C = f.shape[0]
        dev = xhat.device
        ex = ctx.ex
        grad_inputs = None
        with torch.cuda.device(dev):
            if ctx.needs_input_grad[0]:
                g = grad_loss.to(torch.float32).contiguous()
                gz = torch.empty((B, C), dtype=torch.float32, device=dev)
                grad_inputs = torch.empty((B, D), dtype=torch.float32, device=dev)
                # with the PRE-update centroids (cm.py:26,56)
                call("reid_cm_backward", ptr(g), ptr(z), ptr(t), ptr(f), ptr(xhat), ptr(inv_norm), B, C, D, ctx.temp,
                     ptr(gz), ptr(grad_inputs), stream_ptr())
            if ctx.pb is not None:
                if ex.pending is not None and ex.pending[1] is ctx.token:
                    ex.settle()                         # this push's barrier (unless a later forward ran it already)
                recv_t, recv_x = ex.views(ctx.pb.buf)
            else:
                slot_t, slot_x = _Exchange(ex.cap, D, 1).views(ctx.slot)
                recv_t = torch.empty(ex.W * ex.cap, dtype=torch.int64, device=dev)
                recv_x = torch.empty((ex.W * ex.cap, D), dtype=torch.float32, device=dev)
                dist.all_gather_into_tensor(recv_t, slot_t, group=ctx.group)
                dist.all_gather_into_tensor(recv_x, slot_x, group=ctx.group)
            _update(recv_x, recv_t, f, ctx.momentum, ctx.hard)   # the whole batch, rank order, on every replica
        return grad_inputs, None, None, None, None


class DistributedClusterMemory(ClusterMemory):
    """ClusterMemory over the ranks of `group` (default: the world group), as nn.DataParallel runs the reference's:
    forward returns the per-sample loss of this rank's rows, backward updates every rank's `features` with the
    whole batch (all ranks' rows in rank order).  Load `features` with the same centroids on every rank
    (sharded.pseudo_labels(..., centroids=True) returns them replicated).  A forward under torch.no_grad() or on
    inputs that need no gradient exchanges and updates nothing.

    The first training forward agrees on the largest local batch (`cap`, one small all-gather: the module's only
    host synchronisation); a later local batch may be smaller but not larger (ValueError)."""

    def __init__(self, num_features, num_samples, temp=0.05, momentum=0.2, use_hard=False, use_conf=False,
                 group=None):
        super(DistributedClusterMemory, self).__init__(num_features, num_samples, temp, momentum, use_hard, use_conf)
        self.group = group
        self._cap = None

    def _world(self):
        return dist.get_world_size(self.group), dist.get_rank(self.group)

    def _agree(self, B, C, D, dev):
        if self._cap is None:
            W, _ = self._world()
            mine = torch.tensor([B, C, D], dtype=torch.int64, device=dev)
            got = torch.empty(3 * W, dtype=torch.int64, device=dev)
            dist.all_gather_into_tensor(got, mine, group=self.group)
            rows = got.view(W, 3).tolist()
            if any(r[1:] != [C, D] for r in rows):
                raise ValueError("DistributedClusterMemory: the ranks hold memories of different shapes (C, D): %s"
                                 % [tuple(r[1:]) for r in rows])
            self._cap = max(r[0] for r in rows)
        return self._cap

    def forward(self, inputs, targets, gan_inputs=None, conf_weight=None):
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(self.group) == 1:
            return super(DistributedClusterMemory, self).forward(inputs, targets, gan_inputs, conf_weight)
        dev = self.features.device
        if not self.features.is_cuda:
            raise RuntimeError("DistributedClusterMemory must live on a CUDA device (call .cuda(), train_usl.py:189)")
        inputs = inputs.to(dev)
        targets = targets.to(dev)
        if self.features.dtype != torch.float32 or not self.features.is_contiguous():
            self.features = self.features.to(torch.float32).contiguous()
        push = torch.is_grad_enabled() and inputs.requires_grad
        return _DistClusterLoss.apply(inputs, targets, self.features, self, push)
