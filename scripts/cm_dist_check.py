"""Multi-GPU check of DistributedClusterMemory (run under torchrun): K training steps through the module on every rank
must leave every rank's centroids byte-identical to ONE ClusterMemory fed the concatenated batches (nn.DataParallel's
gather order), and the step time (forward + backward + update through autograd, CUDA events, max over ranks) is
measured for both exchanges -- NVLink peer stores from the loss kernel, and the NCCL all-gather fallback.
BASELINE configs[2] shapes: C = 700, D = 2048, temp 0.05, momentum 0.2; 256 rows per rank (weak scaling) and 256 / W
rows per rank (global batch 256).  One line per configuration.
    python -m torch.distributed.run --nproc-per-node W --master-addr 127.0.0.1 scripts/cm_dist_check.py [--json OUT]"""
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
from reid_gan_b200 import sharded  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=10, help="training steps before the digest")
ap.add_argument("--timed", type=int, default=200, help="steps in the timed window")
ap.add_argument("--json", default=None, help="append one JSON object per configuration (rank 0)")
args = ap.parse_args()

rank = int(os.environ["RANK"])
world = int(os.environ["WORLD_SIZE"])
lr = int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(lr)
dev = torch.device("cuda", lr)
dist.init_process_group("nccl", device_id=dev)
C, D, TEMP, MOM = 700, 2048, 0.05, 0.2


def sha(t):
    return hashlib.sha256(np.ascontiguousarray(t.cpu().numpy()).tobytes()).hexdigest()[:16]


card = ""
if rank == 0:
    try:
        card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(lr)],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        card = "unknown (%r)" % (e,)
    print("card: %s; world %d" % (card, world), flush=True)

x, ids = rg.synth(22000, D, C, 0.8, 0)
cen = rg.generate_cluster_features(ids.numpy(), x.to(dev), normalize=True).contiguous()


def batches(rows_per_rank, k, seed):
    """k global batches (rank order = the concatenation), 16 instances per identity."""
    out = []
    n = rows_per_rank * world
    for s in range(k):
        inp, tgt = rg.synth_cm_batch(x, ids, ids, n // 16, 16, seed=seed + s)
        g = torch.Generator().manual_seed(seed + s)
        out.append((inp.to(dev), tgt.to(dev), (torch.rand(n, generator=g) / n).to(dev)))
    return out


def step(mem, inp, tgt, gl):
    xi = inp.detach().requires_grad_(True)
    mem(xi, tgt).backward(gl)


def time_steps(mem, data, n):
    for i in range(5):
        step(mem, *data[i % len(data)])
    torch.cuda.synchronize()
    dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n):
        step(mem, *data[i % len(data)])
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / n], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


ok = True
for rows in sorted({256, max(1, 256 // world)}, reverse=True):
    data = batches(rows, args.steps, 1000 * rows)
    a, b = rank * rows, (rank + 1) * rows
    for hard in (False, True):
        # single-process reference on the concatenated batches (every rank computes it; it is deterministic)
        ref = rg.ClusterMemory(D, C, temp=TEMP, momentum=MOM, use_hard=hard).to(dev)
        ref.features = cen.clone()
        for inp, tgt, gl in data:
            step(ref, inp, tgt, gl)
        ref_digest = sha(ref.features)
        t_single = time_steps(ref, data, args.timed) if rank == 0 else float("nan")
        for exchange in ("peer", "nccl"):
            sharded.PEER_EXCHANGE = exchange == "peer"
            mem = rg.DistributedClusterMemory(D, C, temp=TEMP, momentum=MOM, use_hard=hard).to(dev)
            mem.features = cen.clone()
            for inp, tgt, gl in data:
                step(mem, inp[a:b], tgt[a:b], gl[a:b])
            digests = [None] * world
            dist.all_gather_object(digests, sha(mem.features))
            same = all(d == ref_digest for d in digests)
            ok &= same
            local = [(inp[a:b].contiguous(), tgt[a:b].contiguous(), gl[a:b].contiguous()) for inp, tgt, gl in data]
            t_ms = time_steps(mem, local, args.timed)
            if rank == 0:
                rec = dict(world=world, rows_per_rank=rows, global_batch=rows * world, C=C, D=D, hard=hard,
                           exchange=exchange, steps=args.steps, identical=same, ref_digest=ref_digest,
                           rank_digests=digests, step_ms=round(t_ms, 4), single_gpu_step_ms=round(t_single, 4),
                           timed_steps=args.timed, card=card)
                print("W=%d rows/rank=%4d global=%4d hard=%d %-4s identical=%s ref=%s ranks=%s  step %.3f ms "
                      "(single GPU, global batch: %.3f ms)" % (world, rows, rows * world, hard, exchange, same,
                                                               ref_digest, ",".join(sorted(set(digests))), t_ms, t_single),
                      flush=True)
                if args.json:
                    with open(args.json, "a") as f:
                        f.write(json.dumps(rec) + "\n")
sharded.PEER_EXCHANGE = True
if rank == 0:
    print("CM DIST OK" if ok else "CM DIST MISMATCH", flush=True)
torch.cuda.synchronize()
dist.barrier()
os._exit(0 if ok else 1)
