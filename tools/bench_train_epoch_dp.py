"""Per-batch time of the data-parallel device-resident epoch (LinearModel.train_epoch) against the data-parallel step()
loop over the same batches (launch with torchrun, one process per GPU):

    torchrun --nproc-per-node 2 tools/bench_train_epoch_dp.py [global batch ...]     (default 64 4096 8192)
    python tools/bench_train_epoch_dp.py [global batch ...]                           (one GPU: the same comparison)

LinearModel(1024, 2, residual, batch_norm, max_norm), bf16, dropout 0.5, Adam, SyncBN.  Each arm gets the training set
the way its caller holds it: the epoch the concatenated set plus a permutation (NumPy: uploaded inside the call), the
step() loop the batches already cut and permuted (what get_all_batches returns; NumPy: uploaded per step).  Every shape
is warmed up first; CUDA events around the whole epoch, max over ranks, the median of REPS epochs of each arm, taken alternately.  One JSON line per
(global batch, input kind) on rank 0, with the GPU name and power limit read in the same run."""
import json
import os
import subprocess
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "3d-pose-baseline_b200")]
from p3d import LinearModel  # noqa: E402

NB, REPS, KEEP = 200, 3, 0.5
rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
if world > 1:
    dist.init_process_group("nccl", device_id=dev)


def power_limit():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", str(local)],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip() or None
    except (OSError, subprocess.SubprocessError):
        return None


def timed(fn):
    """ms of fn() between CUDA events, max over ranks"""
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item())


def step_loop(m, xs, ts):
    for xb, tb in zip(xs, ts):
        m.step(None, xb, tb, KEEP, isTraining=True)


gpu, plimit = torch.cuda.get_device_name(local), power_limit()
for B in [int(b) for b in (sys.argv[1:] or [64, 4096, 8192])]:
    n = NB * B
    rs = np.random.RandomState(0)
    X = rs.standard_normal((n, 32)).astype(np.float32)
    T = rs.standard_normal((n, 48)).astype(np.float32)
    perm = rs.permutation(n)
    m = LinearModel(1024, 2, True, True, True, B, 1e-3, mode="bf16", device=local, seed=1, dist=dist if world > 1 else None)
    for kind in ("numpy", "torch"):
        if kind == "numpy":
            Xa, Ta = X, T
            xs = [np.ascontiguousarray(X[perm[b * B:(b + 1) * B]]) for b in range(NB)]
            ts = [np.ascontiguousarray(T[perm[b * B:(b + 1) * B]]) for b in range(NB)]
        else:
            Xa, Ta = torch.from_numpy(X).to(dev), torch.from_numpy(T).to(dev)
            pd = torch.from_numpy(perm).to(dev)
            xs = [Xa[pd[b * B:(b + 1) * B]].contiguous() for b in range(NB)]
            ts = [Ta[pd[b * B:(b + 1) * B]].contiguous() for b in range(NB)]
        # warm-up: both arms' graphs and the NCCL / peer-memory paths of this shape
        m.train_epoch(Xa[:4 * B], Ta[:4 * B], KEEP, shuffle=False)
        step_loop(m, xs[:4], ts[:4])
        eps, sls = [], []
        for _ in range(REPS):      # the two arms alternate, so drift of the shared host hits both
            eps.append(timed(lambda: m.train_epoch(Xa, Ta, KEEP, perm=perm)))
            sls.append(timed(lambda: step_loop(m, xs, ts)))
        ep, sl = sorted(eps)[REPS // 2], sorted(sls)[REPS // 2]
        if rank == 0:
            print(json.dumps({"workload": "train_epoch vs step() loop, per batch (bf16, dropout 0.5, max_norm, Adam, SyncBN when data-parallel)",
                              "gpu": gpu, "power_limit": plimit, "n_gpus": world, "global_batch": B, "inputs": kind,
                              "batches": NB, "us_per_batch_train_epoch": round(ep * 1e3 / NB, 1),
                              "us_per_batch_step_loop": round(sl * 1e3 / NB, 1), "step_loop_over_epoch": round(sl / ep, 3),
                              "peer_memory_reductions": bool(getattr(m, "p2p", False))}), flush=True)
    m.close()
if world > 1:
    dist.destroy_process_group()
