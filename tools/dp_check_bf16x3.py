"""Two-rank check of the bf16x3 training route (launch with torchrun, one process per GPU; tests/test_gpu_train_bf16x3.py
does that with 2 ranks): a data-parallel step of a model with train_matmul="bf16x3" (rows sharded, SyncBN, gradient
all-reduce) against the same route on one GPU on the GLOBAL batch - loss, gathered outputs, gradients and updated
variables.  Prints 'DP BF16X3 OK' on rank 0."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "3d-pose-baseline_b200"), os.path.join(ROOT, "tests")]
from oracle import mlp_ref as M, synth  # noqa: E402
from p3d import LinearModel  # noqa: E402

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))

L, B, keep = 1024, 1030, 0.5           # uneven shards
p = {k: v.astype(np.float32) for k, v in M.init_params(L, 2, seed=4, bn="trained").items()}
dp = LinearModel(L, 2, True, True, True, B, 1e-3, mode="bf16x3", device=local, seed=7, dist=dist, train_matmul="bf16x3")
dp.set_variables(p)
one = LinearModel(L, 2, True, True, True, B, 1e-3, mode="bf16x3", device=local, seed=7, train_matmul="bf16x3")
one.set_variables(p)
why = []
for s in range(2):
    x, t = synth.mlp_inputs(B, seed=20 + s)
    masks = (np.random.RandomState(s).uniform(size=(5, B, L)) < keep).astype(np.uint8)
    l1, _, _, y1 = dp.step(None, x, t, keep, isTraining=True, dropout_mask=masks)
    l2, _, _, y2 = one.step(None, x, t, keep, isTraining=True, dropout_mask=masks)
    if not abs(float(l1) - float(l2)) <= 1e-5 * float(l2):
        why.append("step %d loss %r vs %r" % (s, float(l1), float(l2)))
    if not np.abs(y1 - y2).max() <= 1e-5 * np.abs(y2).max():
        why.append("step %d outputs %.3e" % (s, np.abs(y1 - y2).max()))
    g1, g2 = dp.get_gradients(), one.get_gradients()
    for k, g in g2.items():
        if np.abs(g).max() == 0.0:
            if np.abs(g1[k]).max() != 0.0:
                why.append("step %d %s not zero" % (s, k))
            continue
        rel = np.linalg.norm(g1[k] - g) / np.linalg.norm(g)
        if not rel <= 1e-4:
            why.append("step %d grad %s rel L2 %.3e" % (s, k, rel))
v1, v2 = dp.get_variables(), one.get_variables()
for k in v2:
    if not np.abs(v1[k] - v2[k]).max() <= 2e-3 * max(np.abs(v2[k]).max(), 1e-3):
        why.append("variable %s" % k)
w = torch.from_numpy(v1["linear_model/w4"]).cuda()
w0 = w.clone()
dist.broadcast(w0, 0)
if not torch.equal(w, w0):
    why.append("ranks disagree on w4")
ok = torch.tensor([0 if why else 1], device="cuda")
dist.all_reduce(ok, op=dist.ReduceOp.MIN)
if why:
    print("rank %d: %s" % (rank, "; ".join(why[:8])), flush=True)
if rank == 0 and int(ok.item()) == 1:
    print("DP BF16X3 OK", flush=True)
dp.close()
one.close()
dist.destroy_process_group()
sys.exit(0 if int(ok.item()) == 1 else 1)
