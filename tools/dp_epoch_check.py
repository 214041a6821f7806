"""Data-parallel LinearModel.train_epoch on several GPUs (launch with torchrun, one process per GPU;
tests/test_gpu_dp_epoch.py does that with 2 ranks).  For bf16 at global batch 4096 (fused route: grid barrier and
in-kernel exchange), bf16 at 129 (ragged shards of 65 and 64 rows) and fp32 at 66 (FFMA route, small peer reductions),
each with n not a multiple of the batch and dropout 0.5:
  1. the epoch == the data-parallel step() loop over the same permutation (losses, variables),
  2. the epoch == a single-GPU epoch on the same data, permutation and seed,
  3. variables bit-equal on every rank afterwards, losses and global_step identical,
  4. rank 0's permutation is the one used when another rank passes a different one,
  5. a mismatched n or batch_size raises ValueError on every rank; n < batch_size runs no step.
Prints 'DP EPOCH CHECK OK' on rank 0."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "3d-pose-baseline_b200")]
from oracle import synth  # noqa: E402
from p3d import LinearModel, _lib  # noqa: E402

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
LR = 1e-3
why = []


def same_on_all_ranks(a):
    t = torch.as_tensor(np.ascontiguousarray(a)).to(dev)
    t0 = t.clone()
    dist.broadcast(t0, 0)
    return bool(torch.equal(t, t0))


def model(L, B, mode, *, dp=True, batch_size=None):
    return LinearModel(L, 2, True, True, True, batch_size or B, LR, mode=mode, device=local, seed=11, dist=dist if dp else None)


def close_to_steps(tag, la, va, lb, vb):
    """tests/test_gpu_train.py::test_train_epoch_equals_stepping_through_the_batches: split-K atomics differ in the last bits"""
    if not np.allclose(la, lb, rtol=2e-4, atol=1e-6):
        why.append("%s: losses %s vs %s" % (tag, la, lb))
    for k in va:
        if not np.abs(va[k] - vb[k]).max() <= 2e-3 * max(np.abs(vb[k]).max(), 1e-3):
            why.append("%s: %s differs by %.3e" % (tag, k, np.abs(va[k] - vb[k]).max()))


for mode, L, B, n in (("bf16", 1024, 4096, 3 * 4096 + 100), ("bf16", 1024, 129, 1000), ("fp32", 256, 66, 500)):
    keep, nb = 0.5, n // B
    tag = "%s B=%d" % (mode, B)
    x, t = synth.mlp_inputs(n, seed=B)
    perm = np.random.RandomState(3).permutation(n)
    ma, mb, mc = model(L, B, mode), model(L, B, mode), model(L, B, mode)
    ms = model(L, B, mode, dp=False)
    ms._seed = ma._seed
    ms.set_variables(ma.get_variables())

    # 1. epoch == the step() loop, data parallel
    la, lr = ma.train_epoch(x, t, keep, perm=perm)
    if la.shape != (nb,) or int(ma.global_step) != nb:
        why.append("%s: %s losses, global_step %d after %d batches" % (tag, la.shape, int(ma.global_step), nb))
    lb = []
    for b in range(nb):
        idx = perm[b * B:(b + 1) * B]
        loss, _, lrs, yb = mb.step(None, x[idx], t[idx], keep, isTraining=True)
        lb.append(float(loss))
    va = ma.get_variables()
    close_to_steps(tag + " epoch vs step loop", la, va, np.array(lb), mb.get_variables())
    if abs(lr - float(lrs.value)) > 1e-9:
        why.append("%s: last learning rate %r vs %r" % (tag, lr, float(lrs.value)))
    # the last batch's global outputs are still available after the epoch as after a step
    yg = torch.empty((B, 48), dtype=torch.float32, device=dev)
    rc = _lib.lib.p3d_model_gathered_outputs(ma._handle, yg.data_ptr(), B, _lib.current_stream())
    rel = np.linalg.norm(yg.cpu().numpy() - yb) / np.linalg.norm(yb)
    if rc == 0 and not rel <= 1e-2:        # after nb steps of Adam on each side: same batch, drifted weights
        why.append("%s: gathered outputs of the last batch off by %.3e (relative L2)" % (tag, rel))
    elif rc not in (0, 1):
        why.append("%s: p3d_model_gathered_outputs returned %d" % (tag, rc))

    # 2. data parallel == one GPU (tools/dp_check.py's fused-step tolerances, movement scaled by the number of steps)
    ls, _ = ms.train_epoch(x, t, keep, perm=perm)
    for i in range(nb):
        if not abs(la[i] - ls[i]) <= (2e-5 if i == 0 else 2e-4) * max(1.0, float(ls[i])):
            why.append("%s: batch %d loss %r on %d GPUs vs %r on one" % (tag, i, float(la[i]), world, float(ls[i])))
    vs = ms.get_variables()
    for k in va:
        err = np.abs(va[k].astype(np.float64) - vs[k])
        if not np.quantile(err, 0.99) <= (0.1 if B >= 512 else 0.2) * nb * LR + 1e-5 * np.abs(vs[k]).max():
            why.append("%s: %s 99%% quantile of |dp - single| = %.3e" % (tag, k, np.quantile(err, 0.99)))

    # 3. replicas identical
    for k in va:
        if not same_on_all_ranks(va[k]):
            why.append("%s: %s differs between ranks" % (tag, k))
    if not all([same_on_all_ranks(la), same_on_all_ranks(np.array([int(ma.global_step)]))]):     # lists: every rank broadcasts alike
        why.append("%s: losses or global_step differ between ranks" % tag)

    # 4. rank 0's permutation wins
    lc, _ = mc.train_epoch(x, t, keep, perm=perm if rank == 0 else perm[::-1].copy())
    close_to_steps(tag + " other rank's perm", lc, mc.get_variables(), la, va)

    # 5. disagreement raises everywhere, before any launch; n < batch_size runs no step
    for bad in ("n", "batch_size"):
        mm = ma if bad == "n" else model(L, B, mode, batch_size=B + rank)
        g0 = int(mm.global_step)
        k = n - rank if bad == "n" else n
        try:
            mm.train_epoch(x[:k], t[:k], keep, perm=perm[:k] if bad == "n" else perm)
            why.append("%s: mismatched %s did not raise" % (tag, bad))
        except ValueError:
            pass
        if int(mm.global_step) != g0:
            why.append("%s: mismatched %s stepped" % (tag, bad))
        if mm is not ma:
            mm.close()
    l0, _ = ma.train_epoch(x[:B - 1], t[:B - 1], keep)
    if l0.shape != (0,) or int(ma.global_step) != nb:
        why.append("%s: n < batch_size gave %s losses, global_step %d" % (tag, l0.shape, int(ma.global_step)))

    # torch in -> torch out; shuffled by rank 0 while every rank's NumPy generator differs
    if mode == "bf16" and B == 129:
        np.random.seed(100 + rank)
        lt, lrt = ma.train_epoch(torch.from_numpy(x).to(dev), torch.from_numpy(t).to(dev), keep)
        if not (lt.is_cuda and lt.shape == (nb,) and bool(torch.isfinite(lt).all()) and torch.is_tensor(lrt)):
            why.append("%s: torch epoch returned %s" % (tag, lt))
        if not all([same_on_all_ranks(lt.cpu().numpy())] + [same_on_all_ranks(v) for v in ma.get_variables().values()]):
            why.append("%s: shuffled torch epoch differs between ranks" % tag)
    for m_ in (ma, mb, mc, ms):
        m_.close()

if why:
    print("DP EPOCH CHECK FAILED on rank %d: %s" % (rank, "; ".join(why)), flush=True)
flag = torch.tensor([0 if why else 1], device=dev)
dist.all_reduce(flag, op=dist.ReduceOp.MIN)
if rank == 0:
    print("DP EPOCH CHECK OK" if flag.item() == 1 else "DP EPOCH CHECK FAILED", "(world %d)" % world, flush=True)
dist.destroy_process_group()
sys.exit(0 if flag.item() == 1 else 1)
