"""Data-parallel evaluate_actions on several GPUs (launch with torchrun, one process per GPU;
tests/test_gpu_dp_eval_actions.py does that with 2 ranks).  Every rank stages the same per-action test set; each scores
its row block and one all_reduce gives every rank the sums.  Checks, for an fp32 and a bf16 model, with n odd (ragged
shards) and predict_14 on and off:
  1. the result == evaluate_actions of a single-GPU model with the same variables (fp32: summation order; bf16: the
     shards may take other forward kernels than the whole set, tests/test_gpu_eval_actions.py's 1.2e-2),
  2. identical results on every rank,
  3. ValueError on every rank for mismatched sets or a rank's own bad argument, before anything launches.
Prints 'DP EVAL ACTIONS CHECK OK' on rank 0."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "3d-pose-baseline_b200")]
from oracle import synth  # noqa: E402
from p3d import LinearModel, evaluate  # noqa: E402

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
why = []
ACTIONS = ["Directions", "Eating", "Posing", "Walking"]


def same_on_all_ranks(a):
    t = torch.as_tensor(np.ascontiguousarray(a, dtype=np.float64)).to(dev)
    t0 = t.clone()
    dist.broadcast(t0, 0)
    return bool(torch.equal(t, t0))


def test_set(p14, sizes):
    out = 42 if p14 else 48
    d2, d3 = {}, {}
    for i, (action, n) in enumerate(zip(ACTIONS, sizes)):
        x, t = synth.mlp_inputs(n, out_size=out, seed=10 + i)
        d2[(9, action, "%s.54138969.h5-sh" % action)] = x.astype(np.float64)
        d3[(9, action, "%s.54138969.h5" % action)] = t.astype(np.float64)
    return d2, d3


rng = np.random.RandomState(5)
mean, std = rng.standard_normal(96) * 100, rng.uniform(20, 200, 96)
for mode, p14 in (("fp32", False), ("fp32", True), ("bf16", False), ("bf16", True)):
    tag = "%s%s" % (mode, " predict_14" if p14 else "")
    L = 1024 if mode == "bf16" else 256
    md = LinearModel(L, 2, True, True, True, 64, 1e-3, predict_14=p14, mode=mode, device=local, seed=4, dist=dist)
    ms = LinearModel(L, 2, True, True, True, 64, 1e-3, predict_14=p14, mode=mode, device=local, seed=4)
    ms.set_variables(md.get_variables())
    d2, d3 = test_set(p14, [1001, 517, 2049, 333])
    s = evaluate.stage_actions(md, d2, d3, ACTIONS, True, drop_tail=False)      # n = 3900 ... odd below
    s_odd = evaluate.stage_actions(md, d2, d3, ACTIONS[:3], True, drop_tail=False)
    if s_odd.n % 2 != 1:
        why.append("%s: the ragged set has %d rows" % (tag, s_odd.n))
    tol = 1e-6 if mode == "fp32" else 1.2e-2
    for st in (s, s_odd):
        for proc in (False, True, "both"):
            rd = evaluate.evaluate_actions(None, md, st, mean, std, procrustes=proc, dist=dist)
            r1 = evaluate.evaluate_actions(None, ms, st, mean, std, procrustes=proc)
            pairs = list(zip(rd, r1)) if proc == "both" else [(rd, r1)]
            for a, b in pairs:
                for action in st.actions:
                    if not abs(a.errors[action] - b.errors[action]) <= tol * b.errors[action]:
                        why.append("%s n=%d proc=%s %s: %r on %d GPUs vs %r on one" % (tag, st.n, proc, action,
                                   a.errors[action], world, b.errors[action]))
                    if not np.allclose(a.joint_errors[action], b.joint_errors[action], rtol=tol, atol=1e-9):
                        why.append("%s n=%d %s: joint errors differ" % (tag, st.n, action))
                    if not abs(a.losses[action] - b.losses[action]) <= max(tol, 1e-5) * b.losses[action]:
                        why.append("%s n=%d %s: loss %r vs %r" % (tag, st.n, action, a.losses[action], b.losses[action]))
                vec = [a.average] + [a.errors[k] for k in st.actions] + [a.losses[k] for k in st.actions] + \
                      [x for k in st.actions for x in a.joint_errors[k]]
                if not same_on_all_ranks(vec):
                    why.append("%s n=%d proc=%s: results differ between ranks" % (tag, st.n, proc))
    # mismatched sets and a rank's own argument error raise everywhere
    bad_sets = {
        "n": evaluate.stage_actions(md, d2, d3, ACTIONS, True, drop_tail=rank == 0),
        "actions": evaluate.stage_actions(md, d2, d3, ACTIONS if rank == 0 else ACTIONS[:3], True),
        "offsets": evaluate.stage_actions(md, d2, d3, ACTIONS if rank == 0 else ACTIONS[::-1], True),
    }
    for name, st in bad_sets.items():
        try:
            evaluate.evaluate_actions(None, md, st, mean, std, dist=dist)
            why.append("%s: mismatched %s did not raise" % (tag, name))
        except ValueError:
            pass
    try:
        evaluate.evaluate_actions(None, md, s, mean, std, precision="fp32" if rank == 0 else "fp8", dist=dist)
        why.append("%s: another rank's bad precision did not raise" % tag)
    except ValueError:
        pass
    md.close()
    ms.close()

if why:
    print("DP EVAL ACTIONS CHECK FAILED on rank %d: %s" % (rank, "; ".join(why)), flush=True)
flag = torch.tensor([0 if why else 1], device=dev)
dist.all_reduce(flag, op=dist.ReduceOp.MIN)
if rank == 0:
    print("DP EVAL ACTIONS CHECK OK" if flag.item() == 1 else "DP EVAL ACTIONS CHECK FAILED", "(world %d)" % world, flush=True)
dist.destroy_process_group()
sys.exit(0 if flag.item() == 1 else 1)
