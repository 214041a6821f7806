"""Per-epoch action-wise evaluation: the reference-style loop against evaluate_actions on a staged set, and the
segmented evaluation kernel against the unsegmented one.

    python tools/bench_eval_actions.py [--rounds 7] [--poses 32768] [--out result.json]

1. 15 actions of about `--poses` poses each (2 subjects x 2 cameras per action), batch_size 64, a bf16 width-1024
   model.  Alternating rounds of (a) get_action_subset + get_all_batches + evaluate_batches per action, the loop of
   upstream train() with --evaluateActionWise, and (b) evaluate_actions on the set staged once; median and spread.
   The one-time stage_actions cost is reported on its own.
2. Kernel time (CUDA events over 20 launches, after a warm-up) of p3d_mpjpe_segments against p3d_procrustes_mpjpe on
   2^20 poses (403 MB of rows, beyond the 126 MB L2), with 1 and 120 segments, each kind alone and both.  HBM share =
   384 bytes per pose (two fp32 rows of 48) over the kernel time, against 7.7 TB/s.
The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "3d-pose-baseline_b200")]
from p3d import LinearModel, _lib, evaluate  # noqa: E402

ACTIONS = ["Directions", "Discussion", "Eating", "Greeting", "Phoning", "Photo", "Posing", "Purchases", "Sitting",
           "SittingDown", "Smoking", "Waiting", "WalkDog", "Walking", "WalkTogether"]
HBM = 7.7e12


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 else "unknown"


def test_set(poses, rng):
    d2, d3 = {}, {}
    for a, action in enumerate(ACTIONS):
        n = poses + int(rng.randint(-poses // 8, poses // 8))
        for subj in (9, 11):
            for cam in ("54138969", "55011271"):
                k = n // 4
                f = "%s.%s.h5" % (action, cam)
                d2[(subj, action, f + "-sh")] = rng.standard_normal((k, 32))
                d3[(subj, action, f)] = rng.standard_normal((k, 48))
    return d2, d3


def reference_loop(m, d2, d3, mean, std):
    cum = 0.0
    for action in ACTIONS:
        enc, dec = m.get_all_batches(evaluate.get_action_subset(d2, action), evaluate.get_action_subset(d3, action),
                                     True, training=False)
        err, _, _, _ = evaluate.evaluate_batches(None, m, mean, std, None, None, None, None, None, None, 0, enc, dec)
        cum += err
    return cum / len(ACTIONS)


def kernel_times(N=1 << 20, reps=20):
    g = torch.Generator(device="cuda").manual_seed(0)
    gt = torch.randn((N, 48), device="cuda", generator=g)
    pred = gt + 0.2 * torch.randn((N, 48), device="cuda", generator=g)
    rng = np.random.RandomState(1)
    mean, std = rng.standard_normal(96) * 100, rng.uniform(20, 200, 96)
    mp, sp = _lib.np_ptr(mean), _lib.np_ptr(std)
    sums = torch.zeros((120, 35), dtype=torch.float64, device="cuda")
    st = _lib.current_stream()
    seg = {1: np.array([0, N], dtype=np.int64),
           120: np.linspace(0, N, 121).astype(np.int64)}

    def run(fn):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps * 1e-3

    out = {}
    for proc in (0, 1):
        t = run(lambda: _lib.check(_lib.lib.p3d_procrustes_mpjpe(pred.data_ptr(), gt.data_ptr(), mp, sp, 0, proc, N, None,
                                                                 sums.data_ptr(), st)))
        out["unsegmented %s" % ("aligned" if proc else "plain")] = t
    for S, offs in seg.items():
        for kinds, name in ((1, "plain"), (2, "aligned"), (3, "both")):
            t = run(lambda: _lib.check(_lib.lib.p3d_mpjpe_segments(pred.data_ptr(), gt.data_ptr(), mp, sp, 0, kinds, N, 0,
                                                                   _lib.np_ptr(offs), S, sums.data_ptr(), st)))
            out["S=%d %s" % (S, name)] = t
    return {k: {"ms": v * 1e3, "GB/s": 384 * N / v / 1e9, "hbm_share": 384 * N / v / HBM} for k, v in out.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--poses", type=int, default=1 << 15)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_eval_actions needs a CUDA device")
    rng = np.random.RandomState(0)
    d2, d3 = test_set(args.poses, rng)
    mean, std = rng.standard_normal(96) * 100, rng.uniform(20, 200, 96)
    m = LinearModel(1024, 2, True, True, True, 64, 1e-3, mode="bf16", device=0, seed=1)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    s = evaluate.stage_actions(m, d2, d3, ACTIONS, True)
    torch.cuda.synchronize()
    staging = time.perf_counter() - t0
    ref_err = reference_loop(m, d2, d3, mean, std)                  # warm-up of both sides
    new_err = evaluate.evaluate_actions(None, m, s, mean, std).average
    ref_t, new_t = [], []
    for _ in range(args.rounds):
        t0 = time.perf_counter()
        reference_loop(m, d2, d3, mean, std)
        ref_t.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        evaluate.evaluate_actions(None, m, s, mean, std)
        new_t.append(time.perf_counter() - t0)
    res = {
        "card": card(),
        "actions": len(ACTIONS), "poses": s.n, "batch_size": 64, "model": "bf16 width 1024, 2 blocks",
        "staging_s": staging,
        "reference_loop_s": {"median": float(np.median(ref_t)), "min": min(ref_t), "max": max(ref_t)},
        "evaluate_actions_s": {"median": float(np.median(new_t)), "min": min(new_t), "max": max(new_t)},
        "speedup_median": float(np.median(ref_t) / np.median(new_t)),
        "err_mm": {"reference_loop": ref_err, "evaluate_actions": new_err},
        "kernels_2^20_poses": kernel_times(),
    }
    m.close()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
