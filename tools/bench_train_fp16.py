"""Training-step time of the fp16 training route (train_matmul="fp16") against the bf16 route, alternating in one
process, and the gradient error of both against an fp32-mode model.

    python tools/bench_train_fp16.py [--quick] [--rounds R]

LinearModel(1024, 2, residual, batch_norm, max_norm), dropout keep 0.5, Adam, the same trained-BN weights (oracle init,
seed 1) in both routes (bf16-mode models), torch CUDA tensors in, generated dropout: steps at B = 64, 1024, 4096 and
32768 (replayed CUDA graphs).  Per batch size both models are warmed up (the first step of a shape runs directly, the
second captures), then R rounds (default 7) in which the two routes take turns, each timed by CUDA events over a run of
back-to-back steps (about 0.2 s of work, 3 steps at least).  Printed: median ms per step of each route, min / max over
the rounds, the fp16 / bf16 ratio of the medians.  Accuracy: one step of each route and of an fp32-mode model (FFMA,
fp32-class) on the same variables, inputs and injected masks; the relative L2 of each weight gradient against the fp32
model's, max and median over the six weight tensors.  The card's name, power limit and SM clocks are read in the same
run, before and after."""
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "3d-pose-baseline_b200")]
from oracle import mlp_ref as M  # noqa: E402
from p3d import LinearModel  # noqa: E402


def card():
    return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]


def model(mode, tm):
    p = {k: v.astype(np.float32) for k, v in M.init_params(1024, 2, seed=1, bn="trained").items()}
    m = LinearModel(1024, 2, True, True, True, 64, 1e-3, mode=mode, seed=1, train_matmul=tm)
    m.set_variables(p)
    return m


def run_time(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / 1e3 / n


def speed(sizes, rounds):
    routes = {"bf16": model("bf16", None), "fp16": model("bf16", "fp16")}
    print("\nLinearModel(1024, 2 blocks, residual, batch_norm, max_norm), dropout 0.5, Adam, replayed graphs: ms per step")
    print(f"{'B':>6} {'bf16 ms':>9} {'fp16 ms':>9} {'fp16/bf16':>10} {'bf16 min..max':>17} {'fp16 min..max':>17}")
    for B in sizes:
        g = torch.Generator(device="cuda").manual_seed(B)
        x = torch.randn((B, 32), device="cuda", generator=g)
        t = torch.randn((B, 48), device="cuda", generator=g)
        fns = {k: (lambda m=m: m.step(None, x, t, 0.5, isTraining=True)) for k, m in routes.items()}
        for f in fns.values():
            for _ in range(3):
                f()
        torch.cuda.synchronize()
        one = run_time(fns["bf16"], 3)
        n = int(min(2000, max(3, 0.2 / max(one, 1e-6))))
        times = {k: [] for k in fns}
        for _ in range(rounds):
            for k in ("bf16", "fp16"):
                times[k].append(run_time(fns[k], n))
        mb, mf = np.median(times["bf16"]), np.median(times["fp16"])
        print(f"{B:>6} {mb * 1e3:9.4f} {mf * 1e3:9.4f} {mf / mb:10.3f} "
              f"{min(times['bf16']) * 1e3:8.4f}..{max(times['bf16']) * 1e3:<8.4f} "
              f"{min(times['fp16']) * 1e3:8.4f}..{max(times['fp16']) * 1e3:<8.4f}", flush=True)
    for m in routes.values():
        m.close()


def accuracy(sizes):
    print("\nweight-gradient relative L2 against an fp32-mode model (one step, same variables / inputs / masks): max / median")
    print(f"{'B':>6} {'bf16 route':>20} {'fp16 route':>20}")
    for B in sizes:
        rs = np.random.RandomState(B)
        x = rs.standard_normal((B, 32)).astype(np.float32)
        t = rs.standard_normal((B, 48)).astype(np.float32)
        masks = (rs.uniform(size=(5, B, 1024)) < 0.5).astype(np.uint8)
        grads = {}
        for name, mode, tm in (("fp32", "fp32", None), ("bf16", "bf16", None), ("fp16", "bf16", "fp16")):
            m = model(mode, tm)
            m.step(None, x, t, 0.5, isTraining=True, dropout_mask=masks)
            grads[name] = {k: v.astype(np.float64) for k, v in m.get_gradients().items() if k.rsplit("/", 1)[-1][0] == "w"}
            m.close()
        row = []
        for r in ("bf16", "fp16"):
            e = [np.linalg.norm(grads[r][k] - g) / np.linalg.norm(g) for k, g in grads["fp32"].items()]
            row.append(f"{max(e):.2e} / {np.median(e):.2e}")
        print(f"{B:>6} {row[0]:>20} {row[1]:>20}", flush=True)


def main():
    quick = "--quick" in sys.argv
    rounds = int(sys.argv[sys.argv.index("--rounds") + 1]) if "--rounds" in sys.argv else 7
    sizes = [64, 1024] if quick else [64, 1024, 4096, 32768]
    print(f"card: {card()}")
    speed(sizes, rounds)
    accuracy(sizes)
    print(f"card after: {card()}")


if __name__ == "__main__":
    main()
