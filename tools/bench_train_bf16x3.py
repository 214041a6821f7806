"""Training-step time of the bf16x3 training route (train_matmul="bf16x3") against the FFMA route of fp32 mode and the
tcgen05 bf16 route of bf16 mode.

    python tools/bench_train_bf16x3.py [--quick]

LinearModel(1024, 2, residual, batch_norm, max_norm), dropout keep 0.5, Adam, the same trained-BN weights (oracle init,
seed 1) in every route, torch CUDA tensors in: steps at B = 64, 1024, 4096 and 32768 (replayed CUDA graphs, generated
dropout), and train_epoch at B = 64 (64 batches of a 4096-row device-resident set).  Every shape is warmed up (the first
step of a shape runs directly, the second captures), then CUDA events time a run of back-to-back steps (about a second
of work, 3 steps at least).  Printed: ms per step, poses/s, the speed-up of bf16x3 over FFMA.  Routes run in the order
bf16x3, FFMA, bf16: nothing runs inference, so no bf16 model leaves the fused inference kernel's persisting-L2 set-aside
behind.  Then a torch.profiler pass over one bf16x3 step at B = 4096 gives the device time per kernel.  The card's
name, power limit and clocks are printed with the numbers."""
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "3d-pose-baseline_b200")]
from oracle import mlp_ref as M  # noqa: E402
from p3d import LinearModel  # noqa: E402

ROUTES = [("bf16x3", "bf16x3", "bf16x3"), ("FFMA", "fp32", None), ("bf16", "bf16", None)]


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True).stdout.strip().splitlines()[0]
    except Exception:
        return "unknown"


def model(mode, tm):
    p = {k: v.astype(np.float32) for k, v in M.init_params(1024, 2, seed=1, bn="trained").items()}
    m = LinearModel(1024, 2, True, True, True, 64, 1e-3, mode=mode, seed=1, train_matmul=tm)
    m.set_variables(p)
    return m


def timed(fn, budget_s=1.0):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    one = a.elapsed_time(b) / 1e3
    n = int(min(2000, max(3, budget_s / max(one, 1e-6))))
    a.record()
    for _ in range(n):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / 1e3 / n


def steps(sizes):
    res = {}
    for name, mode, tm in ROUTES:
        m = model(mode, tm)
        for B in sizes:
            g = torch.Generator(device="cuda").manual_seed(B)
            x = torch.randn((B, 32), device="cuda", generator=g)
            t = torch.randn((B, 48), device="cuda", generator=g)
            res[(name, B)] = timed(lambda: m.step(None, x, t, 0.5, isTraining=True))
        n, B = 4096, 64
        X = torch.randn((n, 32), device="cuda")
        T = torch.randn((n, 48), device="cuda")
        res[(name, "epoch")] = timed(lambda: m.train_epoch(X, T, 0.5, shuffle=False)) / (n // B)
        m.close()
    print(f"\nLinearModel(1024, 2 blocks, residual, batch_norm, max_norm), dropout 0.5, Adam: ms per step")
    print(f"{'B':>8} " + " ".join(f"{n:>10}" for n, _, _ in ROUTES) + f" {'FFMA/bf16x3':>12} {'bf16x3 poses/s':>15}")
    for B in list(sizes) + ["epoch"]:
        row = [res[(n, B)] for n, _, _ in ROUTES]
        rows = 64 if B == "epoch" else B
        lab = "epoch@64" if B == "epoch" else str(B)
        print(f"{lab:>8} " + " ".join(f"{r * 1e3:10.3f}" for r in row) + f" {row[1] / row[0]:11.2f}x {rows / row[0]:15.4g}",
              flush=True)


def profile(B=4096):
    from torch.profiler import ProfilerActivity, profile as prof
    m = model("bf16x3", "bf16x3")
    x = torch.randn((B, 32), device="cuda")
    t = torch.randn((B, 48), device="cuda")
    masks = (torch.rand((5, B, 1024), device="cuda") < 0.5).to(torch.uint8).cpu().numpy()
    for _ in range(2):
        m.step(None, x, t, 0.5, isTraining=True, dropout_mask=masks)     # eager: every kernel is its own launch
    torch.cuda.synchronize()
    with prof(activities=[ProfilerActivity.CUDA]) as pr:
        m.step(None, x, t, 0.5, isTraining=True, dropout_mask=masks)
        torch.cuda.synchronize()
    print(f"\nbf16x3 route, one step at B = {B} (injected masks, eager): device time per kernel")
    rows = [(e.key, e.device_time_total, e.count) for e in pr.key_averages()]
    tot = sum(r[1] for r in rows if r[1] > 0)
    print(f"  total {tot / 1e3:.3f} ms of device time (includes the mask upload)")
    for k, tt, c in sorted(rows, key=lambda r: -r[1]):
        if tt > 0:
            print(f"  {tt / 1e3:9.3f} ms  {100 * tt / tot:5.1f}%  x{c:<4d} {k[:110]}")
    m.close()


def main():
    print(f"card: {card()}")
    quick = "--quick" in sys.argv
    steps([64, 1024] if quick else [64, 1024, 4096, 32768])
    if not quick:
        profile()
    print(f"card after: {card()}")


if __name__ == "__main__":
    main()
