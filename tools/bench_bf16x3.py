"""Throughput of the bf16x3 inference mode against fp32 and bf16 mode, and its accuracy against fp32 mode.

    python tools/bench_bf16x3.py [--quick]

LinearModel(1024, 2, residual, batch_norm, max_norm) at B = 1, 64, 4096, 65536, 2^20 and LinearModel(4096, 4, ...) at
2^18, the same trained-BN weights (oracle init, seed 1) in every mode, torch CUDA tensors in and out.  Per shape and
mode (mode by mode, bf16 last: see run()): every shape is warmed up first, then CUDA events time a run of back-to-back calls (about a quarter second of work,
3 calls at least).  Printed: ms per call, poses/s, useful TFLOP/s (2 (32 L + 2 n L^2 + 48 L) per pose: 8,552,448 at
width 1024) and tensor TFLOP/s (three bf16 products per MatMul in bf16x3 mode) as a share of the 2,250 TFLOP/s dense
bf16 data-sheet figure; and the row-wise max ||y - y_fp32|| / ||y_fp32|| of bf16x3 and bf16 mode on the same inputs.
Between calls the weights stay L2-resident, as they do in use.  First a torch.profiler pass over one bf16x3 call at
2^20 poses gives the device time per kernel (the split across layers).
The card's name and power limit are printed with the numbers."""
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "3d-pose-baseline_b200")]
from oracle import mlp_ref as M  # noqa: E402
from p3d import LinearModel  # noqa: E402

PEAK_BF16 = 2250.0


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True).stdout.strip().splitlines()[0]
    except Exception:
        return "unknown"


def flop_per_pose(L, nl, out=48):
    return 2 * (32 * L + 2 * nl * L * L + L * out)


def timed(fn, budget_s=0.25):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    one = a.elapsed_time(b) / 1e3
    n = int(min(500, max(3, budget_s / max(one, 1e-6))))
    a.record()
    for _ in range(n):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / 1e3 / n


def rowwise(y, ref):
    y, ref = y.double(), ref.double()
    return float(((y - ref).norm(dim=1) / ref.norm(dim=1).clamp_min(1e-30)).max())


def run(shapes, modes):
    """shapes: [(L, nl, [B ...])].  Mode by mode, in the order given: the bf16 fused kernel sets part of the L2
    aside for its activations (persisting window, held until a training step hands it back), which the other modes'
    GEMMs would then run without."""
    outs = {}
    for mode in modes:
        for L, nl, sizes in shapes:
            p = {k: v.astype(np.float32) for k, v in M.init_params(L, nl, seed=1, bn="trained").items()}
            m = LinearModel(L, nl, True, True, True, 64, 1e-3, mode=mode, seed=1)
            m.set_variables(p)
            fpp = flop_per_pose(L, nl)
            print(f"\n{mode}, width {L}, {nl} blocks, residual, batch_norm, max_norm: {fpp:,} FLOP per pose")
            print(f"{'B':>8} {'ms/call':>10} {'poses/s':>12} {'useful TF/s':>12} {'tensor TF/s':>12} {'% of 2250':>9}")
            for B in sizes:
                x = torch.randn((B, 32), device="cuda", generator=torch.Generator(device="cuda").manual_seed(B))
                outs[(mode, L, B)] = m.step(None, x, None, 1.0, isTraining=False)[2].clone()
                t = timed(lambda: m.step(None, x, None, 1.0, isTraining=False))
                useful = B * fpp / t / 1e12
                tensor = {"bf16x3": 3 * useful, "bf16": useful}.get(mode)
                ts = f"{tensor:12.1f} {100 * tensor / PEAK_BF16:8.1f}%" if tensor else f"{'-':>12} {'-':>9}"
                print(f"{B:8d} {t * 1e3:10.3f} {B / t:12.4g} {useful:12.1f} {ts}", flush=True)
            m.close()
    print("\nrow-wise max ||y - y_fp32|| / ||y_fp32|| on the same inputs")
    for (mode, L, B), y in outs.items():
        if mode != "fp32":
            print(f"  {mode:>7} width {L:5d} B {B:8d}: {rowwise(y, outs[('fp32', L, B)]):.2e}")


def profile(B=1 << 20):
    from torch.profiler import ProfilerActivity, profile as prof
    p = {k: v.astype(np.float32) for k, v in M.init_params(1024, 2, seed=1, bn="trained").items()}
    m = LinearModel(1024, 2, True, True, True, 64, 1e-3, mode="bf16x3", seed=1)
    m.set_variables(p)
    x = torch.randn((B, 32), device="cuda")
    m.step(None, x, None, 1.0, isTraining=False)
    torch.cuda.synchronize()
    with prof(activities=[ProfilerActivity.CUDA]) as pr:
        m.step(None, x, None, 1.0, isTraining=False)
        torch.cuda.synchronize()
    print(f"\nbf16x3, width 1024, one call at {B} poses: device time per kernel (all {B // 32768} row chunks)")
    rows = [(e.key, e.device_time_total, e.count) for e in pr.key_averages()]
    tot = sum(r[1] for r in rows)
    for k, t, c in sorted(rows, key=lambda r: -r[1]):
        if t > 0:
            print(f"  {t / 1e3:9.3f} ms  {100 * t / tot:5.1f}%  x{c:<5d} {k[:110]}")
    m.close()


def main():
    print(f"card: {card()}")
    quick = "--quick" in sys.argv
    shapes = [(1024, 2, [1, 64, 4096] if quick else [1, 64, 4096, 65536, 1 << 20])]
    if not quick:
        shapes.append((4096, 4, [1 << 18]))
        profile()
    run(shapes, ["bf16x3", "fp32", "bf16"])


if __name__ == "__main__":
    main()
