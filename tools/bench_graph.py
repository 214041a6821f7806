"""CUDA-graph replay against eager calls of LinearModel inference (LinearModel(1024, 2, residual, batch_norm, max_norm),
bf16, torch CUDA tensors).

    python tools/bench_graph.py [B ...]          (default: 1 64 4096)

Per batch size: median CUDA-event time of one call (eager model.step / one g.replay()), and the back-to-back time per
call over 1000 calls ending in a synchronise (what a caller that keeps the stream full sees: host overhead included).
The graph holds exactly what one eager step launches.  Prints the card name and power limit with the numbers."""
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "3d-pose-baseline_b200")]
from p3d import LinearModel  # noqa: E402

N = 1000


def timed(fn, st):
    for _ in range(100):
        fn()
    torch.cuda.synchronize()
    ev = []
    for _ in range(N):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(st)
        fn()
        b.record(st)
        b.synchronize()
        ev.append(a.elapsed_time(b) * 1e3)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(N):
        fn()
    torch.cuda.synchronize()
    return statistics.median(ev), (time.perf_counter() - t0) * 1e6 / N


def main():
    try:
        card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                              capture_output=True, text=True).stdout.strip().splitlines()[0]
    except Exception:
        card = "unknown"
    print(f"card: {card}")
    m = LinearModel(1024, 2, True, True, True, 64, 1e-3, seed=1)
    st = torch.cuda.current_stream()
    for B in [int(b) for b in (sys.argv[1:] or ["1", "64", "4096"])]:
        x = torch.randn((B, 32), device="cuda")

        def eager():
            m.step(None, x, None, 1.0, isTraining=False)
        eager()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            m.step(None, x, None, 1.0, isTraining=False)
        e_dev, e_b2b = timed(eager, st)
        g_dev, g_b2b = timed(g.replay, st)
        print(f"B={B}: eager p50 device {e_dev:.1f} us, back-to-back {e_b2b:.1f} us/call | "
              f"graph replay p50 device {g_dev:.1f} us, back-to-back {g_b2b:.1f} us/call")
        del g
    m.close()


if __name__ == "__main__":
    main()
