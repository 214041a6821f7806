"""fp16 inference mode against bf16 mode: speed, alternating in one process, and accuracy against fp32 mode.

    python tools/bench_fp16.py [--quick] [--rounds R]

LinearModel(1024, 2, residual, batch_norm, max_norm) at B = 1, 8, 64, 1024, 4096, 65536, 2^20 and
LinearModel(4096, 4, ...) at 2^18, the same trained-BN weights (oracle init, seed 1) in fp16, bf16 and fp32 mode, torch
CUDA tensors in and out.  Per shape: both modes warmed up, then R rounds (default 7) in which bf16 and fp16 take turns,
each timed by CUDA events over a run of back-to-back calls (about 0.2 s of work, 3 calls at least).  Printed: the
median ms per call of each mode, min / max over the rounds, and the fp16 / bf16 ratio of the medians.  Accuracy: the
row-wise max and median ||y - y_fp32|| / ||y_fp32|| of both modes on the timed rows (fp32 mode: the FFMA chain, within
1e-4 of the fp64 oracle).  The weights stay L2-resident between calls, as they do in use.  NVML samples the SM clock
and the board power every 5 ms during the timed runs: printed are each mode's median clock and mean power, and the
fp16 / bf16 ratio of time x clock (cycles per call), which separates a clock drop under the power limit from a
difference in the kernels.  The card's name, power limit and maximum SM clock are read in the same run."""
import os
import subprocess
import sys
import threading

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "3d-pose-baseline_b200")]
from oracle import mlp_ref as M  # noqa: E402
from p3d import LinearModel  # noqa: E402


def card():
    return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]


class Sampler(threading.Thread):
    """(SM MHz, board W) every 5 ms until stop()."""

    def __init__(self):
        super().__init__(daemon=True)
        import pynvml
        pynvml.nvmlInit()
        self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(torch.cuda.current_device())
        self.samples, self.done = [], threading.Event()
        self.start()

    def run(self):
        while not self.done.is_set():
            self.samples.append((self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM),
                                 self.nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0))
            self.done.wait(0.005)

    def stop(self):
        self.done.set()
        self.join()
        return self.samples


def timed(fn, budget_s=0.2):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    n = int(min(1000, max(3, budget_s / max(a.elapsed_time(b) / 1e3, 1e-6))))
    a.record()
    for _ in range(n):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / n


def rowwise(y, ref):
    y, ref = y.double(), ref.double()
    r = (y - ref).norm(dim=1) / ref.norm(dim=1).clamp_min(1e-30)
    return float(r.max()), float(r.median())


def model(L, nl, mode):
    p = {k: v.astype(np.float32) for k, v in M.init_params(L, nl, seed=1, bn="trained").items()}
    m = LinearModel(L, nl, True, True, True, 64, 1e-3, mode=mode, seed=1)
    m.set_variables(p)
    return m


def main():
    print(f"card (name, power limit, max SM clock): {card()}")
    quick = "--quick" in sys.argv
    rounds = int(sys.argv[sys.argv.index("--rounds") + 1]) if "--rounds" in sys.argv else 7
    shapes = [(1024, 2, [1, 8, 64, 1024, 4096] if quick else [1, 8, 64, 1024, 4096, 65536, 1 << 20])]
    if not quick:
        shapes.append((4096, 4, [1 << 18]))
    for L, nl, sizes in shapes:
        ms = {mode: model(L, nl, mode) for mode in ("fp32", "bf16", "fp16")}
        print(f"\nwidth {L}, {nl} blocks, residual, batch_norm, max_norm; {rounds} alternating rounds")
        print(f"{'B':>8} {'bf16 ms':>10} {'fp16 ms':>10} {'fp16/bf16':>10} {'bf16 min..max':>18} {'fp16 min..max':>18}"
              f"  {'bf16 err max / med':>20} {'fp16 err max / med':>20}  {'MHz bf16':>8} {'fp16':>6} {'W bf16':>6}"
              f" {'fp16':>6} {'cycles f/b':>8}")
        for B in sizes:
            x = torch.randn((B, 32), device="cuda", generator=torch.Generator(device="cuda").manual_seed(B))
            ys = {mode: m.step(None, x, None, 1.0, isTraining=False)[2].clone() for mode, m in ms.items()}
            calls = {mode: (lambda m=ms[mode]: m.step(None, x, None, 1.0, isTraining=False)) for mode in ("bf16", "fp16")}
            for f in calls.values():
                f()
                f()
            t = {"bf16": [], "fp16": []}
            smp = {"bf16": [], "fp16": []}
            for _ in range(rounds):
                for mode in ("bf16", "fp16"):
                    sm = Sampler()
                    t[mode].append(timed(calls[mode]))
                    smp[mode] += sm.stop()
            med = {k: float(np.median(v)) for k, v in t.items()}
            mhz = {k: float(np.median([c for c, _ in v])) for k, v in smp.items()}
            watt = {k: float(np.mean([w for _, w in v])) for k, v in smp.items()}
            eb, e16 = rowwise(ys["bf16"], ys["fp32"]), rowwise(ys["fp16"], ys["fp32"])
            print(f"{B:8d} {med['bf16']:10.4f} {med['fp16']:10.4f} {med['fp16'] / med['bf16']:10.3f}"
                  f" {min(t['bf16']):8.4f}..{max(t['bf16']):8.4f} {min(t['fp16']):8.4f}..{max(t['fp16']):8.4f}"
                  f"  {eb[0]:9.2e} / {eb[1]:8.2e} {e16[0]:9.2e} / {e16[1]:8.2e}"
                  f"  {mhz['bf16']:6.0f} {mhz['fp16']:6.0f} {watt['bf16']:6.0f} {watt['fp16']:6.0f}"
                  f" {med['fp16'] * mhz['fp16'] / (med['bf16'] * mhz['bf16']):8.3f}", flush=True)
        for m in ms.values():
            m.close()


if __name__ == "__main__":
    main()
