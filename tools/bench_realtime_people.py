"""Host wall clock of lifting every person of one realtime frame (keypoints on the host -> un-normalised 3D poses on the
host), linear_size 1024, bf16, for P people per frame:
  people      RealtimeLifter.step_people: one cluster-kernel launch for P <= 8 (the staged batched step above 8)
  sequential  P calls of RealtimeLifter.step, one launch and one flag spin each
  batch       RealtimeLifter.step_batch on a NumPy [P,36] array (uploads, three launches, downloads, a synchronise)
time.perf_counter around each Python call, p50 / p99 over N calls per arm after warm-up; the arms alternate in rounds
of 100 calls.  Prints one JSON line with the card name, power limit and SM clock read in the same run.

    python tools/bench_realtime_people.py [N]"""
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "3d-pose-baseline_b200")]
from p3d import LinearModel  # noqa: E402
from p3d.realtime import RealtimeLifter  # noqa: E402

N = int(sys.argv[1]) if len(sys.argv) > 1 else 5000
ROUND = 100


def smi():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(","), [v.strip() for v in out.split(",")]))
    except Exception as e:                      # the timing does not depend on it; say what is missing
        return {"error": str(e)}


g = np.load(os.path.join(ROOT, "tests", "golden", "realtime.npz"))
m2, s2, use2, m3, s3, use3 = (g[k] for k in ["mean2d", "std2d", "use2d", "mean3d", "std3d", "use3d"])
model = LinearModel(1024, 2, True, True, True, 64, 1e-3, seed=1)
lifter = RealtimeLifter(model, m2, s2, use2, m3, s3, use3)
rng = np.random.RandomState(0)
frames = rng.uniform(100, 900, size=(16, 16, 36))          # 16 different frames of up to 16 people


def arms(P):
    def people(kp):
        return lifter.step_people(kp)

    def sequential(kp):
        return [lifter.step(kp[i]) for i in range(P)]

    def batch(kp):
        return lifter.step_batch(kp)
    return {"step_people": people, "sequential_step": sequential, "step_batch": batch}


def bench(P):
    fns = arms(P)
    # the three arms compute the same people: equal per person for P <= 8 (one launch), step_batch's route above
    a, b, c = (fns[k](frames[0, :P]) for k in fns)
    same_single = all(np.array_equal(a[2][i], b[i][2][0]) for i in range(P))
    same_batch = bool(np.array_equal(a[2], c[2]))
    for f in fns.values():                                   # warm-up
        for i in range(200):
            f(frames[i % 16, :P])
    t = {k: [] for k in fns}
    done = 0
    while done < N:
        for k, f in fns.items():
            for i in range(done, done + ROUND):
                kp = frames[i % 16, :P]
                t0 = time.perf_counter()
                f(kp)
                t[k].append((time.perf_counter() - t0) * 1e6)
        done += ROUND
    res = {"P": P, "equal_to_step": bool(same_single), "equal_to_step_batch": same_batch}
    for k, v in t.items():
        v.sort()
        res[k] = {"p50_us": round(statistics.median(v), 2), "p99_us": round(v[int(0.99 * len(v))], 2)}
    return res


card = smi()
rows = [bench(P) for P in (1, 2, 4, 8, 16)]
print(json.dumps({"workload": "every person of one realtime frame, host keypoints -> host 3D poses (linear_size 1024, "
                              "bf16), host wall clock through the Python call", "calls_per_arm": N, "gpu": card,
                  "gpu_after": smi(), "rows": rows}))
lifter.close()
model.close()
