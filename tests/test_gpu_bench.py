"""bench.py --dump-outputs on the device: the sample of the timed step's predictions is the same in two runs, and it is
what the timed model computes for those rows (the fp64 oracle on the same weights and inputs, bf16 tolerance)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def dump(d):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0", "--no-secondary",
                        "--no-cpu-baseline", "--dump-outputs", str(d)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 1
    assert os.listdir(d) == ["y.npy"]
    return np.load(os.path.join(d, "y.npy"))


def test_dump_outputs_repeat_and_match_the_oracle(tmp_path):
    import torch

    import bench
    from oracle import mlp_ref as M
    a, b = dump(tmp_path / "a"), dump(tmp_path / "b")
    assert a.dtype == np.float32 and a.shape == (bench.DUMP_ROWS, bench.OUT)
    assert np.array_equal(a, b)
    m = bench.timed_model(0)
    p = {k: np.asarray(v, np.float64) for k, v in m.get_variables().items()}
    m.close()
    x = bench.timed_inputs(torch, torch.device("cuda", 0), 0).cpu().numpy()[bench.dump_rows(bench.B_PER_GPU)]
    ref = M.forward(p, x.astype(np.float64), M.Config(bench.L, bench.NL, True, True, True), training=False)
    rel = np.linalg.norm(a - ref, axis=1) / np.linalg.norm(ref, axis=1)
    assert rel.max() < 1e-2, rel.max()
