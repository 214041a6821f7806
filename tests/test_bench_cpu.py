"""bench.py's contract as far as a box without a GPU can check it: the reference arm (the CPU restatement of the
reference graph, the one place besides the tests where oracle/ is executed) prints ONE JSON line with the keys the
driver reads; our arm refuses to run without a CUDA device instead of falling back to anything."""
import json
import os
import re
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*flags, env=None):
    e = dict(os.environ, **(env or {}))
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *flags], capture_output=True, text=True, env=e, timeout=600)


def test_reference_arm_prints_one_json_line_with_the_contract_keys(tmp_path):
    r = run_bench("--impl", "reference", "--steps", "2", "--warmup", "1", "--dump-outputs", str(tmp_path),
                  env={"P3D_BENCH_REF_BUDGET_S": "6"})
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"].startswith("poses/sec") and d["unit"] == "poses/s"
    assert d["higher_is_better"] is True and d["steps"] == 2 and d["warmup"] == 1 and d["n_gpus"] == 1
    assert d["value"] > 0 and abs(d["value"] - d["config"]["sample_poses"] / (d["ms_per_step"] * 1e-3)) <= 1e-6 * d["value"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "poses per step" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "poses/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"].startswith("LinearModel(linear_size=1024,num_layers=2")
    # --dump-outputs: the last step's predictions of the first 4096 poses, whatever the sample size, as the oracle
    # computes them from the same weights and inputs
    from oracle import mlp_ref as M
    from oracle import synth
    assert os.listdir(tmp_path) == ["y.npy"]
    y = np.load(tmp_path / "y.npy")
    assert y.dtype == np.float32 and y.shape == (4096, 48)
    p = {k: v.astype(np.float32) for k, v in M.init_params(1024, 2, seed=1, bn="trained").items()}
    x, _ = synth.mlp_inputs(4096, seed=0)
    ref = M.forward(p, x, M.Config(1024, 2, True, True, True), training=False)
    np.testing.assert_allclose(y, ref, rtol=1e-5, atol=1e-5)


def test_steps_below_one_are_refused():
    r = run_bench("--impl", "reference", "--steps", "0")
    assert r.returncode == 2 and "--steps" in r.stderr


def test_our_arm_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is present: the arm runs")
    r = run_bench("--steps", "1", "--warmup", "1")
    assert r.returncode == 2
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert "no CUDA device" in d["error"]


def test_design_switch_table_names_every_environment_variable_the_library_reads():
    """DESIGN.md section 6 is the list of run-time switches: every getenv("P3D_...") in csrc/ and every P3D_ variable the
    Python host layer reads must appear there (a switch that exists but is not documented is how unmeasured paths hide)."""
    names = set()
    csrc = os.path.join(ROOT, "3d-pose-baseline_b200", "csrc")
    for f in os.listdir(csrc):
        with open(os.path.join(csrc, f)) as fh:
            names.update(re.findall(r'getenv\("(P3D_[A-Z0-9_]+)"\)', fh.read()))
    pkg = os.path.join(ROOT, "3d-pose-baseline_b200", "p3d")
    for f in os.listdir(pkg):
        if f.endswith(".py"):
            with open(os.path.join(pkg, f)) as fh:
                names.update(re.findall(r'environ(?:\.get)?[\(\[]"(P3D_[A-Z0-9_]+)"', fh.read()))
    assert len(names) >= 20
    with open(os.path.join(ROOT, "DESIGN.md")) as fh:
        design = fh.read()
    table = design[design.index("## 6. Run-time switches"):]
    # the table abbreviates families as `P3D_GEMM_DBG_PTR`, `_MODE`, `_LAYER`: expand "`_X`" against the last full name
    documented, last = set(), None
    for tok in re.findall(r"`(P3D_[A-Z0-9_]+|_[A-Z0-9_]+)(?:=[^`]*)?`", table):
        if tok.startswith("P3D_"):
            documented.add(tok); last = tok
        elif last:
            documented.add(last.rsplit("_", 1)[0] + tok)
    missing = sorted(n for n in names if n not in documented)
    assert not missing, f"switches read by the code but absent from DESIGN.md section 6: {missing}"
