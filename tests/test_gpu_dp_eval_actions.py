"""Data-parallel evaluate_actions on two GPUs (skipped on a single-GPU box): torchrun spawns two ranks of
tools/dp_eval_actions_check.py - the same numbers as one GPU, identical results on both ranks, ragged shards, ValueError
on every rank for mismatched sets.  tests/test_eval_actions_cpu.py covers the agreement check on CPU (gloo)."""
import os
import socket
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
@pytest.mark.parametrize("p2p", ["1", "0"], ids=["peer-memory", "nccl-only"])
def test_two_rank_action_wise_evaluation(p2p):
    env = dict(os.environ, P3D_P2P=p2p, P3D_SYNC_TIMEOUT_S="60")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(free_port()), os.path.join(ROOT, "tools", "dp_eval_actions_check.py")]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "DP EVAL ACTIONS CHECK OK" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
