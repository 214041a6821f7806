"""world_size-2 gloo test (CPU) of the argument check a data-parallel LinearModel.train_epoch runs before it launches
anything: ranks that pass different sizes, or a rank that rejects its own arguments, make EVERY rank raise ValueError
instead of leaving the others in a collective.  tests/test_gpu_dp_epoch.py runs the epoch itself on two GPUs."""
import os
import socket
import types

import torch.distributed as dist
import torch.multiprocessing as mp

CASES = [  # per rank: (n, batch_size, keep_prob, permuted, own error) -> expected outcome on every rank
    ("agree", [(1000, 64, 0.5, True, None), (1000, 64, 0.5, True, None)], "ok"),
    ("n", [(1000, 64, 0.5, True, None), (999, 64, 0.5, True, None)], "n 999..1000"),
    ("batch_size", [(1000, 64, 0.5, True, None), (1000, 128, 0.5, True, None)], "batch_size 64..128"),
    ("keep_prob", [(1000, 64, 0.5, True, None), (1000, 64, 1.0, True, None)], "dropout_keep_prob"),
    ("shuffle", [(1000, 64, 0.5, True, None), (1000, 64, 0.5, False, None)], "shuffle or perm"),
    ("rejected", [(1000, 64, 0.5, True, None), (1000, 64, 0.5, True, "bad shape")], "rejected|bad shape"),
]


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, q):
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path[:0] = [root, os.path.join(root, "3d-pose-baseline_b200")]
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from p3d.linear_model import LinearModel
    out = {}
    for name, args, _ in CASES:
        n, B, keep, permuted, err = args[rank]
        fake = types.SimpleNamespace(_dist=dist, batch_size=B, device=0)
        try:
            LinearModel._dp_epoch_agree(fake, n, keep, permuted, err)
            out[name] = "ok"
        except ValueError as e:
            out[name] = "ValueError: " + str(e)
    q.put((rank, out))
    dist.destroy_process_group()


def test_mismatched_epoch_arguments_raise_on_every_rank():
    import re
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for name, _, want in CASES:
        for rank in range(2):
            got = res[rank][name]
            if want == "ok":
                assert got == "ok", (name, rank, got)
            else:
                assert got.startswith("ValueError") and re.search(want, got), (name, rank, got)
