"""CPU half of action-wise evaluation (p3d.evaluate.stage_actions / evaluate_actions):
  * the host staging against the reference-style loop of get_action_subset + the existing get_all_batches, bit-exact,
    on a synthetic test set of several subjects and actions with '-sh' keys (camera frame) and world-frame keys;
  * the NumPy restatement of the per-action loop (oracle/eval_actions_ref.py) against per-action oracle MPJPE calls;
  * the data-parallel agreement check on two gloo ranks.
tests/test_gpu_eval_actions.py runs the kernel and the end-to-end call on the GPU."""
import os
import socket

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import eval_actions_ref as R
from oracle import geometry_ref as G

ACTIONS = ["Directions", "Eating", "Walking", "Sitting"]


def _host_model(batch_size, out=48):
    from p3d.linear_model import LinearModel
    m = LinearModel.__new__(LinearModel)       # host-side methods only: no device, no library call
    m._handle = None
    m.input_size, m.output_size, m.batch_size = 32, out, batch_size
    return m


def _test_set(camera_frame, seed=0):
    """2D and 3D dicts keyed (subject, action, file) as data_utils builds them; interleaved actions, uneven sizes."""
    rng = np.random.RandomState(seed)
    d2, d3 = {}, {}
    sizes = {(subj, action): int(rng.randint(3, 40)) for subj in (9, 11) for action in ACTIONS + ["Photo"]}
    for subj in (9, 11):
        for cam in ("54138969", "55011271"):
            for action in ACTIONS + ["Photo"]:
                n = sizes[(subj, action)]     # every camera sees the same frames
                f2 = "%s 1.%s.h5-sh" % (action, cam)
                d2[(subj, action, f2)] = rng.standard_normal((n, 32))
                f3 = f2[:-3] if camera_frame else "%s 1.h5" % action
                d3.setdefault((subj, action, f3), rng.standard_normal((n, 48)))
    return d2, d3


def _reference_loop(model, d2, d3, actions, camera_frame):
    from p3d.evaluate import get_action_subset
    xs, ts = [], []
    for action in actions:
        enc, dec = model.get_all_batches(get_action_subset(d2, action), get_action_subset(d3, action), camera_frame,
                                         training=False)
        xs.append(np.concatenate(enc, 0)); ts.append(np.concatenate(dec, 0))
    return xs, ts


def test_get_action_subset_keeps_order():
    from p3d.evaluate import get_action_subset
    d2, _ = _test_set(True)
    sub = get_action_subset(d2, "Eating")
    assert list(sub) == [k for k in d2 if k[1] == "Eating"] and all(sub[k] is d2[k] for k in sub)
    assert get_action_subset(d2, "Smoking") == {}


@pytest.mark.parametrize("camera_frame", [True, False], ids=["camera-sh", "world"])
def test_staging_matches_the_reference_loop(camera_frame):
    from p3d.evaluate import stage_actions_host
    d2, d3 = _test_set(camera_frame)
    m = _host_model(8)
    actions = ["Walking", "Directions", "Eating"]            # not the dict order: the staging follows `actions`
    s = stage_actions_host(m, d2, d3, actions, camera_frame)
    xs, ts = _reference_loop(m, d2, d3, actions, camera_frame)
    assert s.actions == actions and s.batch_size == 8
    assert s.offsets.tolist() == np.concatenate([[0], np.cumsum([x.shape[0] for x in xs])]).tolist()
    assert s.batches == [x.shape[0] // 8 for x in xs] and all(x.shape[0] % 8 == 0 for x in xs)
    assert s.X.dtype == np.float32 and s.T.dtype == np.float32
    assert np.array_equal(s.X, np.concatenate(xs).astype(np.float32))
    assert np.array_equal(s.T, np.concatenate(ts).astype(np.float32))


def test_staging_without_tail_drop_keeps_every_pose():
    from p3d.evaluate import get_action_subset, stage_actions_host
    d2, d3 = _test_set(True, seed=1)
    m = _host_model(8)
    s = stage_actions_host(m, d2, d3, ACTIONS, True, drop_tail=False)
    ns = [sum(v.shape[0] for v in get_action_subset(d2, a).values()) for a in ACTIONS]
    assert np.diff(s.offsets).tolist() == ns and s.batches == [-(-n // 8) for n in ns]
    # every pose, in get_all_batches order: with a batch of 1 get_all_batches drops nothing
    xs, ts = _reference_loop(_host_model(1), d2, d3, ACTIONS, True)
    assert np.array_equal(s.X, np.concatenate(xs).astype(np.float32))
    assert np.array_equal(s.T, np.concatenate(ts).astype(np.float32))


def test_staging_refusals():
    from p3d.evaluate import stage_actions_host
    d2, d3 = _test_set(True)
    with pytest.raises(ValueError, match="Smoking"):
        stage_actions_host(_host_model(8), d2, d3, ["Eating", "Smoking"], True)
    few, few3 = {k: v[:2] for k, v in d2.items()}, {k: v[:2] for k, v in d3.items()}   # 4 entries x 2 poses per action
    with pytest.raises(ValueError, match="Eating.*fewer than batch_size 9"):
        stage_actions_host(_host_model(9), few, few3, ["Eating"], True)
    s = stage_actions_host(_host_model(9), few, few3, ["Eating"], True, drop_tail=False)
    assert s.offsets.tolist() == [0, 8]
    with pytest.raises(ValueError):
        stage_actions_host(_host_model(8), d2, d3, [], True)
    with pytest.raises(ValueError):
        stage_actions_host(_host_model(8), d2, d3, ["Eating", "Eating"], True)


@pytest.mark.parametrize("p14", [False, True])
@pytest.mark.parametrize("use_proc", [False, True])
def test_oracle_per_action_loop(p14, use_proc):
    """The restated loop (one batched pass, split by offsets) == one oracle mpjpe call per action."""
    rng = np.random.RandomState(7)
    width = 42 if p14 else 48
    mean3d, std3d = rng.standard_normal(96) * 100, rng.uniform(20, 200, 96)
    use3, ign3 = G.dims_to_use(3, p14)
    offsets = np.array([0, 64, 64 + 128, 64 + 128 + 8, 64 + 128 + 8 + 256])
    gt = rng.standard_normal((offsets[-1], width))
    pred = (gt + 0.1 * rng.standard_normal(gt.shape)).astype(np.float32)
    errors, joints, losses, avg = R.evaluate_actions(pred, gt, offsets, mean3d, std3d, ign3, use3, use_proc, p14)
    for a in range(offsets.size - 1):
        sl = slice(offsets[a], offsets[a + 1])
        d = G.mpjpe(pred[sl], gt[sl], mean3d, std3d, ign3, use3, procrustes=use_proc, predict_14=p14)
        assert abs(errors[a] - d.mean()) < 1e-9 * d.mean()
        np.testing.assert_allclose(joints[a], d.mean(axis=0), rtol=1e-12, atol=1e-12)
        # evaluate_batches' loss: the mean of per-batch MSEs of equal batches (8 rows each here)
        bl = [np.mean((pred[i:i + 8].astype(np.float64) - gt[i:i + 8]) ** 2) for i in range(offsets[a], offsets[a + 1], 8)]
        assert abs(losses[a] - np.mean(bl)) < 1e-12 * np.mean(bl)
    assert abs(avg - np.mean(errors)) < 1e-12


# ---------------------------------------------------------------------------------------------- two gloo ranks
CASES = [  # per rank: (n, S, batch_size, offsets checksum, own error) -> expected outcome on every rank
    ("agree", [(1000, 15, 64, 123.0, None), (1000, 15, 64, 123.0, None)], "ok"),
    ("n", [(1000, 15, 64, 123.0, None), (992, 15, 64, 123.0, None)], "n 992..1000"),
    ("actions", [(1000, 15, 64, 123.0, None), (1000, 14, 64, 123.0, None)], "actions 14..15"),
    ("batch_size", [(1000, 15, 64, 123.0, None), (1000, 15, 128, 123.0, None)], "batch_size 64..128"),
    ("offsets", [(1000, 15, 64, 123.0, None), (1000, 15, 64, 124.0, None)], "offsets checksum"),
    ("rejected", [(1000, 15, 64, 123.0, None), (1000, 15, 64, 123.0, "bad precision")], "rejected|bad precision"),
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
    from p3d import evaluate
    out = {}
    for name, args, _ in CASES:
        n, S, B, ck, err = args[rank]
        try:
            evaluate._dp_agree(dist, 0, [n, S, B, ck], ("n", "actions", "batch_size", "offsets checksum"), err,
                               "evaluate_actions")
            out[name] = "ok"
        except ValueError as e:
            out[name] = "ValueError: " + str(e)
    q.put((rank, out))
    dist.destroy_process_group()


def test_offsets_checksum_sees_a_moved_boundary():
    from p3d.evaluate import _offsets_checksum
    a = _offsets_checksum([0, 100, 200, 300])
    assert a == _offsets_checksum(np.array([0, 100, 200, 300]))
    assert a != _offsets_checksum([0, 101, 200, 300]) and a != _offsets_checksum([0, 200, 100, 300])


def test_mismatched_action_sets_raise_on_every_rank():
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
