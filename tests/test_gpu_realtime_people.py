"""Every person of a realtime frame in one launch (RealtimeLifter.step_people, p3d_realtime_step_people_host): bit
identity to one-person frames, the reference lines around the lifter, the launch count per route, the staged route,
the mapped-flag protocol across calls, predict_14 and the refusals."""
import ctypes as C
import os

import numpy as np
import pytest

from helpers import emulate_bf16_forward, make_model, rowwise_rel
from oracle import geometry_ref as G, mlp_ref as M

pytestmark = pytest.mark.gpu
CASES = ["coco54", "tfpose36", "body25_75", "wide_87"]


@pytest.fixture(scope="module")
def gold(golden_dir):
    return np.load(os.path.join(golden_dir, "realtime.npz"))


def _lifter(model, gold, use3=None):
    from p3d.realtime import RealtimeLifter
    return RealtimeLifter(model, gold["mean2d"], gold["std2d"], gold["use2d"], gold["mean3d"], gold["std3d"],
                          gold["use3d"] if use3 is None else use3)


def _launches():
    from p3d import _lib
    return _lib.lib.p3d_launch_count()


def _equal(a, b):
    return all(np.array_equal(x, y) for x, y in zip(a, b))


@pytest.mark.parametrize("mode", ["bf16", "fp16"])
@pytest.mark.parametrize("num_layers,residual", [(2, True), (1, False)])
def test_people_equal_single_frames(gold, mode, num_layers, residual):
    """Per person, enc / y / pose of one launch for P people equal that person's one-person frame exactly."""
    cfg = M.Config(1024, num_layers, residual, True, True)
    model, _ = make_model(cfg, seed=21, mode=mode)           # trained BatchNorm statistics
    lifter = _lifter(model, gold)
    kp = np.random.RandomState(7).uniform(50, 950, size=(8, 40))
    single = [lifter.step(kp[i]) for i in range(8)]
    for P in range(1, 9):
        l0 = _launches()
        enc, y, pose = lifter.step_people(kp[:P])
        assert _launches() - l0 == 1
        assert enc.shape == (P, 32) and y.shape == (P, 48) and pose.shape == (P, 96)
        for i in range(P):
            assert np.array_equal(enc[i], single[i][0][0])
            assert np.array_equal(y[i], single[i][1][0])
            assert np.array_equal(pose[i], single[i][2][0])
    # lists of different lengths (only the first 36 values count)
    xys = [kp[0].tolist(), kp[1, :36].tolist(), kp[2].tolist() + [1.0, 2.0]]
    assert _equal(lifter.step_people(xys), lifter.step_people(kp[:3]))
    lifter.close()
    model.close()


@pytest.mark.parametrize("mode", ["bf16", "fp16"])
def test_people_match_reference_lines(gold, mode):
    """The 12 golden frames as groups of up to 8 people: front-end and back-end bit exact, the lifter within the mode's
    tolerances of the oracle and the weights-only emulation."""
    from p3d.realtime import keypoints_to_xy
    cfg = M.Config(1024, 2, True, True, True)
    model, p = make_model(cfg, seed=3, mode=mode)
    lifter = _lifter(model, gold)
    m3, s3, ig3 = gold["mean3d"], gold["std3d"], gold["ignore3d"]
    frames = [(case, f) for case in CASES for f in range(3)]
    for g0 in (0, 8):
        group = frames[g0:g0 + 8]
        xys = [keypoints_to_xy(gold["%s_kp%d" % cf].tolist()) for cf in group]
        enc, y, pose = lifter.step_people(xys)
        want_enc = np.concatenate([gold["%s_enc%d" % cf] for cf in group])
        assert np.array_equal(enc, want_enc.astype(np.float32))
        assert np.array_equal(pose, G.unnormalize(y, m3, s3, ig3))
        ref = M.forward(p, enc.astype(np.float64), cfg, training=False)
        if mode == "bf16":
            assert rowwise_rel(y, ref).max() <= 1e-2
            assert rowwise_rel(y, emulate_bf16_forward(p, enc, cfg, small_batch=True)).max() <= 2e-3
        else:
            from test_oracle_fp16 import CONTRACT, emulate_fp16_forward
            assert rowwise_rel(y, ref).max() <= CONTRACT
            assert rowwise_rel(y, emulate_fp16_forward(p, enc, cfg, small_batch=True)).max() <= 3e-4
    lifter.close()
    model.close()


def _staged_check(lifter, kp):
    """step_people on the staged route equals step_batch on the same keypoints, with the same launch count."""
    lifter.step_batch(kp)                                    # the weight fold and buffer growth outside the counts
    l0 = _launches()
    want = lifter.step_batch(kp)
    n_batch = _launches() - l0
    l0 = _launches()
    got = lifter.step_people(kp)
    assert _launches() - l0 == n_batch
    assert _equal(got, want)
    return got


@pytest.mark.parametrize("P", [9, 33, 300])
def test_staged_many_people(gold, P):
    cfg = M.Config(1024, 2, True, True, True)
    model, p = make_model(cfg, seed=5)
    lifter = _lifter(model, gold)
    kp = np.random.RandomState(P).uniform(50, 950, size=(P, 36))
    enc, y, pose = _staged_check(lifter, kp)
    assert rowwise_rel(y, M.forward(p, enc.astype(np.float64), cfg, training=False)).max() <= 1e-2
    lifter.close()
    model.close()


@pytest.mark.parametrize("width,mode,tol", [(256, "bf16", 1e-2), (1024, "fp32", 1e-4), (1024, "bf16x3", 1e-4)])
def test_staged_other_models(gold, width, mode, tol):
    """Models the cluster kernel does not serve: every P takes the staged route."""
    cfg = M.Config(width, 2, True, True, True)
    model, p = make_model(cfg, seed=9, mode=mode)
    lifter = _lifter(model, gold)
    kp = np.random.RandomState(1).uniform(50, 950, size=(8, 36))
    for P in (1, 3, 8):
        enc, y, pose = _staged_check(lifter, kp[:P])
        if P == 1:                                           # one person: the same route as step()
            assert _equal((enc, y, pose), lifter.step(kp[0]))
        assert rowwise_rel(y, M.forward(p, enc.astype(np.float64), cfg, training=False)).max() <= tol
    lifter.close()
    model.close()


def test_flag_protocol_across_calls(gold):
    """200 calls cycling P through 1..8, interleaved with the other entry points, repeat their first results; a weight
    change is seen by the next call."""
    import torch
    cfg = M.Config(1024, 2, True, True, True)
    model, _ = make_model(cfg, seed=4)
    lifter = _lifter(model, gold)
    kp = np.random.RandomState(3).uniform(50, 950, size=(8, 36))
    x = np.random.RandomState(4).normal(size=(5, 32)).astype(np.float32)
    first, others = {}, {}
    for it in range(200):
        P = 1 + it % 8
        got = lifter.step_people(kp[:P])
        if P not in first:
            first[P] = got
        assert _equal(got, first[P]), (it, P)
        kind = it % 3
        if kind == 0:
            res = lifter.step(kp[it % 8])
            key = ("step", it % 8)
        elif kind == 1:
            res = lifter.step_batch(kp[:1 + it % 5])
            key = ("batch", it % 5)
        else:
            res = model.step(None, x, np.zeros((5, 48)), 1.0, isTraining=False)[2]
            res = (res.cpu().numpy() if isinstance(res, torch.Tensor) else res,)
            key = ("model",)
        others.setdefault(key, res)
        assert _equal(res, others[key]), (it, key)
    before = lifter.step_people(kp)
    model.set_variable("linear_model/b4", np.zeros(48, dtype=np.float32))
    after = lifter.step_people(kp)
    assert not np.array_equal(after[1], before[1])
    for i in range(8):
        assert _equal([a[i:i + 1] for a in after], lifter.step(kp[i]))
    lifter.close()
    model.close()


def test_predict_14(gold, golden_dir):
    tab = np.load(os.path.join(golden_dir, "tables.npz"))
    cfg = M.Config(1024, 2, True, True, True)
    model, _ = make_model(cfg, seed=6, predict_14=True)
    lifter = _lifter(model, gold, use3=tab["use3d_14"])
    ig = np.asarray(tab["ignore3d_14"])
    kp = np.random.RandomState(2).uniform(50, 950, size=(8, 36))
    for P in (1, 5, 8):
        enc, y, pose = lifter.step_people(kp[:P])
        assert y.shape == (P, 42)
        assert np.array_equal(pose[:, ig], np.broadcast_to(gold["mean3d"][ig], (P, ig.size)))
        assert np.array_equal(pose, G.unnormalize(y, gold["mean3d"], gold["std3d"], ig))
        for i in range(P):
            assert _equal([a[i:i + 1] for a in (enc, y, pose)], lifter.step(kp[i]))
    lifter.close()
    model.close()


def test_refusals_and_edges(gold):
    from p3d import _lib
    cfg = M.Config(1024, 2, True, True, True)
    model, _ = make_model(cfg, seed=8)
    lifter = _lifter(model, gold)
    kp = np.random.RandomState(5).uniform(50, 950, size=(3, 36))
    lifter.step_people(kp)                                   # fold and first launch outside the counts
    l0 = _launches()
    enc, y, pose = lifter.step_people([])
    assert enc.shape == (0, 32) and y.shape == (0, 48) and pose.shape == (0, 96)
    assert enc.dtype == np.float32 and y.dtype == np.float32 and pose.dtype == np.float64
    assert _launches() == l0
    with pytest.raises(IndexError):
        lifter.step_people([kp[0].tolist(), kp[1, :35].tolist()])
    assert _launches() == l0
    buf = np.zeros((1, 96))
    rc = _lib.lib.p3d_realtime_step_people_host(lifter._handle, _lib.np_ptr(kp), -1, None, None, _lib.np_ptr(buf))
    assert rc == -1                                          # P3D_ERR_ARG
    rc = _lib.lib.p3d_realtime_step_people_host(lifter._handle, None, 1, None, None, _lib.np_ptr(buf))
    assert rc == -1
    assert _launches() == l0
    lifter.close()
    with pytest.raises(RuntimeError):
        lifter.step_people(kp)
    model.close()
