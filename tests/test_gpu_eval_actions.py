"""Action-wise evaluation on the GPU: p3d_mpjpe_segments[_f64] against the unsegmented evaluation kernels and the
executed reference (tests/golden/driver.npz), and evaluate_actions against the reference-style per-action loop over
evaluate_batches.  tests/test_eval_actions_cpu.py covers the host staging and the data-parallel agreement check."""
import os

import numpy as np
import pytest
import torch

from oracle import synth

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)


def _stats(seed=5):
    rng = np.random.RandomState(seed)
    return rng.standard_normal(96) * 100, rng.uniform(20, 200, 96)


def _pairs(n, width, seed=0):
    rng = np.random.RandomState(seed)
    gt = rng.standard_normal((n, width)).astype(np.float32)
    pred = (gt + 0.2 * rng.standard_normal(gt.shape)).astype(np.float32)
    return torch.from_numpy(pred).to(DEV), torch.from_numpy(gt).to(DEV)


def _segments(pred, gt, mean, std, p14, kinds, offsets, row0=0, precision="fp32", rows=None):
    """Raw call: rows [row0, row0 + len) of the global table; returns (rc, sums[S, 2J+1])."""
    from p3d import _lib
    fn = _lib.lib.p3d_mpjpe_segments if precision == "fp32" else _lib.lib.p3d_mpjpe_segments_f64
    offs = np.ascontiguousarray(offsets, dtype=np.int64)
    S = max(offs.size - 1, 1)
    J = 14 if p14 else 17
    sums = torch.zeros((S, 2 * J + 1), dtype=torch.float64, device=DEV)
    N = pred.shape[0] if rows is None else rows
    rc = fn(pred.data_ptr(), gt.data_ptr(), _lib.np_ptr(np.ascontiguousarray(mean)), _lib.np_ptr(np.ascontiguousarray(std)),
            int(p14), kinds, N, row0, _lib.np_ptr(offs), offs.size - 1, sums.data_ptr(), _lib.current_stream())
    return rc, sums.cpu().numpy()


def _layouts(N):
    """name -> ascending offsets covering [0, N)."""
    rng = np.random.RandomState(1)
    residues = np.cumsum([32 + r for r in range(32)])          # a boundary at every residue mod 32
    ones = np.arange(0, 40)                                     # 1-pose segments at the start
    mid = np.arange(1000, 1040)                                 # and 1-pose segments in the middle
    big = np.sort(rng.choice(np.arange(1, N), 1023, replace=False))
    return {
        "one": np.array([0, N]),
        "residues": np.concatenate([[0], residues[residues < N], [N]]),
        "singles": np.unique(np.concatenate([ones, mid, [N]])),
        "S1024": np.concatenate([[0], big, [N]]),
        "empty": np.array([0, 10, 10, 500, 500, N]),
    }


N_SEG = 4133


@pytest.mark.parametrize("precision", ["fp32", "fp64"])
@pytest.mark.parametrize("p14", [False, True])
def test_segments_against_the_unsegmented_kernel(p14, precision):
    from p3d import evaluate
    width, J = (42, 14) if p14 else (48, 17)
    mean, std = _stats()
    pred, gt = _pairs(N_SEG, width)
    ref_sq = ((pred.double() - gt.double()) ** 2).sum(1).cpu().numpy()
    # fp32: lane partials of up to 64 poses in fp32, grouped by tile position, which the segment start shifts
    rtol = 1e-6 if precision == "fp32" else 1e-9
    for name, offs in _layouts(N_SEG).items():
        assert offs.size - 1 <= 1024
        runs = {k: _segments(pred, gt, mean, std, p14, k, offs, precision=precision) for k in (1, 2, 3)}
        for k, (rc, s) in runs.items():
            assert rc == 0, (name, k)
        for a in range(offs.size - 1):
            lo, hi = int(offs[a]), int(offs[a + 1])
            for k, first in ((1, 0), (2, J)):
                got = runs[k][1][a]
                if hi == lo:
                    assert not got.any(), (name, a)
                    continue
                _, joint = evaluate.mpjpe(pred[lo:hi].clone(), gt[lo:hi].clone(), mean, std, procrustes=k == 2, predict_14=p14,
                                          precision=precision)
                np.testing.assert_allclose(got[first:first + J], joint * (hi - lo), rtol=rtol, atol=1e-9,
                                           err_msg="%s seg %d kind %d" % (name, a, k))
                assert not got[J - first:2 * J - first].any()          # the other kind is left untouched
                np.testing.assert_allclose(got[2 * J], ref_sq[lo:hi].sum(), rtol=1e-6, atol=1e-9)
                # kinds = 3: each half equals the single-kind run
                np.testing.assert_allclose(runs[3][1][a][first:first + J], got[first:first + J], rtol=rtol, atol=1e-9)
            np.testing.assert_allclose(runs[3][1][a][2 * J], runs[1][1][a][2 * J], rtol=1e-6, atol=1e-9)


@pytest.mark.parametrize("precision", ["fp32", "fp64"])
@pytest.mark.parametrize("p14", [False, True])
def test_row0_scores_a_row_block_against_the_global_table(p14, precision):
    width, J = (42, 14) if p14 else (48, 17)
    mean, std = _stats()
    pred, gt = _pairs(N_SEG, width, seed=2)
    offs = _layouts(N_SEG)["residues"]
    _, whole = _segments(pred, gt, mean, std, p14, 3, offs, precision=precision)
    acc = np.zeros_like(whole)
    for lo, hi in ((0, 1030), (1030, 2502), (2502, N_SEG)):        # even starts: 42-wide rows stay 16-byte aligned
        rc, part = _segments(pred[lo:], gt[lo:], mean, std, p14, 3, offs, row0=lo, precision=precision, rows=hi - lo)
        assert rc == 0
        touched = np.nonzero(part.any(axis=1))[0]
        assert offs[touched.min()] <= lo and offs[touched.max() + 1] >= hi        # only the block's own segments
        acc += part
    np.testing.assert_allclose(acc, whole, rtol=1e-6 if precision == "fp32" else 1e-9, atol=1e-9)


@pytest.mark.parametrize("p14", [False, True])
def test_golden_driver_cases_one_segment_and_per_batch(golden_dir, p14):
    """The reference's executed evaluate_batches (tests/test_gpu_zz_driver_golden.py's tolerances)."""
    drv = np.load(os.path.join(golden_dir, "driver.npz"))
    tag, width, J = ("p14", 42, 14) if p14 else ("p17", 48, 17)
    dec, pred = drv["evb_%s_dec" % tag], drv["evb_%s_pred" % tag]
    NB, B = dec.shape[:2]
    gt_d = torch.from_numpy(dec.reshape(-1, width).astype(np.float32)).to(DEV)
    pr_d = torch.from_numpy(pred.reshape(-1, width)).to(DEV)
    for precision in ("fp32", "fp64"):
        for offs in (np.array([0, NB * B]), np.arange(NB + 1) * B):
            rc, s = _segments(pr_d, gt_d, drv["mean3d"], drv["std3d"], p14, 3, offs, precision=precision)
            assert rc == 0
            tot = s.sum(axis=0)
            for pt, first in (("plain", 0), ("proc", J)):
                joint = tot[first:first + J] / (NB * B)
                assert abs(joint.sum() / J - float(drv["evb_%s_%s_total" % (tag, pt)])) < 1e-3
                assert np.abs(joint - drv["evb_%s_%s_joint" % (tag, pt)]).max() < 1e-3
                # the reference's loss: the mean of the per-batch losses of its model's outputs
                assert abs(tot[2 * J] / (NB * B * width) - float(drv["evb_%s_%s_loss" % (tag, pt)])) < 1e-6
            if offs.size == NB + 1:
                np.testing.assert_allclose(s[:, 2 * J] / (B * width), drv["evb_%s_losses" % tag], rtol=1e-6)


def test_refusals_return_codes():
    from p3d import _lib
    mean, std = _stats()
    pred, gt = _pairs(256, 48)
    ok = np.array([0, 100, 256])
    for precision in ("fp32", "fp64"):
        assert _segments(pred, gt, mean, std, False, 1, ok, precision=precision)[0] == 0
        bad = [
            dict(offsets=np.array([0, 200, 100, 256])),                  # descending
            dict(offsets=np.array([0])),                                 # S = 0
            dict(offsets=np.arange(1026) * 1),                           # S = 1025 (rows 0..1025 would cover 256)
            dict(offsets=ok, row0=1),                                    # row0 + N past the table
            dict(offsets=np.array([10, 100, 300]), row0=0),              # row0 before the table
            dict(offsets=ok, kinds=0),
            dict(offsets=ok, kinds=4),
        ]
        for b in bad:
            kinds = b.pop("kinds", 1)
            rc, s = _segments(pred, gt, mean, std, False, kinds, precision=precision, **b)
            assert rc != 0 and not s.any(), b
            assert _lib.lib.p3d_last_error()
        buf = torch.zeros(256 * 48 + 4, device=DEV)
        skew = buf[1:1 + 255 * 48].view(255, 48)                   # rows 4 bytes off a 16-byte boundary
        rc, _ = _segments(skew, gt, mean, std, False, 1, np.array([0, 255]), precision=precision)
        assert rc != 0 and b"aligned" in _lib.lib.p3d_last_error()
    # the library is still healthy: a good call after the refusals
    assert _segments(pred, gt, mean, std, False, 3, ok)[0] == 0
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------- end to end
ACTIONS = ["Directions", "Discussion", "Eating", "Greeting", "Phoning"]


def _test_set(p14, seed=3):
    """Camera-frame dicts with '-sh' 2D keys; action sizes uneven, one of them not a multiple of the batch (64)."""
    rng = np.random.RandomState(seed)
    out = 42 if p14 else 48
    d2, d3 = {}, {}
    sizes = [700, 321, 1024, 450, 130]
    for action, n in zip(ACTIONS, sizes):
        for subj, part in ((9, n // 2), (11, n - n // 2)):
            x, t = synth.mlp_inputs(part, out_size=out, seed=int(rng.randint(1 << 30)))
            f = "%s.54138969.h5" % action
            d2[(subj, action, f + "-sh")] = x.astype(np.float64)
            d3[(subj, action, f)] = t.astype(np.float64)
    return d2, d3


def _model(mode, p14):
    from p3d import LinearModel
    return LinearModel(1024 if mode == "bf16" else 256, 2, True, True, True, 64, 1e-3, predict_14=p14, mode=mode,
                       device=0, seed=4)


@pytest.mark.parametrize("p14", [False, True])
@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_evaluate_actions_matches_the_reference_loop(mode, p14):
    """The reference loop forwards each action on its own (batch = the action's rows) and the staged call forwards all
    rows at once.  fp32 mode: the FFMA forward of a row does not depend on the batch, so the two agree to summation
    order.  bf16: different batch sizes may take different forward kernels; each is within the bf16 contract of the
    fp32 forward (row-wise 5.6e-3 relative at width 1024, DESIGN), so two routes differ by at most twice that: 1.2e-2
    relative on the errors and losses (the means over hundreds of poses are far closer)."""
    from p3d import evaluate
    d2, d3 = _test_set(p14)
    m = _model(mode, p14)
    mean, std = _stats()
    s = evaluate.stage_actions(m, d2, d3, ACTIONS, True)
    assert s.X.is_cuda and s.n == sum(n // 64 * 64 for n in (700, 321, 1024, 450, 130))
    tol_err, tol_loss = (1e-6, 1e-5) if mode == "fp32" else (1.2e-2, 1.2e-2)
    for proc in (False, True):
        res = evaluate.evaluate_actions(None, m, s, mean, std, procrustes=proc)
        cum = 0.0
        for action in ACTIONS:
            enc, dec = m.get_all_batches(evaluate.get_action_subset(d2, action), evaluate.get_action_subset(d3, action),
                                         True, training=False)
            err, joint, _, loss = evaluate.evaluate_batches(None, m, mean, std, None, None, None, None, None, None, 0,
                                                            enc, dec, procrustes=proc)
            cum += err
            assert abs(res.errors[action] - err) <= tol_err * err, (action, res.errors[action], err)
            np.testing.assert_allclose(res.joint_errors[action], joint, rtol=tol_err, atol=1e-9)
            assert abs(res.losses[action] - loss) <= tol_loss * loss, (action, res.losses[action], loss)
        assert abs(res.average - cum / len(ACTIONS)) <= tol_err * res.average
        assert res.step_time > 0
    both = evaluate.evaluate_actions(None, m, s, mean, std, procrustes="both")
    plain = evaluate.evaluate_actions(None, m, s, mean, std, procrustes=False)
    aligned = evaluate.evaluate_actions(None, m, s, mean, std, procrustes=True)
    for a in ACTIONS:
        assert abs(both[0].errors[a] - plain.errors[a]) <= 1e-6 * plain.errors[a]
        assert abs(both[1].errors[a] - aligned.errors[a]) <= 1e-6 * aligned.errors[a]
        assert both[1].errors[a] < both[0].errors[a]
    f64 = evaluate.evaluate_actions(None, m, s, mean, std, procrustes=True, precision="fp64")
    assert all(abs(f64.errors[a] - aligned.errors[a]) < 1e-3 for a in ACTIONS)
    # drop_tail=False keeps the 321- and 130-pose actions whole
    full = evaluate.stage_actions(m, d2, d3, ACTIONS, True, drop_tail=False)
    assert full.n == 700 + 321 + 1024 + 450 + 130
    r = evaluate.evaluate_actions(None, m, full, mean, std)
    assert set(r.errors) == set(ACTIONS) and all(np.isfinite(v) for v in r.errors.values())
    m.close()


def test_one_evaluation_launch_and_one_download():
    from p3d import _lib, evaluate
    d2, d3 = _test_set(False)
    m = _model("bf16", False)
    mean, std = _stats()
    for actions in (ACTIONS, ACTIONS[:1]):
        s = evaluate.stage_actions(m, d2, d3, actions, True)
        evaluate.evaluate_actions(None, m, s, mean, std, procrustes="both")          # warm-up
        torch.cuda.synchronize()
        c0 = _lib.lib.p3d_launch_count()
        m.step(None, s.X, None, 1.0, isTraining=False)
        torch.cuda.synchronize()
        fwd = _lib.lib.p3d_launch_count() - c0
        c1 = _lib.lib.p3d_launch_count()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            evaluate.evaluate_actions(None, m, s, mean, std, procrustes="both")
            torch.cuda.synchronize()
        assert _lib.lib.p3d_launch_count() - c1 == fwd + 1, (len(actions), fwd)
        names = [e.name for e in prof.events()]
        assert sum("DtoH" in n for n in names) == 1, [n for n in names if "Memcpy" in n]
        assert sum("HtoD" in n for n in names) == 0, [n for n in names if "Memcpy" in n]
        assert any("mpjpe_f32_kernel" in n for n in names)
    m.close()


def test_evaluate_actions_argument_errors():
    from p3d import evaluate
    d2, d3 = _test_set(False)
    m = _model("fp32", False)
    mean, std = _stats()
    s = evaluate.stage_actions(m, d2, d3, ACTIONS[:2], True)
    with pytest.raises(ValueError, match="precision"):
        evaluate.evaluate_actions(None, m, s, mean, std, precision="fp16")
    with pytest.raises(ValueError, match="procrustes"):
        evaluate.evaluate_actions(None, m, s, mean, std, procrustes="yes")
    with pytest.raises(ValueError, match="96"):
        evaluate.evaluate_actions(None, m, s, mean[:48], std)
    host = evaluate.stage_actions_host(m, d2, d3, ACTIONS[:2], True)
    with pytest.raises(ValueError, match="stage_actions"):
        evaluate.evaluate_actions(None, m, host, mean, std)
    m.close()
