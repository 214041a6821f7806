"""The per-action evaluation loop of upstream 3d-pose-baseline's train() (--evaluateActionWise), restated in NumPy.
Restated, not executed: the reference source is not in this tree, and oracle/make_golden_driver.py pins only the two
pieces the loop calls, get_all_batches and evaluate_batches.  The loop, per epoch:
    for action in actions:
        enc, dec = model.get_all_batches(get_action_subset(test_set_2d, action), get_action_subset(test_set_3d, action),
                                         camera_frame, training=False)
        act_err, _, _, loss = evaluate_batches(..., enc, dec)
        cum_err += act_err
    err_mm = cum_err / len(actions)
Given the concatenated rows of every action (offsets[a]:offsets[a+1] hold action a), this returns what that loop
computes, from one batched MPJPE over all rows."""
from __future__ import annotations

import numpy as np

from oracle import geometry_ref as G


def evaluate_actions(pred_n, gt_n, offsets, mean3d, std3d, ignore3d, use3d, procrustes=False, predict_14=False):
    """-> (errors[S], joint_errors[S,J], losses[S], err_mm): per action np.mean(dists), np.mean(dists, axis=0), the mean
    squared error of the normalised rows (the mean of equal per-batch losses), and the unweighted mean over actions."""
    d = G.mpjpe(pred_n, gt_n, mean3d, std3d, ignore3d, use3d, procrustes=procrustes, predict_14=predict_14)
    sq = ((np.asarray(pred_n, np.float64) - np.asarray(gt_n, np.float64)) ** 2).mean(axis=1)
    o = np.asarray(offsets)
    errors = np.array([d[o[a]:o[a + 1]].mean() for a in range(o.size - 1)])
    joints = np.stack([d[o[a]:o[a + 1]].mean(axis=0) for a in range(o.size - 1)])
    losses = np.array([sq[o[a]:o[a + 1]].mean() for a in range(o.size - 1)])
    return errors, joints, losses, float(errors.mean())
