"""The arithmetic of the reference's `predict_3dpose.evaluate_batches` (src/predict_3dpose.py:399-442)
as one fused CUDA pass: un-normalise ground truth and prediction, keep [0,1,2] U dim_to_use_3d
(17 joints incl. the hip), optional per-pose Procrustes alignment (procrustes.py:2-63 with
compute_optimal_scale=True, re-applied as b*out.dot(T)+c), per-joint Euclidean error."""
from __future__ import annotations

import time
from dataclasses import dataclass

import numpy as np

from . import _dev, _lib
from ._lib import lib, check


def mpjpe(poses3d_n, dec_out_n, data_mean_3d, data_std_3d, procrustes=False, predict_14=False,
          return_dists=False, dist=None, precision="fp32"):
    """poses3d_n / dec_out_n: normalised prediction / ground truth [N,48|42] (NumPy or torch CUDA).
    Returns (total_err, joint_err[J]) in mm, plus dists[N,J] if return_dists.
    `dist`: a torch.distributed module/process group owner - when given, the per-joint sums and the
    pose count are all-reduced so that every rank returns the global error (SURVEY 8e).
    `precision`: "fp32" = the HBM-bound kernel (means within 1e-5 mm of the float64 reference, single
    distances within 1e-3 mm); "fp64" = all alignment arithmetic in double (distances within 1e-6 mm)."""
    if precision not in ("fp32", "fp64"):
        raise ValueError("precision must be 'fp32' or 'fp64'")
    kernel = lib.p3d_procrustes_mpjpe if precision == "fp32" else lib.p3d_procrustes_mpjpe_f64
    torch = _lib.require_cuda()
    pd, _ = _dev.to_device(poses3d_n, torch.float32)
    gd, _ = _dev.to_device(dec_out_n, torch.float32, pd.device)
    width = 42 if predict_14 else 48
    if pd.dim() != 2 or pd.shape[1] != width or pd.shape != gd.shape:
        raise ValueError("expected two [N,%d] arrays" % width)
    N = int(pd.shape[0])
    J = 14 if predict_14 else 17
    mean = _dev.host_f64(data_mean_3d); std = _dev.host_f64(data_std_3d)
    if mean.size != 96 or std.size != 96:
        raise ValueError("data_mean_3d / data_std_3d must have 96 entries")
    sums = torch.zeros(J + 1, dtype=torch.float64, device=pd.device)
    dists = torch.empty((N, J), dtype=torch.float32, device=pd.device) if return_dists else None
    with torch.cuda.device(pd.device):
        check(kernel(pd.data_ptr(), gd.data_ptr(), _lib.np_ptr(mean), _lib.np_ptr(std),
                                       int(predict_14), int(bool(procrustes)), N,
                                       dists.data_ptr() if return_dists else None, sums.data_ptr(),
                                       _lib.current_stream()))
    sums[J] = N
    if dist is not None and dist.is_initialized() and dist.get_world_size() > 1:
        red = sums if dist.get_backend() == "nccl" else sums.cpu()
        dist.all_reduce(red)
        sums = red
    s = sums.cpu().numpy()
    n_all = s[J]
    joint_err = s[:J] / n_all                   # np.mean(all_dists, axis=0)   (predict_3dpose.py:441)
    total_err = s[:J].sum() / (n_all * J)       # np.mean(all_dists)           (:442)
    if return_dists:
        return total_err, joint_err, dists
    return total_err, joint_err


def evaluate_batches(sess, model,
                     data_mean_3d, data_std_3d, dim_to_use_3d, dim_to_ignore_3d,
                     data_mean_2d, data_std_2d, dim_to_use_2d, dim_to_ignore_2d,
                     current_step, encoder_inputs, decoder_outputs, current_epoch=0, *, procrustes=False, dist=None):
    """`predict_3dpose.evaluate_batches` (src/predict_3dpose.py:352-444) with its signature: evaluates a list of
    batches (what `model.get_all_batches(..., training=False)` returns) and gives back
    (total_err, joint_err, step_time, loss).  `--procrustes` is a keyword here (the reference reads the global FLAGS,
    :413), `predict_14` is taken from the model.

    The reference walks the batches one `session.run` at a time with a Python loop per pose inside; here the batches
    are stacked once, uploaded once, lifted by one `model.step` and scored by one `mpjpe` pass - every pose is
    independent at test time (moving BatchNorm statistics, keep probability 1), so the numbers are the same.  Like
    the reference (:410-411,433) every batch must hold `model.batch_size` poses; `loss` is the mean of the per-batch
    losses, which for equal batches is the mean over all elements."""
    nbatches = len(encoder_inputs)
    if nbatches == 0 or len(decoder_outputs) != nbatches:
        raise ValueError("encoder_inputs / decoder_outputs must be equally long, non-empty lists of batches")
    for e, d in zip(encoder_inputs, decoder_outputs):
        assert e.shape[0] == model.batch_size and d.shape[0] == model.batch_size, "every batch must hold model.batch_size poses"
    torch = _lib.require_cuda()
    start_time = time.time()
    dev = torch.device("cuda", model.device)
    if hasattr(encoder_inputs[0], "is_cuda"):
        enc, dec = torch.cat(list(encoder_inputs), 0), torch.cat(list(decoder_outputs), 0)
    else:
        enc = torch.from_numpy(np.concatenate([np.asarray(e, dtype=np.float32) for e in encoder_inputs], 0)).to(dev)
        dec = torch.from_numpy(np.concatenate([np.asarray(d, dtype=np.float32) for d in decoder_outputs], 0)).to(dev)
    loss, _, poses3d = model.step(sess, enc, dec, 1.0, isTraining=False)      # dropout keep probability is 1 at test time
    total_err, joint_err = mpjpe(poses3d, dec, data_mean_3d, data_std_3d, procrustes=procrustes,
                                 predict_14=model.predict_14, dist=dist)
    loss = float(loss)
    step_time = (time.time() - start_time) / nbatches
    return total_err, joint_err, step_time, loss


# ---------------------------------------------------------------------------------------------- action-wise evaluation
# The --evaluateActionWise loop that upstream 3d-pose-baseline's train() runs after every epoch, restated:
#     for action in actions:
#         action_test_set_2d = get_action_subset(test_set_2d, action)
#         action_test_set_3d = get_action_subset(test_set_3d, action)
#         encoder_inputs, decoder_outputs = model.get_all_batches(action_test_set_2d, action_test_set_3d,
#                                                                 camera_frame, training=False)
#         act_err, _, step_time, loss = evaluate_batches(...)
#         cum_err = cum_err + act_err
#     model.err_mm_summary(cum_err / float(len(actions)))          # unweighted mean over actions
# Here the test set is staged on the device once per run (stage_actions) and every epoch scores all actions with one
# forward and one segmented evaluation launch (evaluate_actions).

MAX_SEGMENTS = 1024       # p3d_mpjpe_segments: the offsets travel in the kernel's parameters


def get_action_subset(poses_set, action):
    """The reference helper: the entries of `poses_set` whose key (subject, action, name) has this action, in order."""
    return {k: v for k, v in poses_set.items() if k[1] == action}


@dataclass
class ActionSet:
    """A test set staged for evaluate_actions: the rows of every action, concatenated in `actions` order.
    X [n,32] / T [n,out] are fp32 (torch CUDA after stage_actions, NumPy after stage_actions_host); action a holds rows
    offsets[a]:offsets[a+1]; batches[a] is the number of model.batch_size batches the reference loop evaluates."""
    actions: list
    offsets: np.ndarray
    batches: list
    batch_size: int
    X: object
    T: object

    @property
    def n(self):
        return int(self.offsets[-1])


def stage_actions_host(model, test_set_2d, test_set_3d, actions, camera_frame, *, drop_tail=True):
    """The host half of stage_actions (no device needed): for each action, model.get_all_batches(subset_2d, subset_3d,
    camera_frame, training=False) exactly as the reference loop calls it (its 2D -> 3D key mapping and its drop of the
    n % batch_size tail), concatenated and cast to fp32 once.  drop_tail=False keeps every pose of every action."""
    actions = list(actions)
    if not actions or len(actions) > MAX_SEGMENTS:
        raise ValueError("actions must name 1..%d actions" % MAX_SEGMENTS)
    if len(set(actions)) != len(actions):
        raise ValueError("actions must not repeat")
    B = int(model.batch_size)
    xs, ts, counts, batches = [], [], [], []
    for action in actions:
        sub2d, sub3d = get_action_subset(test_set_2d, action), get_action_subset(test_set_3d, action)
        if not sub2d:
            raise ValueError("action %r has no entry in the test set" % (action,))
        n = sum(int(v.shape[0]) for v in sub2d.values())
        if drop_tail:
            if n < B:     # get_all_batches cannot split it, and evaluate_batches refuses an empty list
                raise ValueError("action %r has %d poses, fewer than batch_size %d" % (action, n, B))
            enc, dec = model.get_all_batches(sub2d, sub3d, camera_frame, training=False)
            x, t = np.concatenate(enc, 0), np.concatenate(dec, 0)
            batches.append(len(enc))
        else:
            x, t = model.stack_pairs(sub2d, sub3d, camera_frame)
            batches.append(-(-n // B))
        xs.append(x.astype(np.float32))
        ts.append(t.astype(np.float32))
        counts.append(x.shape[0])
    offsets = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    return ActionSet(actions, offsets, batches, B, np.ascontiguousarray(np.concatenate(xs, 0)),
                     np.ascontiguousarray(np.concatenate(ts, 0)))


def stage_actions(model, test_set_2d, test_set_3d, actions, camera_frame, *, drop_tail=True):
    """Stage the per-action test set once per training run: stage_actions_host, then one upload of X and T to the
    model's device.  Raises ValueError for an action without entries and, with drop_tail, for an action with fewer
    than batch_size poses (the reference loop cannot evaluate it)."""
    torch = _lib.require_cuda()
    s = stage_actions_host(model, test_set_2d, test_set_3d, actions, camera_frame, drop_tail=drop_tail)
    dev = torch.device("cuda", model.device)
    s.X, s.T = torch.from_numpy(s.X).to(dev), torch.from_numpy(s.T).to(dev)
    return s


@dataclass
class ActionErrors:
    """evaluate_actions' result: per action the MPJPE in mm (the reference's act_err), the per-joint errors, the
    evaluation loss (evaluate_batches' mean of the per-batch losses); `average` is the unweighted mean of the action
    errors (what the reference logs as err_mm); `step_time` the call's wall time per batch, as evaluate_batches."""
    errors: dict
    joint_errors: dict
    losses: dict
    average: float
    step_time: float


def _dp_agree(dist, device, values, names, err, what):
    """Before a data-parallel call launches anything: raise ValueError on EVERY rank when any rank rejected its
    arguments (`err`) or the ranks disagree on `values` - one all_reduce(MAX) over (v, -v) gives the maximum and the
    minimum (the pattern of LinearModel._dp_epoch_agree)."""
    import torch
    v = [float(a) for a in values] + [1.0 if err else 0.0]
    dev = torch.device("cuda", device) if dist.get_backend() == "nccl" else "cpu"
    t = torch.tensor(v + [-a for a in v], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    k = len(v)
    hi, lo = t[:k].tolist(), [-a for a in t[k:].tolist()]
    if err:
        raise ValueError(err)
    if hi[-1] > 0:
        raise ValueError("%s: another rank rejected its arguments" % what)
    if hi != lo:
        diff = ", ".join("%s %.10g..%.10g" % (nm, a, b) for nm, a, b in zip(names, lo, hi) if a != b)
        raise ValueError("%s: the ranks disagree on %s; every rank must stage the same set" % (what, diff))


def _offsets_checksum(offsets):
    """Position-weighted sum of the offsets, exact in float64 for any set that fits in memory."""
    o = np.asarray(offsets, dtype=np.int64)
    return float(int(np.dot(o % (1 << 20), np.arange(1, o.size + 1, dtype=np.int64))) % (1 << 52))


def evaluate_actions(sess, model, action_set, data_mean_3d, data_std_3d, current_step=None, *, procrustes=False,
                     precision="fp32", dist=None):
    """Every action of a staged set (stage_actions) evaluated on the model's current variables with one forward
    (model.step(None, X, None, 1.0, isTraining=False)), one p3d_mpjpe_segments launch and one download.
    Returns ActionErrors; procrustes="both" returns (plain, aligned) from the same pass.  `precision` as in mpjpe.
    `sess` and `current_step` are accepted for the reference's call shape and unused.

    Data parallel (`dist` initialised with world > 1): every rank stages the same set; each scores its row block
    shard_rows(n, rank, world) and one all_reduce of the sums gives every rank the same result.  Ranks that disagree on
    the set, or a rank that rejects its arguments, raise ValueError on every rank before anything launches."""
    from .linear_model import shard_rows
    torch = _lib.require_cuda()
    start_time = time.time()
    s = action_set
    S, n = len(s.actions), s.n
    J = 14 if model.predict_14 else 17
    width = 42 if model.predict_14 else 48
    mean, std = _dev.host_f64(data_mean_3d), _dev.host_f64(data_std_3d)
    err = None
    if precision not in ("fp32", "fp64"):
        err = "precision must be 'fp32' or 'fp64'"
    elif procrustes not in (False, True, "both"):
        err = "procrustes must be False, True or 'both'"
    elif mean.size != 96 or std.size != 96:
        err = "data_mean_3d / data_std_3d must have 96 entries"
    elif not (hasattr(s.X, "is_cuda") and s.X.is_cuda) or tuple(s.X.shape) != (n, model.input_size) \
            or tuple(s.T.shape) != (n, width):
        err = "action_set must come from stage_actions for a model with %d outputs" % width
    elif s.batch_size != model.batch_size:
        err = "action_set was staged for batch_size %d, the model has %d" % (s.batch_size, model.batch_size)
    rank, world = 0, 1
    if dist is not None and dist.is_initialized() and dist.get_world_size() > 1:
        rank, world = dist.get_rank(), dist.get_world_size()
        _dp_agree(dist, model.device, [n, S, s.batch_size, _offsets_checksum(s.offsets)],
                  ("n", "actions", "batch_size", "offsets checksum"), err, "evaluate_actions")
    elif err:
        raise ValueError(err)
    kinds = {False: 1, True: 2, "both": 3}[procrustes]
    kernel = lib.p3d_mpjpe_segments if precision == "fp32" else lib.p3d_mpjpe_segments_f64
    lo, hi = shard_rows(n, rank, world)
    dev = torch.device("cuda", model.device)
    with torch.cuda.device(dev):
        sums = torch.zeros((S, 2 * J + 1), dtype=torch.float64, device=dev)
        if hi > lo:
            X, T = s.X[lo:hi], s.T[lo:hi]
            if T.data_ptr() % 16:      # a 42-wide row block starting at an odd row
                T = T.clone()
            _, _, y = model.step(None, X, None, 1.0, isTraining=False)      # dropout keep probability 1 at test time
            offs = np.ascontiguousarray(s.offsets, dtype=np.int64)
            check(kernel(y.data_ptr(), T.data_ptr(), _lib.np_ptr(mean), _lib.np_ptr(std), int(model.predict_14), kinds,
                         hi - lo, lo, _lib.np_ptr(offs), S, sums.data_ptr(), _lib.current_stream()))
        if world > 1:
            red = sums if dist.get_backend() == "nccl" else sums.cpu()
            dist.all_reduce(red)
            sums = red
        tab = sums.cpu().numpy()
    counts = np.diff(s.offsets).astype(np.float64)
    step_time = (time.time() - start_time) / max(1, sum(s.batches))

    def result(first):
        errors, joints, losses = {}, {}, {}
        for a, action in enumerate(s.actions):
            js = tab[a, first:first + J]
            joints[action] = js / counts[a]                                  # np.mean(all_dists, axis=0)
            errors[action] = float(js.sum() / (counts[a] * J))              # np.mean(all_dists)
            losses[action] = float(tab[a, 2 * J] / (counts[a] * width))      # mean over the action's equal batches
        return ActionErrors(errors, joints, losses, float(np.mean([errors[a] for a in s.actions])), step_time)

    if kinds == 3:
        return result(0), result(J)
    return result(0 if kinds == 1 else J)
