"""Realtime front-end around the lifter: the frame loop of the reference's
`openpose_3dpose_sandbox_realtime.py` (src/openpose_3dpose_sandbox_realtime.py:67-195) without TensorFlow.

    lifter = RealtimeLifter(model, data_mean_2d, data_std_2d, dim_to_use_2d,
                            data_mean_3d, data_std_3d, dim_to_use_3d)
    xy = keypoints_to_xy(json.load(f)["people"][0]["pose_keypoints_2d"])      # :69-135 (list handling)
    enc_in, poses3d_norm, poses3d = lifter.step(xy)                            # :137-171 (one CUDA launch)

    xys, frame = read_openpose_json(path, all_people=True)                     # every person of the frame
    enc_in, poses3d_norm, poses3d = lifter.step_people(xys)                    # [P,32], [P,out], [P,96]

`step` runs keypoint re-ordering, hip/neck/thorax synthesis, normalisation, the six-layer lifter and
unNormalizeData in a single 16-CTA cluster kernel that reads from and writes to mapped pinned memory
(p3d_realtime_step_host).  `step_people` lifts up to 8 people of one frame in that same single launch, each person
bit-identical to its own `step` (p3d_realtime_step_people_host; more people, or a model the cluster kernel does not
serve, take one staged batched step).  `step_batch` does the same for many frames on device buffers.
JSON parsing / list surgery stays on the host exactly as in the reference; plotting is out of scope -
`display_transform` is the coordinate shuffle the reference applies right before viz.show3Dpose (:178-195).
"""
from __future__ import annotations

import ctypes as C
import json
import re

import numpy as np

from . import _lib
from ._lib import lib, check

# OpenPose/COCO keypoint i goes to H3.6M joint ORDER[i] (openpose_3dpose_sandbox_realtime.py:20)
ORDER = [15, 12, 25, 26, 27, 17, 18, 19, 1, 2, 3, 6, 7, 8]


def keypoints_to_xy(pose_keypoints_2d):
    """The list handling of openpose_3dpose_sandbox_realtime.py:69-135: strip the confidence scores of an OpenPose
    record (len >= 53, :71-76; tf-pose-estimation lists are already x,y pairs, :77-79), and for lists of more than 54
    coordinates drop BODY_25's joint 8 (MidHip) so that joints 9..18 become COCO's 8..17 (:86-135).
    Returns the coordinate list the frame loop indexes (at least 36 values)."""
    _data = list(pose_keypoints_2d)
    if len(_data) >= 53:
        xy = []
        for o in range(0, len(_data), 3):
            xy.append(_data[o])
            xy.append(_data[o + 1])
    else:
        xy = _data
    if len(xy) > 54:
        # net effect of the reference's del/overwrite loop (:88-133): joints 0..7 kept, joint 8 removed, 9..18 shifted down
        xy = list(xy[0:16]) + list(xy[18:38])
    return xy


def read_openpose_json(path, all_people=False):
    """First person of an OpenPose JSON file (:67-69) -> (xy list, frame number from the file name :81-82).
    all_people=True: ([xy list of every person], frame number); [] for a frame with nobody in it."""
    with open(path) as f:
        data = json.load(f)
    idx = re.findall(r"(\d+)", path)
    frame = int(idx[-1]) if idx else 0
    if all_people:
        return [keypoints_to_xy(p["pose_keypoints_2d"]) for p in data["people"]], frame
    return keypoints_to_xy(data["people"][0]["pose_keypoints_2d"]), frame


def display_transform(poses3d, spine_x, spine_y):
    """The in-place coordinate shuffle before plotting (:178-195): swap y/z, flip the new z inside its own range, shift
    by the 2D spine position.  NumPy (it is plotting glue, 96 numbers per frame); returns a new [n,96] array."""
    p = np.array(poses3d, dtype=np.float64, copy=True).reshape(-1, 32, 3)
    p[:, :, [1, 2]] = p[:, :, [2, 1]]
    zmax = max(float(p[:, :, 2].max()), 0.0)          # _max starts at 0 (:178)
    zmin = min(float(p[:, :, 2].min()), 10000.0)      # _min starts at 10000 (:179)
    p[:, :, 2] = zmax - p[:, :, 2] + zmin
    p[:, :, 0] += (spine_x - 630)
    p[:, :, 2] += (500 - spine_y)
    return p.reshape(-1, 96)


class RealtimeLifter(object):
    """Owns the device tables and the mapped host block of one realtime session (p3d_realtime_*)."""

    MAX_PEOPLE = 8          # people of one frame step_people lifts in one launch (p3d_realtime_step_people_host)

    def __init__(self, model, data_mean_2d, data_std_2d, dim_to_use_2d, data_mean_3d, data_std_3d, dim_to_use_3d):
        self.model = model
        mu2 = np.ascontiguousarray(data_mean_2d, dtype=np.float64).reshape(-1)
        sd2 = np.ascontiguousarray(data_std_2d, dtype=np.float64).reshape(-1)
        mu3 = np.ascontiguousarray(data_mean_3d, dtype=np.float64).reshape(-1)
        sd3 = np.ascontiguousarray(data_std_3d, dtype=np.float64).reshape(-1)
        u2 = np.ascontiguousarray(dim_to_use_2d, dtype=np.int32).reshape(-1)
        u3 = np.ascontiguousarray(dim_to_use_3d, dtype=np.int32).reshape(-1)
        if mu2.size != 64 or sd2.size != 64 or u2.size != 32:
            raise ValueError("2D statistics must be [64] with 32 used dimensions")
        if mu3.size != 96 or sd3.size != 96 or u3.size != model.output_size:
            raise ValueError("3D statistics must be [96] with %d used dimensions" % model.output_size)
        self.output_size = int(model.output_size)
        h = C.c_void_p()
        check(lib.p3d_realtime_create(model._handle, _lib.np_ptr(mu2), _lib.np_ptr(sd2), _lib.np_ptr(u2),
                                      _lib.np_ptr(mu3), _lib.np_ptr(sd3), _lib.np_ptr(u3), C.byref(h)))
        self._handle = h
        # per-frame buffers and their addresses are made once: the frame call itself is ~50 us, ctypes argument
        # conversion of four fresh arrays was a fifth of that
        self._kp = np.zeros(36, dtype=np.float64)
        self._enc = np.empty((1, 32), dtype=np.float32)
        self._y = np.empty((1, self.output_size), dtype=np.float32)
        self._pose = np.empty((1, 96), dtype=np.float64)
        self._args = (self._handle, C.c_void_p(self._kp.ctypes.data), C.c_void_p(self._enc.ctypes.data),
                      C.c_void_p(self._y.ctypes.data), C.c_void_p(self._pose.ctypes.data))
        # the same for the up to MAX_PEOPLE people of one frame that step_people serves in one launch
        self._kps = np.zeros((self.MAX_PEOPLE, 36), dtype=np.float64)
        self._encs = np.empty((self.MAX_PEOPLE, 32), dtype=np.float32)
        self._ys = np.empty((self.MAX_PEOPLE, self.output_size), dtype=np.float32)
        self._poses = np.empty((self.MAX_PEOPLE, 96), dtype=np.float64)
        self._people_ptrs = tuple(C.c_void_p(a.ctypes.data) for a in (self._kps, self._encs, self._ys, self._poses))

    def step(self, xy):
        """One frame: xy = at least 36 coordinates (x0,y0,x1,y1,...; :137-142 use the first 36).
        Returns (enc_in [1,32] fp32, poses3d_normalised [1,out] fp32, poses3d [1,96] fp64) - the reference's
        enc_in after :163, the model output of :168 and its unNormalizeData of :171."""
        if len(xy) < 36:
            raise IndexError("need at least 36 keypoint coordinates, got %d" % len(xy))   # the reference's xy[o] raises too
        if self._handle is None:
            raise RuntimeError("RealtimeLifter is closed")
        self._kp[:] = xy[:36]
        check(lib.p3d_realtime_step_host(*self._args))
        return self._enc.copy(), self._y.copy(), self._pose.copy()      # fresh arrays, like the reference returns

    def step_people(self, xys):
        """Every person of one frame: xys = P coordinate lists (or a [P, >=36] array), the first 36 values of each used
        as in `step`.  Returns fresh (enc_in [P,32] fp32, poses3d_normalised [P,out] fp32, poses3d [P,96] fp64); row p
        equals `step(xys[p])` bit for bit when P <= 8 and the model runs `step` as one launch (width 1024, bf16 or fp16).
        Otherwise the people run as one staged batch and equal `step_batch` of the same keypoints."""
        P = len(xys)
        for xy in xys:
            if len(xy) < 36:
                raise IndexError("need at least 36 keypoint coordinates, got %d" % len(xy))
        if self._handle is None:
            raise RuntimeError("RealtimeLifter is closed")
        if P == 0:
            return (np.empty((0, 32), np.float32), np.empty((0, self.output_size), np.float32),
                    np.empty((0, 96), np.float64))
        if P <= self.MAX_PEOPLE:
            kp, enc, y, pose = self._kps, self._encs, self._ys, self._poses
            ptrs = self._people_ptrs
        else:
            kp = np.empty((P, 36), np.float64)
            enc = np.empty((P, 32), np.float32)
            y = np.empty((P, self.output_size), np.float32)
            pose = np.empty((P, 96), np.float64)
            ptrs = tuple(C.c_void_p(a.ctypes.data) for a in (kp, enc, y, pose))
        for i, xy in enumerate(xys):
            kp[i] = xy[:36]
        check(lib.p3d_realtime_step_people_host(self._handle, ptrs[0], P, ptrs[1], ptrs[2], ptrs[3]))
        return enc[:P].copy(), y[:P].copy(), pose[:P].copy()

    def step_batch(self, xy):
        """Many frames at once: xy [B,36] (NumPy or torch CUDA fp64) -> (enc_in [B,32], y [B,out], poses3d [B,96])."""
        torch = _lib.require_cuda()
        is_torch = hasattr(xy, "is_cuda")
        dev = torch.device("cuda", self.model.device)
        k = (xy if is_torch else torch.from_numpy(np.ascontiguousarray(xy, dtype=np.float64))).to(dev, torch.float64).contiguous()
        if k.dim() != 2 or k.shape[1] != 36:
            raise ValueError("xy must be [B,36]")
        B = int(k.shape[0])
        with torch.cuda.device(dev):
            enc = torch.empty((B, 32), dtype=torch.float32, device=dev)
            y = torch.empty((B, self.output_size), dtype=torch.float32, device=dev)
            pose = torch.empty((B, 96), dtype=torch.float64, device=dev)
            check(lib.p3d_realtime_step(self._handle, k.data_ptr(), enc.data_ptr(), y.data_ptr(), pose.data_ptr(), B,
                                        _lib.current_stream()))
        if is_torch:
            return enc, y, pose
        return enc.cpu().numpy(), y.cpu().numpy(), pose.cpu().numpy()

    def close(self):
        if self._handle is not None:
            lib.p3d_realtime_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
