"""read_openpose_json(all_people=True): every person of an OpenPose frame through the reference's list handling
(src/openpose_3dpose_sandbox_realtime.py:67-135), ready for RealtimeLifter.step_people."""
import json

import numpy as np

from oracle import realtime_ref as R


def _person(n, seed):
    return np.random.RandomState(seed).uniform(10, 900, size=n).round(3).tolist()


def test_all_people(tmp_path):
    from p3d.realtime import read_openpose_json
    people = [_person(54, 1), _person(75, 2), _person(36, 3)]      # COCO with scores, BODY_25 with scores, tf-pose x,y
    path = tmp_path / "clip_000000000042_keypoints.json"
    path.write_text(json.dumps({"version": 1.2, "people": [{"pose_keypoints_2d": p} for p in people]}))
    xys, frame = read_openpose_json(str(path), all_people=True)
    assert frame == 42 and len(xys) == 3
    for xy, p in zip(xys, people):
        assert xy == R.keypoints_to_xy(p)
        assert len(xy) >= 36
    # the default call still returns the first person only
    xy0, frame0 = read_openpose_json(str(path))
    assert xy0 == R.keypoints_to_xy(people[0]) and frame0 == 42


def test_frame_with_nobody(tmp_path):
    from p3d.realtime import read_openpose_json
    path = tmp_path / "empty_7.json"
    path.write_text(json.dumps({"version": 1.2, "people": []}))
    assert read_openpose_json(str(path), all_people=True) == ([], 7)
