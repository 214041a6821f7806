"""Parity of the camera-frame preprocessing kernels with golden vectors from the reference's NumPy code
(tests/golden/geometry.npz) and with the oracle at larger sizes.  fp64 kernels: 1e-9 relative;
fused fp32 kernel: 1e-4 in normalised units (fp32 arithmetic on ~1000 px / ~5000 mm coordinates)."""
import os

import numpy as np
import pytest
import torch

from oracle import geometry_ref as G
from oracle import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def geo(golden_dir):
    return np.load(os.path.join(golden_dir, "geometry.npz"))


def cams_of(geo):
    return [tuple(geo[f"cam{i}_{n}"] for n in "RTfckp") for i in range(4)]


def test_project_point_radial_golden(geo):
    from p3d import cameras
    P = geo["world"].reshape(-1, 3)[: len(geo["cam0_proj"])]      # the per-point arrays hold the first 48 poses
    for i, cam in enumerate(cams_of(geo)):
        proj, D, radial, tan, r2 = cameras.project_point_radial(P, *cam)
        assert proj.shape == (P.shape[0], 2) and proj.dtype == np.float64
        np.testing.assert_allclose(proj, geo[f"cam{i}_proj"], rtol=1e-11, atol=1e-8)
        np.testing.assert_allclose(D, geo[f"cam{i}_D"], rtol=1e-12)
        np.testing.assert_allclose(radial, geo[f"cam{i}_radial"], rtol=1e-12)
        np.testing.assert_allclose(tan, geo[f"cam{i}_tan"], rtol=1e-11, atol=1e-14)
        np.testing.assert_allclose(r2, geo[f"cam{i}_r2"], rtol=1e-12)
    with pytest.raises(AssertionError):
        cameras.project_point_radial(np.zeros((4, 2)), *cams_of(geo)[0])


def test_world_camera_roundtrip_golden(geo):
    from p3d import cameras
    P = geo["world"].reshape(-1, 3)[: len(geo["cam0_w2c"])]
    for i, cam in enumerate(cams_of(geo)):
        w2c = cameras.world_to_camera_frame(P, cam[0], cam[1])
        np.testing.assert_allclose(w2c, geo[f"cam{i}_w2c"], rtol=1e-12, atol=1e-8)
        c2w = cameras.camera_to_world_frame(w2c, cam[0], cam[1])
        np.testing.assert_allclose(c2w, geo[f"cam{i}_c2w"], rtol=1e-12, atol=1e-8)
        np.testing.assert_allclose(c2w, P, atol=1e-8)


def test_dictionary_drivers_batch_sequences_per_subject(geo):
    """project_to_cameras / transform_world_to_camera send all sequences of a subject to the device in one buffer and
    run each camera once: keys, shapes and values must equal the per-sequence, per-camera calls of the reference loop
    (data_utils.py:243-255, 349-362) - ragged sequence lengths, two subjects with different cameras."""
    from p3d import cameras, data_utils
    cams = cams_of(geo)
    rcams = {(s, ci + 1): cams[(ci + s) % 4] + (f"c{s}{ci}",) for s in (1, 5) for ci in range(4)}
    w = geo["world"]
    poses = {(1, "Walking", "Walking 1.h5"): w[:7].copy(), (1, "Eating", "Eating.h5"): w[7:20].copy(),
             (5, "Sitting", "Sitting 2.h5"): w[20:21].copy()}
    t2d = data_utils.project_to_cameras(poses, rcams, ncams=4)
    t3d = data_utils.transform_world_to_camera(poses, rcams, ncams=4)
    assert len(t2d) == 12 and len(t3d) == 12
    for (subj, a, seq), arr in poses.items():
        for ci in range(4):
            R, T, f, c, k, p_, name = rcams[(subj, ci + 1)]
            key = (subj, a, seq[:-3] + "." + name + ".h5")
            ref2 = cameras.project_point_radial(arr.reshape(-1, 3), R, T, f, c, k, p_)[0].reshape(-1, 64)
            ref3 = cameras.world_to_camera_frame(arr.reshape(-1, 3), R, T).reshape(-1, 96)
            assert t2d[key].shape == ref2.shape and t3d[key].shape == ref3.shape
            assert np.array_equal(t2d[key], ref2) and np.array_equal(t3d[key], ref3)


def test_dictionary_pipeline_golden(geo):
    """train()'s preprocessing calls (predict_3dpose.py:197-207) through the mirrored data_utils API."""
    from p3d import data_utils
    cams = cams_of(geo)
    rcams = {(1, ci + 1): cams[ci] + (f"cam{ci}",) for ci in range(4)}
    poses = {(1, "Walking", "Walking 1.h5"): geo["world"].copy()}
    t2d = data_utils.project_to_cameras(poses, rcams, ncams=4)
    t3d = data_utils.transform_world_to_camera(poses, rcams, ncams=4)
    assert sorted("|".join(map(str, k)) for k in t2d) == sorted(geo["keys2d"].tolist())
    t3d, roots = data_utils.postprocess_3d(t3d)
    keys = sorted(t2d.keys())
    np.testing.assert_allclose(np.stack([roots[k] for k in keys]), geo["roots"], rtol=1e-12, atol=1e-8)
    all2d = np.vstack([t2d[k] for k in keys]); all3d = np.vstack([t3d[k] for k in keys])
    m2, s2, ig2, use2 = data_utils.normalization_stats(all2d, dim=2)
    m3, s3, ig3, use3 = data_utils.normalization_stats(all3d, dim=3)
    np.testing.assert_allclose(m2, geo["mean2d"], rtol=1e-11, atol=1e-9)
    np.testing.assert_allclose(s2, geo["std2d"], rtol=1e-11, atol=1e-9)
    np.testing.assert_allclose(m3, geo["mean3d"], rtol=1e-10, atol=1e-8)
    np.testing.assert_allclose(s3, geo["std3d"], rtol=1e-11, atol=1e-9)
    assert np.array_equal(use2, geo["use2d"]) and np.array_equal(ig3, geo["ignore3d"])
    n2 = data_utils.normalize_data(t2d, geo["mean2d"], geo["std2d"], use2)
    n3 = data_utils.normalize_data(t3d, geo["mean3d"], geo["std3d"], use3)
    np.testing.assert_allclose(np.stack([n2[k] for k in keys]), geo["x2d_norm"], rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(np.stack([n3[k] for k in keys]), geo["y3d_norm"], rtol=1e-9, atol=1e-9)
    assert t2d[keys[0]].shape[1] == 32            # the input dict was mutated like the reference (:275)
    u2 = data_utils.unNormalizeData(geo["x2d_norm"][1], geo["mean2d"], geo["std2d"], geo["ignore2d"])
    u3 = data_utils.unNormalizeData(geo["y3d_norm"][1], geo["mean3d"], geo["std3d"], geo["ignore3d"])
    np.testing.assert_allclose(u2, geo["un2d"], rtol=1e-14, atol=1e-11)
    np.testing.assert_allclose(u3, geo["un3d"], rtol=1e-14, atol=1e-11)
    with pytest.raises(ValueError):
        data_utils.normalize_data({"k": all2d}, geo["mean2d"], geo["std2d"], np.arange(10))


def test_fused_project_normalize_golden_and_ragged(geo):
    from p3d import data_utils
    cams = cams_of(geo)
    world = geo["world"]
    x2d, y3d = data_utils.camera_frame_dataset(world.astype(np.float32), cams, geo["mean2d"], geo["std2d"],
                                               geo["mean3d"], geo["std3d"])
    assert x2d.shape == (4, 64, 32) and y3d.shape == (4, 64, 48) and x2d.dtype == np.float32
    np.testing.assert_allclose(x2d, geo["x2d_norm"], atol=1e-4)
    np.testing.assert_allclose(y3d, geo["y3d_norm"], atol=1e-4)
    for n in (1, 15, 16, 17, 37):                  # ragged tiles (16 poses per block)
        x2, y3 = data_utils.camera_frame_dataset(world[:n].astype(np.float32), cams[:3], geo["mean2d"], geo["std2d"],
                                                 geo["mean3d"], geo["std3d"])
        np.testing.assert_allclose(x2, geo["x2d_norm"][:3, :n], atol=1e-4)
        np.testing.assert_allclose(y3, geo["y3d_norm"][:3, :n], atol=1e-4)
    x2, none = data_utils.camera_frame_dataset(world.astype(np.float32), cams, geo["mean2d"], geo["std2d"], want_3d=False)
    assert none is None and np.array_equal(x2, x2d)


def test_fused_predict_14_and_large_against_oracle():
    from p3d import data_utils
    N = 50001
    cams = synth.cameras(4, seed=11)
    world = synth.world_poses(N, seed=12).astype(np.float32)
    w64 = world.astype(np.float64)
    all2d = np.vstack([G.project_point_radial(w64.reshape(-1, 3), *c)[0].reshape(-1, 64) for c in cams])
    m2, s2, _, use2 = G.normalization_stats(all2d, 2)
    all3d = np.vstack([G.postprocess_3d(G.world_to_camera(w64.reshape(-1, 3), c[0], c[1]).reshape(-1, 96))[0] for c in cams])
    for p14 in (False, True):
        m3, s3, _, use3 = G.normalization_stats(all3d, 3, p14)
        s3 = np.where(s3 == 0, 1.0, s3)           # hip columns are all-zero after root-centring
        ref2 = G.project_normalize(w64, cams, m2, s2, use2)
        ref3 = G.camera_frame_normalize(w64, cams, m3, s3, use3)
        wd = torch.from_numpy(world).cuda()
        x2d, y3d = data_utils.camera_frame_dataset(wd, cams, m2, s2, m3, s3, predict_14=p14)
        assert x2d.is_cuda and y3d.shape == (4, N, 42 if p14 else 48)
        np.testing.assert_allclose(x2d.cpu().numpy(), ref2, atol=2e-4)
        np.testing.assert_allclose(y3d.cpu().numpy(), ref3, atol=2e-4)


def test_normalise_unnormalise_roundtrip_property():
    """normalise o unnormalise = id on the used dims, up to the reference's fp32 truncation (1.3e-7)."""
    from p3d import data_utils
    rng = np.random.RandomState(0)
    data = rng.normal(0, 200, (1000, 96))
    mean = data.mean(0); std = data.std(0)
    use, ign = G.dims_to_use(3)
    n = data_utils.normalize_data({"a": data.copy()}, mean, std, use)["a"]
    back = data_utils.unNormalizeData(n, mean, std, ign)
    np.testing.assert_allclose(back[:, use], data[:, use], rtol=1e-6, atol=1e-4)
    assert np.array_equal(back[:, ign], np.tile(mean[ign], (1000, 1)))
