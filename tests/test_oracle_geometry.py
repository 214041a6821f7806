"""The CPU oracle (oracle/geometry_ref.py) against golden vectors produced by the reference's
own NumPy code (oracle/make_golden.py).  This is what pins the oracle."""
import os

import numpy as np
import pytest

from oracle import geometry_ref as G


@pytest.fixture(scope="module")
def geo(golden_dir):
    return np.load(os.path.join(golden_dir, "geometry.npz"))


@pytest.fixture(scope="module")
def proc(golden_dir):
    return np.load(os.path.join(golden_dir, "procrustes.npz"))


def cams_of(geo):
    return [tuple(geo[f"cam{i}_{n}"] for n in "RTfckp") for i in range(4)]


def test_index_tables(golden_dir):
    t = np.load(os.path.join(golden_dir, "tables.npz"))
    for dim, p14, u, i in [(2, False, "use2d", "ignore2d"), (3, False, "use3d", "ignore3d"),
                           (3, True, "use3d_14", "ignore3d_14")]:
        use, ign = G.dims_to_use(dim, p14)
        assert np.array_equal(use, t[u]) and np.array_equal(ign, t[i])
    assert len(G.dims_to_use(2)[0]) == 32 and len(G.dims_to_use(3)[0]) == 48
    assert len(G.dims_to_use(3, True)[0]) == 42
    # the reference's only known-answer assert (data_utils.py:135-136)
    assert t["sh_to_gt_perm"].tolist() == [6, 2, 1, 0, 3, 4, 5, 7, 8, 9, 13, 14, 15, 12, 11, 10]


def test_project_point_radial(geo):
    P = geo["world"].reshape(-1, 3)[: len(geo["cam0_proj"])]      # the per-point arrays hold the first 48 poses
    for i, cam in enumerate(cams_of(geo)):
        proj, D, radial, tan, r2 = G.project_point_radial(P, *cam)
        np.testing.assert_allclose(proj, geo[f"cam{i}_proj"], rtol=1e-12, atol=1e-9)
        np.testing.assert_allclose(D, geo[f"cam{i}_D"], rtol=1e-13)
        np.testing.assert_allclose(radial, geo[f"cam{i}_radial"], rtol=1e-13)
        np.testing.assert_allclose(tan, geo[f"cam{i}_tan"], rtol=1e-12, atol=1e-15)
        np.testing.assert_allclose(r2, geo[f"cam{i}_r2"], rtol=1e-13)
        assert (D > 0).all()


def test_world_camera_roundtrip(geo):
    P = geo["world"].reshape(-1, 3)[: len(geo["cam0_w2c"])]
    for i, cam in enumerate(cams_of(geo)):
        w2c = G.world_to_camera(P, cam[0], cam[1])
        np.testing.assert_allclose(w2c, geo[f"cam{i}_w2c"], rtol=1e-13, atol=1e-9)
        np.testing.assert_allclose(G.camera_to_world(w2c, cam[0], cam[1]), geo[f"cam{i}_c2w"],
                                   rtol=1e-13, atol=1e-9)
        np.testing.assert_allclose(G.camera_to_world(w2c, cam[0], cam[1]), P, atol=1e-8)


def test_stats_and_normalise(geo):
    cams = cams_of(geo)
    x2 = G.project_normalize(geo["world"], cams, geo["mean2d"], geo["std2d"], geo["use2d"])
    np.testing.assert_allclose(x2, geo["x2d_norm"], rtol=1e-10, atol=1e-10)
    y3 = G.camera_frame_normalize(geo["world"], cams, geo["mean3d"], geo["std3d"], geo["use3d"])
    np.testing.assert_allclose(y3, geo["y3d_norm"], rtol=1e-10, atol=1e-10)
    # statistics themselves
    all2d = np.vstack([G.project_point_radial(geo["world"].reshape(-1, 3), *c)[0].reshape(-1, 64) for c in cams])
    m, s, ign, use = G.normalization_stats(all2d, 2)
    np.testing.assert_allclose(m, geo["mean2d"], rtol=1e-12)
    np.testing.assert_allclose(s, geo["std2d"], rtol=1e-12)


def test_unnormalise(geo):
    u2 = G.unnormalize(geo["x2d_norm"][1], geo["mean2d"], geo["std2d"], geo["ignore2d"])
    assert np.array_equal(u2, geo["un2d"])          # same fp32 truncation, same fp64 arithmetic
    u3 = G.unnormalize(geo["y3d_norm"][1], geo["mean3d"], geo["std3d"], geo["ignore3d"])
    assert np.array_equal(u3, geo["un3d"])
    # ignored dims come back as the mean
    assert np.array_equal(u3[:, geo["ignore3d"]], np.tile(geo["mean3d"][geo["ignore3d"]], (u3.shape[0], 1)))


def test_similarity_transform(proc):
    X, Y = proc["X"], proc["Y"]
    d, Z, T, b, c = G.similarity_transform(X, Y, compute_optimal_scale=True)
    np.testing.assert_allclose(d, proc["proc_d"], rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(Z, proc["proc_Z"], rtol=1e-9, atol=1e-8)
    np.testing.assert_allclose(T, proc["proc_T"], rtol=1e-9, atol=1e-10)
    np.testing.assert_allclose(b, proc["proc_b"], rtol=1e-10)
    np.testing.assert_allclose(c, proc["proc_c"], rtol=1e-9, atol=1e-8)
    assert np.allclose(np.linalg.det(T), 1.0)          # incl. the reflected pose 5
    d, Z, T, b, c = G.similarity_transform(X, Y, compute_optimal_scale=False)
    np.testing.assert_allclose(d, proc["ns_d"], rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(Z, proc["ns_Z"], rtol=1e-9, atol=1e-8)
    np.testing.assert_allclose(T, proc["ns_T"], rtol=1e-9, atol=1e-10)
    np.testing.assert_allclose(c, proc["ns_c"], rtol=1e-9, atol=1e-8)
    assert np.all(b == 1)


def test_mpjpe(proc):
    args = (proc["pred_n"], proc["gt_n"], proc["mean3d"], proc["std3d"], proc["ignore3d"], proc["use3d"])
    np.testing.assert_allclose(G.mpjpe(*args, procrustes=False), proc["dists_plain"], rtol=1e-12, atol=1e-10)
    np.testing.assert_allclose(G.mpjpe(*args, procrustes=True), proc["dists_procrustes"], rtol=1e-9, atol=1e-8)


def test_procrustes_invariance():
    """Property: aligning a similarity-transformed copy gives zero residual."""
    from oracle import synth
    rng = np.random.RandomState(0)
    X = rng.normal(0, 300, (8, 17, 3))
    for i in range(8):
        R = synth.random_rotation(rng)
        Y = 1.7 * X[i] @ R + rng.normal(0, 100, (1, 3))
        d, Z, T, b, c = G.similarity_transform(X[i], Y, True)
        assert abs(d) < 1e-12
        np.testing.assert_allclose(b * Y @ T + c, X[i], atol=1e-8)
