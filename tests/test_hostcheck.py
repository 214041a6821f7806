"""The device math header (csrc/math_hd.h) compiled for the host with g++ and compared with the
oracle/golden vectors - catches arithmetic mistakes in the kernels' inner functions without a GPU."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def hc():
    src = os.path.join(HERE, "hostcheck", "hostcheck.cpp")
    out_dir = os.path.join(HERE, "hostcheck", "_build")
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, "libhostcheck.so")
    subprocess.run(["g++", "-O2", "-shared", "-fPIC", "-ffp-contract=off", "-o", so, src], check=True)
    return ctypes.CDLL(so)


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def test_kabsch_matches_reference_svd(hc, golden_dir):
    g = np.load(os.path.join(golden_dir, "procrustes.npz"))
    X, Y = g["X"], g["Y"]
    X0 = X - X.mean(1, keepdims=True); Y0 = Y - Y.mean(1, keepdims=True)
    nx = np.sqrt((X0 ** 2).sum((1, 2))); ny = np.sqrt((Y0 ** 2).sum((1, 2)))
    A = np.ascontiguousarray(np.swapaxes(X0 / nx[:, None, None], 1, 2) @ (Y0 / ny[:, None, None]))
    n = A.shape[0]
    T = np.zeros((n, 3, 3)); tr = np.zeros(n)
    hc.hc_kabsch(_p(A), _p(T), _p(tr), n)
    np.testing.assert_allclose(T, g["proc_T"], atol=1e-10)
    b = tr * nx / ny
    np.testing.assert_allclose(b, g["proc_b"], rtol=1e-10)
    np.testing.assert_allclose(1 - tr ** 2, g["proc_d"], atol=1e-11)
    assert np.allclose(np.linalg.det(T), 1.0)


def test_kabsch_random_and_reflections(hc):
    from oracle import geometry_ref as G
    rng = np.random.RandomState(5)
    n = 500
    X = rng.normal(0, 1, (n, 17, 3)); Y = rng.normal(0, 1, (n, 17, 3))
    Y[::3] = X[::3] * np.array([1, 1, -1.0]) + rng.normal(0, 0.05, (len(X[::3]), 17, 3))   # mirrored copies
    Y[1::7, :, 2] *= 1e-4                                                                    # nearly planar
    d, Z, Tref, bref, c = G.similarity_transform(X, Y, True)
    X0 = X - X.mean(1, keepdims=True); Y0 = Y - Y.mean(1, keepdims=True)
    nx = np.sqrt((X0 ** 2).sum((1, 2))); ny = np.sqrt((Y0 ** 2).sum((1, 2)))
    A = np.ascontiguousarray(np.swapaxes(X0 / nx[:, None, None], 1, 2) @ (Y0 / ny[:, None, None]))
    T = np.zeros((n, 3, 3)); tr = np.zeros(n)
    hc.hc_kabsch(_p(A), _p(T), _p(tr), n)
    np.testing.assert_allclose(T, Tref, atol=1e-8)
    np.testing.assert_allclose(tr * nx / ny, bref, rtol=1e-9, atol=1e-12)


def test_project_point(hc, golden_dir):
    g = np.load(os.path.join(golden_dir, "geometry.npz"))
    P = np.ascontiguousarray(g["world"].reshape(-1, 3)[: len(g["cam0_proj"])])     # the first 48 poses
    for i in range(4):
        cam = np.concatenate([g[f"cam{i}_{k}"].reshape(-1) for k in "RTfckp"]).astype(np.float64)
        out = np.zeros((P.shape[0], 6))
        hc.hc_project_f64(_p(P), _p(cam), _p(out), P.shape[0])
        np.testing.assert_allclose(out[:, :2], g[f"cam{i}_proj"], rtol=1e-12, atol=1e-9)
        np.testing.assert_allclose(out[:, 2], g[f"cam{i}_D"], rtol=1e-13)
        np.testing.assert_allclose(out[:, 3], g[f"cam{i}_radial"], rtol=1e-13)
        np.testing.assert_allclose(out[:, 4], g[f"cam{i}_tan"], rtol=1e-12, atol=1e-15)
        np.testing.assert_allclose(out[:, 5], g[f"cam{i}_r2"], rtol=1e-13)
        P32 = P.astype(np.float32); out32 = np.zeros((P.shape[0], 6), np.float32)
        hc.hc_project_f32(_p(P32), _p(cam), _p(out32), P.shape[0])
        # fp32 arithmetic on ~1000 px coordinates: 1e-3 px absolute
        np.testing.assert_allclose(out32[:, :2], g[f"cam{i}_proj"], atol=2e-3)


def _f32_consts(mean, std, p14):
    """What p3d_procrustes_mpjpe precomputes on the host (csrc/procrustes.cu)."""
    from oracle import geometry_ref as G
    use, ign = G.dims_to_use(3, p14)
    J = len(use) // 3 + (0 if p14 else 1)
    mu = mean[use].reshape(-1, 3)
    mbar = (mu.sum(0) + (0 if p14 else mean[:3])) / J
    return use, ign, J, std[use].astype(np.float32), (mu - mbar).reshape(-1).astype(np.float32), (mean[:3] - mbar).astype(np.float32)


def test_kabsch_f32_random_and_reflections(hc):
    """One-sided Jacobi in fp32 (the MPJPE kernel's rotation) against the float64 SVD of the oracle."""
    from oracle import geometry_ref as G
    rng = np.random.RandomState(5)
    n = 5000
    X = rng.normal(0, 1, (n, 17, 3)); Y = rng.normal(0, 1, (n, 17, 3))
    Y[::3] = X[::3] * np.array([1, 1, -1.0]) + rng.normal(0, 0.05, (len(X[::3]), 17, 3))   # mirrored copies
    Y[1::7, :, 2] *= 1e-4                                                                    # nearly planar
    Y[2::5] = X[2::5] + rng.normal(0, 0.1, (len(X[2::5]), 17, 3))                           # good predictions
    d, Z, Tref, bref, c = G.similarity_transform(X, Y, True)
    X0 = X - X.mean(1, keepdims=True); Y0 = Y - Y.mean(1, keepdims=True)
    nx = np.sqrt((X0 ** 2).sum((1, 2))); ny = np.sqrt((Y0 ** 2).sum((1, 2)))
    A = np.ascontiguousarray((np.swapaxes(X0 / nx[:, None, None], 1, 2) @ (Y0 / ny[:, None, None])).astype(np.float32))
    T = np.zeros((n, 3, 3), np.float32); tr = np.zeros(n, np.float32)
    hc.hc_kabsch_f32(_p(A), _p(T), _p(tr), n)
    err = np.abs(T - Tref).max((1, 2))
    # conditioning of the rotation: 1 / (s2 + s3') where s3' carries the reflection sign
    assert np.median(err) < 5e-7 and err.max() < 1e-4
    np.testing.assert_allclose(tr * nx / ny, bref, rtol=2e-6, atol=1e-6)
    assert np.abs(np.linalg.det(T.astype(np.float64)) - 1).max() < 1e-5


@pytest.mark.parametrize("p14", [False, True])
@pytest.mark.parametrize("use_proc", [True, False])
def test_pose_errors_f32_against_oracle(hc, p14, use_proc):
    from oracle import geometry_ref as G
    from oracle import synth
    N = 20011
    gt96, pr96 = synth.eval_pairs(N, seed=21)
    rng = np.random.RandomState(2)
    mean = rng.normal(0, 50, 96); mean[:3] = 0
    std = rng.uniform(50, 200, 96)
    use, ign, J, sd, mc, hipc = _f32_consts(mean, std, p14)
    gt_n = np.ascontiguousarray(((gt96[:, use] - mean[use]) / std[use]).astype(np.float32))
    pr_n = np.ascontiguousarray(((pr96[:, use] - mean[use]) / std[use]).astype(np.float32))
    ref = G.mpjpe(pr_n, gt_n, mean, std, ign, use, procrustes=use_proc, predict_14=p14)
    d = np.zeros((N, J), np.float32)
    hc.hc_pose_errors_f32(_p(gt_n), _p(pr_n), _p(sd), _p(mc), _p(hipc), len(use), int(use_proc), _p(d), N)
    assert np.abs(d - ref).max() < 1e-3                                   # every single distance, mm
    assert abs(d.astype(np.float64).mean() - ref.mean()) < 1e-5           # MPJPE
    assert np.abs(d.astype(np.float64).mean(0) - ref.mean(0)).max() < 1e-4


def test_pose_errors_f32_golden(hc, golden_dir):
    from oracle import geometry_ref as G
    g = np.load(os.path.join(golden_dir, "procrustes.npz"))
    use, ign, J, sd, mc, hipc = _f32_consts(g["mean3d"], g["std3d"], False)
    gt32 = np.ascontiguousarray(g["gt_n"].astype(np.float32)); pr = np.ascontiguousarray(g["pred_n"].astype(np.float32))
    for use_proc in (True, False):
        d = np.zeros((len(pr), J), np.float32)
        hc.hc_pose_errors_f32(_p(gt32), _p(pr), _p(sd), _p(mc), _p(hipc), 48, int(use_proc), _p(d), len(pr))
        gold = g["dists_procrustes"] if use_proc else g["dists_plain"]
        assert np.abs(d - gold).max() < 1e-3
