"""Generate tests/golden/*.npz by RUNNING THE REFERENCE's own NumPy code.

Run in the build container only (needs /root/reference):
    python oracle/make_golden.py
The fixtures are committed; nothing at test/bench time reads /root/reference.

What is pinned:
  geometry.npz  - cameras.project_point_radial / world_to_camera_frame / camera_to_world_frame
                  (src/cameras.py:13-90), data_utils.normalization_stats / normalize_data /
                  unNormalizeData / postprocess_3d / project_to_cameras /
                  transform_world_to_camera (src/data_utils.py:195-311,339-364,474-494)
  procrustes.npz- procrustes.compute_similarity_transform (src/procrustes.py:2-63) per pose, both
                  scale modes, including a reflection case, and the MPJPE arithmetic of
                  predict_3dpose.evaluate_batches (src/predict_3dpose.py:399-442) re-typed here
                  around the reference's functions (predict_3dpose.py itself needs TensorFlow).
  tables.npz    - index tables and the SH->H36M permutation assert (data_utils.py:135-136).
The MLP (linear_model.py) cannot be executed (TensorFlow absent): no golden vectors for it.
"""
import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

for n in ["h5py", "matplotlib", "matplotlib.pyplot", "matplotlib.image", "mpl_toolkits",
          "mpl_toolkits.mplot3d", "viz"]:
    sys.modules[n] = types.ModuleType(n)
sys.modules["mpl_toolkits.mplot3d"].Axes3D = object
sys.path.insert(0, "/root/reference/src")
import cameras as ref_cam            # noqa: E402
import data_utils as ref_du          # noqa: E402
import procrustes as ref_pr          # noqa: E402

from oracle import synth             # noqa: E402

out_dir = os.path.join(ROOT, "tests", "golden")
os.makedirs(out_dir, exist_ok=True)

# ------------------------------------------------------------------ geometry
N = 64
cams = synth.cameras(4, seed=3)
world = synth.world_poses(N, seed=3)                          # [N,96] float64
g = {"world": world}
pts = world[:48].reshape(-1, 3)          # per-point camera arrays for the first 48 poses: keeps the file under 1 MB
for ci, (R, T, f, c, k, p) in enumerate(cams):
    g[f"cam{ci}_R"], g[f"cam{ci}_T"], g[f"cam{ci}_f"] = R, T, f
    g[f"cam{ci}_c"], g[f"cam{ci}_k"], g[f"cam{ci}_p"] = c, k, p
    proj, D, radial, tan, r2 = ref_cam.project_point_radial(pts, R, T, f, c, k, p)
    g[f"cam{ci}_proj"], g[f"cam{ci}_D"], g[f"cam{ci}_radial"] = proj, D, radial
    g[f"cam{ci}_tan"], g[f"cam{ci}_r2"] = tan, r2
    w2c = ref_cam.world_to_camera_frame(pts, R, T)
    g[f"cam{ci}_w2c"] = w2c
    g[f"cam{ci}_c2w"] = ref_cam.camera_to_world_frame(w2c, R, T)

# dictionary drivers, exactly as train() calls them (predict_3dpose.py:197-207)
rcams = {(1, ci + 1): cams[ci] + (f"cam{ci}",) for ci in range(4)}
poses_set = {(1, "Walking", "Walking 1.h5"): world.copy()}
t2d = ref_du.project_to_cameras(poses_set, rcams, ncams=4)
t3d = ref_du.transform_world_to_camera(poses_set, rcams, ncams=4)
t3d_keys = sorted(t3d.keys())
t3d, roots = ref_du.postprocess_3d(t3d)
all2d = np.vstack([t2d[k] for k in sorted(t2d.keys())])
all3d = np.vstack([t3d[k] for k in t3d_keys])
m2, s2, ig2, use2 = ref_du.normalization_stats(all2d, dim=2)
m3, s3, ig3, use3 = ref_du.normalization_stats(all3d, dim=3)
m3_14, s3_14, ig3_14, use3_14 = ref_du.normalization_stats(all3d, dim=3, predict_14=True)
n2d = ref_du.normalize_data({k: v.copy() for k, v in t2d.items()}, m2, s2, use2)
n3d = ref_du.normalize_data({k: v.copy() for k, v in t3d.items()}, m3, s3, use3)
g["keys2d"] = np.array(["|".join(map(str, k)) for k in sorted(t2d.keys())])
g["x2d_norm"] = np.stack([n2d[k] for k in sorted(t2d.keys())])      # [4,N,32]
g["y3d_norm"] = np.stack([n3d[k] for k in t3d_keys])                # [4,N,48]
g["roots"] = np.stack([roots[k] for k in t3d_keys])
g.update(mean2d=m2, std2d=s2, ignore2d=ig2, use2d=use2, mean3d=m3, std3d=s3, ignore3d=ig3, use3d=use3)
g["un2d"] = ref_du.unNormalizeData(g["x2d_norm"][1], m2, s2, ig2)
g["un3d"] = ref_du.unNormalizeData(g["y3d_norm"][1], m3, s3, ig3)
np.savez_compressed(os.path.join(out_dir, "geometry.npz"), **g)

np.savez_compressed(os.path.join(out_dir, "tables.npz"),
                    use2d=use2, ignore2d=ig2, use3d=use3, ignore3d=ig3,
                    use3d_14=use3_14, ignore3d_14=ig3_14,
                    sh_to_gt_perm=np.array([ref_du.SH_NAMES.index(h) for h in ref_du.H36M_NAMES
                                            if h != "" and h in ref_du.SH_NAMES]))

# ------------------------------------------------------------------ procrustes + MPJPE
M = 48
gt96, pr96 = synth.eval_pairs(M, seed=4)
# make pose 5 a reflection case and pose 6 nearly planar
pr96 = pr96.copy()
tmp = pr96[5].reshape(32, 3).copy(); tmp[:, 0] *= -1.0; pr96[5] = tmp.reshape(-1)
tmp = pr96[6].reshape(32, 3).copy(); tmp[:, 2] *= 1e-3; pr96[6] = tmp.reshape(-1)
gt_n = (gt96[:, use3] - m3[use3]) / s3[use3]
pr_n = (pr96[:, use3] - m3[use3]) / s3[use3]
pr_n32 = pr_n.astype(np.float32)        # model outputs are float32
res = {"gt_n": gt_n, "pred_n": pr_n32, "mean3d": m3, "std3d": s3, "ignore3d": ig3, "use3d": use3}


def reference_eval(dec_out_n, poses3d_n, use_procrustes):
    """predict_3dpose.py:399-432 typed around the reference's own functions."""
    dec_out = ref_du.unNormalizeData(dec_out_n, m3, s3, ig3)
    poses3d = ref_du.unNormalizeData(poses3d_n, m3, s3, ig3)
    dtu3d = np.hstack((np.arange(3), use3))
    dec_out = dec_out[:, dtu3d]
    poses3d = poses3d[:, dtu3d]
    aux = []
    if use_procrustes:
        for j in range(dec_out.shape[0]):
            gt = np.reshape(dec_out[j, :], [-1, 3])
            out = np.reshape(poses3d[j, :], [-1, 3])
            d, Z, T, b, c = ref_pr.compute_similarity_transform(gt, out, compute_optimal_scale=True)
            aux.append((d, Z, T, b, c))
            out = (b * out.dot(T)) + c
            poses3d[j, :] = np.reshape(out, [-1, 17 * 3])
    sqerr = (poses3d - dec_out) ** 2
    dists = np.zeros((sqerr.shape[0], 17))
    for di, k in enumerate(np.arange(0, 17 * 3, 3)):
        dists[:, di] = np.sqrt(np.sum(sqerr[:, k:k + 3], axis=1))
    return dists, aux


d_plain, _ = reference_eval(gt_n, pr_n32, False)
d_proc, aux = reference_eval(gt_n, pr_n32, True)
res["dists_plain"], res["dists_procrustes"] = d_plain, d_proc
res["proc_d"] = np.array([a[0] for a in aux]); res["proc_Z"] = np.stack([a[1] for a in aux])
res["proc_T"] = np.stack([a[2] for a in aux]); res["proc_b"] = np.array([a[3] for a in aux])
res["proc_c"] = np.stack([a[4] for a in aux])
# un-scaled mode on raw 17x3 arrays
gtu = ref_du.unNormalizeData(gt_n, m3, s3, ig3)[:, np.hstack((np.arange(3), use3))].reshape(M, 17, 3)
pru = ref_du.unNormalizeData(pr_n32, m3, s3, ig3)[:, np.hstack((np.arange(3), use3))].reshape(M, 17, 3)
ns = [ref_pr.compute_similarity_transform(gtu[j], pru[j], compute_optimal_scale=False) for j in range(M)]
res["X"], res["Y"] = gtu, pru
res["ns_d"] = np.array([a[0] for a in ns]); res["ns_Z"] = np.stack([a[1] for a in ns])
res["ns_T"] = np.stack([a[2] for a in ns]); res["ns_c"] = np.stack([a[4] for a in ns])
np.savez_compressed(os.path.join(out_dir, "procrustes.npz"), **res)
print("golden vectors written to", out_dir)
for fn in sorted(os.listdir(out_dir)):
    print(" ", fn, os.path.getsize(os.path.join(out_dir, fn)), "bytes")
