"""ctypes binding of libp3d.so (include/p3d.h).

The library is the ONLY compute path: there is no NumPy/torch fallback anywhere in this package.
If libp3d.so has not been built this module raises at import, and every compute entry fails
loudly on a machine without a B200-class device.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libp3d.so")


class P3DError(RuntimeError):
    pass


if not os.path.exists(LIB_PATH):
    raise ImportError(f"{LIB_PATH} is missing - build it with `python 3d-pose-baseline_b200/build.py` "
                      "(there is no CPU fallback)")

lib = C.CDLL(LIB_PATH)

c_void_p, c_int, c_int64, c_size_t, c_float, c_char_p = C.c_void_p, C.c_int, C.c_int64, C.c_size_t, C.c_float, C.c_char_p


class Cfg(C.Structure):
    _fields_ = [("linear_size", c_int), ("num_layers", c_int), ("residual", c_int), ("batch_norm", c_int),
                ("max_norm", c_int), ("predict_14", c_int), ("mode", c_int), ("device", c_int),
                ("learning_rate", c_float)]


class Camera(C.Structure):
    _fields_ = [("R", C.c_double * 9), ("T", C.c_double * 3), ("f", C.c_double * 2), ("c", C.c_double * 2),
                ("k", C.c_double * 3), ("p", C.c_double * 2)]


MODE_BF16, MODE_FP32, MODE_BF16X3, MODE_FP16 = 0, 1, 2, 3
TRAIN_MATMUL_DEFAULT, TRAIN_MATMUL_BF16X3 = 0, 1

# name -> (restype, argtypes): every symbol include/p3d.h declares
PROTOTYPES = {
    "p3d_last_error": (c_char_p, []),
    "p3d_version": (c_int, []),
    "p3d_launch_count": (c_int64, []),
    "p3d_profile_enable": (c_int, [c_int]),
    "p3d_profile_read": (c_int, [C.POINTER(C.c_double), C.POINTER(c_int64)]),
    "p3d_host_alloc": (c_int, [C.POINTER(c_void_p), c_size_t]),
    "p3d_host_free": (c_int, [c_void_p]),
    "p3d_model_create": (c_int, [C.POINTER(Cfg), C.POINTER(c_void_p)]),
    "p3d_model_destroy": (None, [c_void_p]),
    "p3d_model_set_param_host": (c_int, [c_void_p, c_char_p, c_void_p, c_size_t]),
    "p3d_model_get_param_host": (c_int, [c_void_p, c_char_p, c_void_p, c_size_t]),
    "p3d_model_param_count": (c_int, [c_void_p]),
    "p3d_model_param_name": (c_int, [c_void_p, c_int, c_char_p, c_size_t, C.POINTER(c_size_t)]),
    "p3d_model_prepare_inference": (c_int, [c_void_p, c_void_p]),
    "p3d_model_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "p3d_model_mse": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "p3d_model_step_eval_host": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, C.POINTER(c_float), c_int64]),
    "p3d_model_train_step": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_float, C.c_uint64, c_void_p, c_int64,
                                     c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "p3d_nccl_unique_id": (c_int, [c_void_p]),
    "p3d_model_attach_nccl": (c_int, [c_void_p, c_void_p, c_int, c_int]),
    "p3d_model_global_step": (c_int64, [c_void_p]),
    "p3d_project_point_radial_f64": (c_int, [c_void_p, C.POINTER(Camera), c_void_p, c_void_p, c_void_p, c_void_p,
                                             c_void_p, c_int64, c_void_p]),
    "p3d_project_point_radial_f32": (c_int, [c_void_p, C.POINTER(Camera), c_void_p, c_void_p, c_void_p, c_void_p,
                                             c_void_p, c_int64, c_void_p]),
    "p3d_world_to_camera_f64": (c_int, [c_void_p, C.POINTER(Camera), c_void_p, c_int64, c_void_p]),
    "p3d_camera_to_world_f64": (c_int, [c_void_p, C.POINTER(Camera), c_void_p, c_int64, c_void_p]),
    "p3d_project_normalize": (c_int, [c_void_p, C.POINTER(Camera), c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                      c_int, c_void_p, c_void_p, c_int64, c_void_p]),
    "p3d_normalize_f64": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_int64, c_void_p]),
    "p3d_unnormalize_f64": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_int64, c_void_p]),
    "p3d_column_stats_f64": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "p3d_root_center_f64": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p]),
    "p3d_procrustes_mpjpe": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int64, c_void_p,
                                     c_void_p, c_void_p]),
    "p3d_procrustes_mpjpe_f64": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int64, c_void_p,
                                     c_void_p, c_void_p]),
    "p3d_similarity_transform_f64": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int64, c_void_p, c_void_p, c_void_p,
                                             c_void_p, c_void_p, c_void_p]),
    "p3d_debug_stream_mix": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p]),
    "p3d_debug_latency_stamps": (c_int, [c_void_p, c_void_p, c_int]),
    "p3d_crc32c": (C.c_uint32, [c_void_p, c_size_t, C.c_uint32]),
    "p3d_realtime_create": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, C.POINTER(c_void_p)]),
    "p3d_realtime_destroy": (None, [c_void_p]),
    "p3d_realtime_step_host": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "p3d_realtime_step": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "p3d_model_p2p_handle": (c_int, [c_void_p, c_void_p]),
    "p3d_model_p2p_attach": (c_int, [c_void_p, c_void_p, c_int, c_int]),
    "p3d_model_p2p_detach": (c_int, [c_void_p]),
    "p3d_debug_dp_part": (c_int, [c_void_p, c_int, c_void_p]),
    "p3d_model_gathered_outputs": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    "p3d_model_set_train_matmul": (c_int, [c_void_p, c_int]),
    "p3d_model_train_epoch": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_float, C.c_uint64,
                                      c_void_p, c_void_p, c_void_p]),
    "p3d_debug_tc_gemm": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_int, c_int,
                                  c_void_p, c_void_p, c_float, c_int, c_void_p, c_void_p]),
    "p3d_debug_tc_gemm_seg": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_int,
                                      c_int, c_int, c_void_p, c_float, c_int, c_void_p]),
    "p3d_debug_mma_rate": (c_int, [c_int, c_int, c_void_p, c_void_p]),
    "p3d_debug_umma_gemm": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
}

for _name, (_res, _args) in PROTOTYPES.items():
    _fn = getattr(lib, _name)       # AttributeError here = the library does not export a declared symbol
    _fn.restype = _res
    _fn.argtypes = _args


def check(rc: int) -> None:
    if rc != 0:
        msg = lib.p3d_last_error()
        raise P3DError(f"libp3d error {rc}: {msg.decode() if msg else '?'}")


def make_camera(R, T, f, c, k, p) -> Camera:
    """Camera tuple as returned by cameras.load_camera_params (src/cameras.py:92-120)."""
    cam = Camera()
    R = np.asarray(R, dtype=np.float64).reshape(9)
    T = np.asarray(T, dtype=np.float64).reshape(3)
    f = np.asarray(f, dtype=np.float64).reshape(-1)
    if f.size == 1:      # documented as a scalar (cameras.py:22), loaded as 2x1 (cameras.py:112)
        f = np.repeat(f, 2)
    c = np.asarray(c, dtype=np.float64).reshape(2)
    k = np.asarray(k, dtype=np.float64).reshape(3)
    p = np.asarray(p, dtype=np.float64).reshape(2)
    for i in range(9):
        cam.R[i] = R[i]
    for i in range(3):
        cam.T[i] = T[i]; cam.k[i] = k[i]
    for i in range(2):
        cam.f[i] = f[i]; cam.c[i] = c[i]; cam.p[i] = p[i]
    return cam


def np_ptr(a: np.ndarray):
    return a.ctypes.data_as(c_void_p)


def current_stream():
    import torch
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise P3DError("no CUDA device: libp3d has no CPU fallback")
    return torch
