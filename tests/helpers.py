"""Shared helpers for the parity tests (test infrastructure)."""
import numpy as np

from oracle import mlp_ref as M


def bf16_round(a):
    """Round-to-nearest-even to bfloat16, returned as float32 values."""
    a32 = np.ascontiguousarray(np.asarray(a, dtype=np.float32))
    u = a32.view(np.uint32).astype(np.uint64)
    r = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16) << 16
    return r.astype(np.uint32).view(np.float32).reshape(a32.shape)


def emulate_bf16_forward(p, x, cfg, small_batch=False):
    """What the tcgen05 kernel computes, restated in NumPy: folded weights rounded to bf16, the input
    and every hidden activation rounded to bf16 after bias+ReLU and again after the residual add (the
    residual is added by the L2 through a bf16 TMA reduce-add), fp32 accumulation (here
    float64 - the difference is far below the bf16 rounding).  small_batch: the latency path keeps
    activations in fp32 (only the weights are bf16)."""
    folded = M.fold_inference(p, cfg)
    h = np.asarray(x, np.float64) if small_batch else bf16_round(x).astype(np.float64)
    res = None
    last = len(folded) - 1
    for li, (w, b) in enumerate(folded):
        w = bf16_round(w.astype(np.float32)).astype(np.float64)
        z = h @ w + b.astype(np.float32).astype(np.float64)
        if li == last:
            return z
        r = np.maximum(z, 0)
        if not small_batch:
            r = bf16_round(r).astype(np.float64)          # the epilogue stores relu(.) as bf16 ...
        if li == 0 or li % 2 == 1:
            h = r
        else:
            h = (res + r) if cfg.residual else r          # ... and the L2 adds the residual (TMA reduce-add)
            if not small_batch:
                h = bf16_round(h).astype(np.float64)
        if li == 0 or li % 2 == 0:
            res = h


def assert_matches_emulation(y, emu, rms, ref=None):
    """The kernel and the emulation round at the same points but accumulate in different precision, so
    an activation sitting on a bf16 rounding boundary can flip by one bf16 ulp (0.4 % of ITS value); the
    flips compound over the layers into a heavy tail while the MEDIAN difference stays ~1e-6 rms
    (measured on B200: tools/diag_mlp.py).  A wrong tile / column / residual / dropped K slice shifts
    the median by O(1e-2) and fails.  With `ref` (fp64 oracle) the kernel must also be as accurate as
    the emulation is."""
    err = np.abs(np.asarray(y, np.float64) - emu)
    assert np.median(err) <= 1e-3 * rms + 1e-6, (np.median(err), rms)
    assert np.quantile(err, 0.99) <= 2e-2 * rms + 1e-5, (np.quantile(err, 0.99), rms)
    if ref is not None:
        ek, ee = np.abs(np.asarray(y, np.float64) - ref), np.abs(emu - ref)
        for qv in (0.5, 0.9, 0.99):
            assert np.quantile(ek, qv) <= 1.25 * np.quantile(ee, qv) + 1e-5 * rms, (qv, np.quantile(ek, qv), np.quantile(ee, qv))


def rowwise_rel(y, ref):
    num = np.linalg.norm(np.asarray(y, np.float64) - ref, axis=1)
    den = np.maximum(np.linalg.norm(ref, axis=1), 1e-30)
    return num / den


def make_model(cfg, seed=1, bn="trained", mode="bf16", batch_size=64, lr=1e-3, predict_14=False):
    """LinearModel (CUDA) + the oracle's parameter dict holding the same (fp32-representable) values."""
    from p3d import LinearModel
    out = 42 if predict_14 else 48
    p = M.init_params(cfg.linear_size, cfg.num_layers, out_size=out, seed=seed, batch_norm=cfg.batch_norm, bn=bn)
    m = LinearModel(cfg.linear_size, cfg.num_layers, cfg.residual, cfg.batch_norm, cfg.max_norm, batch_size, lr,
                    predict_14=predict_14, mode=mode, seed=seed)
    p32 = {k: v.astype(np.float32) for k, v in p.items()}
    m.set_variables(p32)
    return m, {k: v.astype(np.float64) for k, v in p32.items()}
