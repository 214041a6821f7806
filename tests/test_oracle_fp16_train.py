"""The fp16 training route (LinearModel(..., train_matmul="fp16"), P3D_TRAIN_MATMUL_FP16) restated in NumPy at its
rounding points, against the exact fp64 graph - the case for the route and for its gradient scale, re-runnable without
a GPU.

The route is the bf16 tensor-core route with fp16 in place of bf16 in every 16-bit MatMul operand: x, h and the
unclipped W in the forward pass (the oracle's `quant=` hook of forward()), dy and dz in the backward pass (the hook of
backward()).  Accumulation, BatchNorm, dropout, the loss and the clip scale stay in high precision.  The gradient
operands are stored as fp16(2^k g) with k = floor(log2(B * out)) and the GEMMs that read them multiply by 2^-k, so the
backward hook is g -> fp16(2^k g) / 2^k.  Without the scale, dy = 2 (y - t) / (B out) sinks into fp16's subnormals as
the batch grows: at batch 32768 the unscaled route's weight gradients are further from the fp64 graph than the bf16
route's.  The GPU tests (tests/test_gpu_train_fp16.py) hold the kernels to this emulation."""
import numpy as np
import pytest

from helpers import bf16_round
from oracle import mlp_ref as M
from oracle import synth
from test_oracle_fp16 import fp16_round


def grad_exp(B, out):
    """k of the route's gradient scale 2^k: floor(log2(B * out)) for the GLOBAL batch B."""
    return (int(B) * int(out)).bit_length() - 1


def fp16_operand(a):
    """Forward operands (x, h, the unclipped W) of the fp16 route."""
    return fp16_round(a).astype(np.float64)


def fp16_gradient_operand(B, out, scaled=True):
    """Backward operands (dy, dz) of the fp16 route: fp16(2^k g) / 2^k, or plain fp16(g) with scaled=False."""
    s = 2.0 ** grad_exp(B, out) if scaled else 1.0
    return lambda g: fp16_round(np.asarray(g) * s).astype(np.float64) / s


def bf16_operand(a):
    return bf16_round(a).astype(np.float64)


def emulated_step(p, x, t, cfg, keep, masks, route="fp16"):
    """(loss, y, gradients, forward cache) of one step of `route` ('fp16', 'fp16_unscaled', 'bf16' or 'fp64')."""
    if route == "fp64":
        qf = qb = None
    elif route == "bf16":
        qf = qb = bf16_operand
    else:
        qf, qb = fp16_operand, fp16_gradient_operand(x.shape[0], cfg.out_size, scaled=(route == "fp16"))
    y, cache = M.forward(p, x, cfg, training=True, keep_prob=keep, masks=masks, want_cache=True, quant=qf)
    g = M.backward(p, x, t, cfg, cache, y, quant=qb)
    return M.loss_fn(y, t), y, g, cache


def weight_errors(g, ref):
    """Relative L2 of every weight gradient against ref."""
    return np.array([np.linalg.norm(g[n] - ref[n]) / np.linalg.norm(ref[n]) for n in ref if n.rsplit("/", 1)[-1][0] == "w"])


def case(B, L=256, seed=5, keep=0.5):
    cfg = M.Config(L, 2, True, True, True)
    p = {k: v.astype(np.float32).astype(np.float64) for k, v in M.init_params(L, 2, seed=seed, bn="trained").items()}
    x, t = synth.mlp_inputs(B, seed=seed)
    masks = list((np.random.RandomState(seed).uniform(size=(5, B, L)) < keep).astype(np.uint8))
    return cfg, p, x.astype(np.float64), t.astype(np.float64), keep, masks


def errors(B):
    cfg, p, x, t, keep, masks = case(B)
    _, y64, g64, _ = emulated_step(p, x, t, cfg, keep, masks, "fp64")
    out = {}
    for route in ("bf16", "fp16", "fp16_unscaled"):
        _, y, g, _ = emulated_step(p, x, t, cfg, keep, masks, route)
        e = weight_errors(g, g64)
        out[route] = (e.max(), np.median(e), np.abs(y - y64).max() / np.abs(y64).max())
    return out


def test_grad_exp_puts_the_scaled_dy_in_one_binade():
    for B, out in [(1, 48), (64, 48), (4096, 48), (32768, 42), (3, 42)]:
        k = grad_exp(B, out)
        assert 2 ** k <= B * out < 2 ** (k + 1)
        f = 2.0 ** k * 2.0 / (B * out)          # 2^k dy / (y - t)
        assert 1.0 < f <= 2.0


# Width 256, 2 blocks, residual, trained BN, max_norm, injected keep-0.5 masks, seed 5.  Relative L2 of the six weight
# gradients against the fp64 graph (max, median) and max |y - y64| / max |y64|, as measured:
#   batch    bf16 route            fp16 route            fp16 without the scale
#   64       9.8e-2 7.8e-2 4.7e-3  2.5e-2 1.7e-2 5.2e-4  2.5e-2 1.7e-2
#   4096     8.8e-2 7.8e-2 3.7e-3  3.1e-2 2.7e-2 4.8e-4  3.2e-2 2.8e-2
#   32768    8.0e-2 6.4e-2 4.2e-3  2.7e-2 2.2e-2 5.2e-4  2.2e-1 1.1e-1
PINNED = {64: {"bf16": (9.84e-2, 7.77e-2), "fp16": (2.53e-2, 1.66e-2), "fp16_unscaled": (2.53e-2, 1.66e-2)},
          4096: {"bf16": (8.79e-2, 7.78e-2), "fp16": (3.12e-2, 2.73e-2), "fp16_unscaled": (3.16e-2, 2.80e-2)},
          32768: {"bf16": (7.96e-2, 6.36e-2), "fp16": (2.71e-2, 2.20e-2), "fp16_unscaled": (2.21e-1, 1.06e-1)}}


@pytest.mark.parametrize("B", [64, 4096, 32768])
def test_fp16_route_gradients_are_closer_to_the_fp64_graph(B):
    e = errors(B)
    for route, (mx, med) in PINNED[B].items():
        assert e[route][0] == pytest.approx(mx, rel=0.05) and e[route][1] == pytest.approx(med, rel=0.05), (route, e[route])
    # at least 2x closer than the bf16 route, worst tensor and median
    assert e["fp16"][0] <= 0.5 * e["bf16"][0] and e["fp16"][1] <= 0.5 * e["bf16"][1], e
    # forward outputs about 8x closer
    assert e["fp16"][2] <= 0.2 * e["bf16"][2], e
    if B == 32768:
        # without the gradient scale the route loses to bf16 at a large batch
        assert e["fp16_unscaled"][0] > 2 * e["bf16"][0] and e["fp16_unscaled"][1] > e["bf16"][1], e
