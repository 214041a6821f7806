"""The bf16x3 training step (LinearModel(..., train_matmul="bf16x3"), P3D_TRAIN_MATMUL_BF16X3) restated in NumPy at its
rounding points and held to the golden fixture (tests/golden/mlp.npz) with the fp32-mode thresholds - the case for
making the route opt-in, re-runnable without a GPU.

Every operand of the three MatMuls of each layer (Z = H W, dH = dZ W^T, dW = H^T dZ; W unclipped, the clip scale
multiplying the product) is split into hi = bf16(a) and lo = bf16(a - hi), and the products hi.hi + lo.hi + hi.lo are
summed in fp32; BatchNorm, ReLU, dropout, the loss and Adam are the oracle's.  The oracle's `quant=` hook (oracle/mlp_ref.py)
already hands every MatMul operand - the unclipped W, the clip scale applied to the product - through one function;
`split_operand` passes each one through unchanged but marked, so that `@` between marked operands is the split product.
As in the CUDA route, the gradient of a bias that feeds a BatchNorm is exactly zero.

At batch <= 64 the emulated step passes the whole fp32-mode golden check (first-step gradients to 2e-4 of each tensor's
max, every step's loss / outputs / learning rate, the final variables after Adam).  At batch 4096 it does not: the split
operands move pre-activations by ~1e-5 relative, which flips the ReLU decision of a few dozen units near zero; the
gradients stay within 1e-2 relative L2 of the fp64 graph, but the max-abs gradient check and the final-variable check
fail.  bf16x3 training is therefore a per-model choice, not the default of bf16x3 models."""
import types

import numpy as np
import pytest

from oracle import mlp_ref as M
from test_oracle_bf16x3 import split
from test_oracle_mlp_golden import GOLD, KEEP, SEED, case_setup


def split_matmul(a, b):
    """a @ b as the bf16x3 GEMMs compute it: fp32 operands split into (hi, lo), hi.hi + lo.hi + hi.lo summed in fp32."""
    ah, al = split(a)
    bh, bl = split(b)
    acc = ah @ bh
    acc += al @ bh
    acc += ah @ bl
    return acc.astype(np.float64)


class SplitOperand(np.ndarray):
    """A MatMul operand of the emulated step: `a @ b` between such operands is split_matmul(a, b)."""

    def __matmul__(self, other):
        return split_matmul(np.asarray(self), np.asarray(other))

    def __rmatmul__(self, other):
        return split_matmul(np.asarray(other), np.asarray(self))


def split_operand(a):
    """The `quant=` function of oracle/mlp_ref.py's forward / backward that turns every MatMul into split_matmul."""
    return np.asarray(a).view(SplitOperand)


def bn_fed_biases(cfg):
    """Names of the biases whose layer feeds a BatchNorm (their true gradient is zero; the CUDA path never moves them)."""
    names = M.layer_names(cfg.num_layers)
    return [b for (_, b, bns) in names[:-1]] if cfg.batch_norm else []


class EmulatedModel:
    """The surface of LinearModel that the golden training check uses, computed by the emulation."""

    def __init__(self, cfg, p, lr0):
        self.cfg, self.p, self.lr0 = cfg, {k: v.copy() for k, v in p.items()}, lr0
        self.st = M.AdamState()
        self.grads = None

    @property
    def global_step(self):
        return self.st.t

    def step(self, session, x, t, keep, isTraining=True):
        cfg, nh = self.cfg, 2 * self.cfg.num_layers + 1
        if not isTraining:
            y = M.forward(self.p, x, cfg, training=False)
            return M.loss_fn(y, t), None, y
        masks = [M.dropout_mask_philox(SEED, self.st.t, li, x.shape[0], cfg.linear_size, keep) for li in range(nh)]
        y, cache = M.forward(self.p, x, cfg, training=True, keep_prob=keep, masks=masks, want_cache=True, quant=split_operand)
        grads = M.backward(self.p, x, t, cfg, cache, y, quant=split_operand)
        for b in bn_fed_biases(cfg):
            grads[b] = np.zeros_like(grads[b])
        if cfg.batch_norm:
            for li, (_, _, bns) in enumerate(M.layer_names(cfg.num_layers)[:-1]):
                mm, mv = bns + "/moving_mean", bns + "/moving_variance"
                self.p[mm] = self.p[mm] * M.BN_MOMENTUM + cache[li]["mean"] * (1.0 - M.BN_MOMENTUM)
                self.p[mv] = self.p[mv] * M.BN_MOMENTUM + cache[li]["var"] * (1.0 - M.BN_MOMENTUM)
        self.grads = {k: v.astype(np.float32) for k, v in grads.items()}
        lr_t = M.adam_update(self.p, grads, self.st, self.lr0)
        return M.loss_fn(y, t), None, types.SimpleNamespace(value=lr_t), y

    def get_gradients(self):
        return self.grads

    def get_variables(self):
        return {k: v.astype(np.float32) for k, v in self.p.items()}

    def close(self):
        pass


def run_golden_training_check(tag, monkeypatch):
    """test_gpu_mlp_golden.test_fp32_training_steps_match_reference_graph with the emulation in place of the model."""
    import test_gpu_mlp_golden as GG
    monkeypatch.setattr(GG, "model_for", lambda cfg, p, B, lr0, mode: EmulatedModel(cfg, p, lr0))
    GG.test_fp32_training_steps_match_reference_graph(np.load(GOLD), tag)


@pytest.mark.parametrize("tag", ["s_res_bn_mn", "s_res_bn", "s_bn_mn_1", "s_res_3", "s_mn", "s_p14", "s_fresh",
                                 "h_1024_b64", "h_1024_b64_nomn"])
def test_small_batches_meet_the_fp32_golden_check(tag, monkeypatch):
    run_golden_training_check(tag, monkeypatch)


def _worst_maxabs(grads, ref):
    return max(np.abs(grads[n] - g).max() / np.abs(g).max() for n, g in ref.items() if np.abs(g).max() > 1e-12)


def test_batch_4096_is_why_the_route_is_opt_in():
    """At h_1024_b4096: ReLU flips against fp64, gradients within 1e-2 relative L2 but not within the 2e-4 max-abs bound,
    losses and outputs within the golden bounds, some final variables outside them."""
    z = np.load(GOLD)
    tag = "h_1024_b4096"
    cfg, p, x, t, B, steps, big, lr0 = case_setup(z, tag)
    nh = 2 * cfg.num_layers + 1
    masks = [M.dropout_mask_philox(SEED, 0, li, B, cfg.linear_size, KEEP) for li in range(nh)]
    y64, c64 = M.forward(p, x, cfg, training=True, keep_prob=KEEP, masks=masks, want_cache=True)
    g64 = M.backward(p, x, t, cfg, c64, y64)
    for b in bn_fed_biases(cfg):
        g64[b] = np.zeros_like(g64[b])
    ye, ce = M.forward(p, x, cfg, training=True, keep_prob=KEEP, masks=masks, want_cache=True, quant=split_operand)
    ge = M.backward(p, x, t, cfg, ce, ye, quant=split_operand)
    flips = sum(int((c64[li]["relu_mask"] != ce[li]["relu_mask"]).sum()) for li in range(nh))
    assert flips > 0
    for n, g in g64.items():
        if np.abs(g).max() > 1e-12:
            assert np.linalg.norm(ge[n] - g) <= 1e-2 * np.linalg.norm(g), n
    assert _worst_maxabs(ge, g64) > 2e-4
    # the multi-step check: losses and outputs pass, the final variables do not
    from test_gpu_mlp_golden import entries
    m = EmulatedModel(cfg, p, lr0)
    for s in range(steps):
        loss, _, lrs, y = m.step(None, x, t, KEEP, isTraining=True)
        rl = float(z[tag + "/train_loss"][s])
        assert abs(loss - rl) <= 2e-4 * max(1.0, rl)
        ref, got = entries(z, tag + "/train_y%d" % s, y)
        assert np.abs(got - ref).max() <= 3e-4 * max(np.abs(ref).max(), 1.0)
    got, move, worst = m.get_variables(), lr0 * steps, 0.0
    for n in p:
        if n in bn_fed_biases(cfg) or n.endswith(("moving_mean", "moving_variance")):
            continue
        ref, g = entries(z, tag + "/final/" + n, got[n])
        err = np.abs(g - ref)          # the two bounds of the golden check, as fractions of their limits
        worst = max(worst, np.quantile(err, 0.995) / (0.02 * move + 1e-6 * np.abs(ref).max()), err.max() / (2.2 * move))
    assert worst > 1.0, worst
