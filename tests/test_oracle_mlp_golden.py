"""oracle/mlp_ref.py held to tests/golden/mlp.npz - the outputs of the REFERENCE's own `src/linear_model.py`
(imported unmodified, `LinearModel.__init__` + `LinearModel.step`) executed over the TensorFlow op stand-in of
tests/tf_shim, and of its TF2 twin `PoseBase.call` (oracle/make_golden_mlp.py wrote the fixture in the build
container).  What this pins: the graph wiring, the loss, the set of trainable variables, the train op's dependency on
the BatchNorm update ops, the step()/tuple contract.  What stays a restatement: the arithmetic of each TensorFlow op as
written in the shim from TensorFlow's sources.  Tolerance: 1e-12 relative (both sides are float64)."""
import os

import numpy as np
import pytest

from oracle import mlp_ref as M
from oracle import synth

KEEP, SEED = 0.5, 1234
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "mlp.npz")


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLD)


def cases(z):
    return sorted({k.split("/")[0] for k in z.files})


def case_setup(z, tag):
    L, nl, res, bn, mn, B, p14, steps, seed, big = [int(v) for v in z[tag + "/cfg"]]
    osz = 42 if p14 else 48
    cfg = M.Config(L, nl, bool(res), bool(bn), bool(mn), osz)
    p = M.init_params(L, nl, out_size=osz, seed=seed, batch_norm=bool(bn), bn=str(z[tag + "/bn_init"]))
    p = {k: v.astype(np.float32).astype(np.float64) for k, v in p.items()}
    if not big:
        p["linear_model/w4"] = (p["linear_model/w4"] * 0.01).astype(np.float32).astype(np.float64)
    x, t = synth.mlp_inputs(B, out_size=osz, seed=5)
    return cfg, p, x.astype(np.float64), t.astype(np.float64), B, steps, bool(big), float(z[tag + "/lr0"])


def strided_sample(a):
    """The entries the fixture keeps under key@sample of a tensor of more than 256 entries: 256 entries of the flattened
    tensor at a stride of 16 * (size // 4093), i.e. every 16th point of the 4093-point sample the reference run
    recorded (thinned to keep the fixture under 1 MB)."""
    flat = np.asarray(a, np.float64).reshape(-1)
    return flat[:: 16 * max(1, flat.size // 4093)][:256]


def head_of(a, head):
    """The leading block of `a` that key@head holds (its first rows, and the first columns of a wide matrix)."""
    return np.asarray(a, np.float64)[tuple(slice(0, n) for n in head.shape)]


def stored(z, key):
    """Every entry the fixture holds of a tensor, flattened: the whole tensor, or its sample and leading block."""
    if key in z.files:
        return z[key].reshape(-1)
    return np.concatenate([z[key + "@sample"], z[key + "@head"].reshape(-1)])


def check(z, key, a, rtol=1e-12, ntol=1e-10):
    """Compare `a` with what the fixture holds under `key` (whole tensor, or strided sample + norm + head)."""
    a = np.asarray(a, np.float64)
    if key in z.files:
        ref = z[key]
        assert ref.shape == a.shape, (key, ref.shape, a.shape)
        scale = max(np.abs(ref).max(), 1e-30)
        assert np.abs(a - ref).max() <= rtol * max(scale, 1e-6), (key, np.abs(a - ref).max(), scale)
        return
    smp = strided_sample(a)
    ref = z[key + "@sample"]
    scale = max(np.abs(ref).max(), 1e-30)
    assert np.abs(smp - ref).max() <= rtol * max(scale, 1e-6), (key, np.abs(smp - ref).max(), scale)
    assert abs(np.linalg.norm(a) - float(z[key + "@norm"])) <= ntol * max(float(z[key + "@norm"]), 1e-6), key
    head = z[key + "@head"]
    assert np.abs(head_of(a, head) - head).max() <= rtol * max(np.abs(head).max(), 1e-6), key


def masks_for(step, n_hidden, B, L):
    return [M.dropout_mask_philox(SEED, step, li, B, L, KEEP) for li in range(n_hidden)]


def test_fixture_lists_the_expected_cases(gold):
    cs = cases(gold)
    assert "h_1024_b64" in cs and "h_1024_b4096" in cs and len(cs) >= 11
    L, nl, res, bn, mn, B = [int(v) for v in gold["h_1024_b64/cfg"][:6]]
    assert (L, nl, res, bn, mn, B) == (1024, 2, 1, 1, 1, 64)        # BASELINE configs[0]: the headline model, batch 64


@pytest.mark.parametrize("tag", ["s_res_bn_mn", "s_res_bn", "s_bn_mn_1", "s_res_3", "s_mn", "s_p14", "s_lr1", "s_fresh",
                                 "h_1024_b64", "h_1024_b64_nomn", "h_1024_b4096"])
def test_oracle_matches_the_executed_reference_graph(gold, tag):
    z = gold
    cfg, p, x, t, B, steps, big, lr0 = case_setup(z, tag)
    n_hidden = 2 * cfg.num_layers + 1
    # inference (LinearModel.step(isTraining=False), linear_model.py:239-245)
    y = M.forward(p, x, cfg, training=False)
    check(z, tag + "/eval_y", y)
    assert abs(M.loss_fn(y, t) - float(z[tag + "/eval_loss"])) <= 1e-12 * float(z[tag + "/eval_loss"])
    # folded inference == the graph too
    check(z, tag + "/eval_y", M.forward_folded(M.fold_inference(p, cfg), x, cfg), rtol=1e-10)
    # gradients of the first step (opt.compute_gradients, linear_model.py:143)
    y0, cache = M.forward(p, x, cfg, training=True, keep_prob=KEEP, masks=masks_for(0, n_hidden, B, cfg.linear_size),
                          want_cache=True)
    g = M.backward(p, x, t, cfg, cache, y0)
    names = [str(n) for n in z[tag + "/grad_names"]]
    assert sorted(names) == sorted(g.keys())
    for n in names:
        gref_key = tag + "/grad0/" + n
        a = g[n]
        if np.abs(stored(z, gref_key)).max() < 1e-13:                      # bias in front of BatchNorm: exactly zero
            assert np.abs(a).max() < 1e-12, n
            continue
        check(z, gref_key, a, rtol=1e-9)
    # training steps (LinearModel.step(isTraining=True), :229-237): loss, outputs, decayed learning rate, variables
    st = M.AdamState()
    for s in range(steps):
        loss, lr_t, ys = M.train_step(p, st, x, t, cfg, lr0, keep_prob=KEEP,
                                      masks=masks_for(s, n_hidden, B, cfg.linear_size))
        assert abs(loss - float(z[tag + "/train_loss"][s])) <= 1e-11 * max(1.0, abs(loss)), (s, loss)
        assert abs(lr_t - float(z[tag + "/train_lr"][s])) <= 1e-14 * lr0
        check(z, tag + "/train_y%d" % s, ys, rtol=1e-10)
    for n in p:
        # Adam divides by sqrt(v)+1e-8: where a gradient is ~0 (biases in front of BN) rounding noise decides the
        # direction of a full-size step in TensorFlow; the oracle and the CUDA path keep those biases unchanged
        if cfg.batch_norm and n.rsplit("/", 1)[-1][0] == "b" and not n.endswith(("b4", "beta")):
            continue
        check(z, tag + "/final/" + n, p[n], rtol=1e-8)
    y2 = M.forward(p, x, cfg, training=False)
    assert abs(M.loss_fn(y2, t) - float(z[tag + "/eval2_loss"])) <= 1e-8
    if not cfg.batch_norm:
        check(z, tag + "/eval2_y", y2, rtol=1e-8)


def test_posebase_twin_agrees_with_linear_model(gold):
    """The TF2 twin executed on the same variables (models.py:442-481): same inference outputs as LinearModel's graph,
    and training=True == batch statistics without dropout; its BatchNormalization layers moved their moving averages
    with momentum 0.99."""
    z = gold
    tag = "h_1024_b64"
    cfg, p, x, t, B, steps, big, lr0 = case_setup(z, tag)
    # PoseBase creates float32 variables (its kaiming() defaults to tf.float32), so this reading runs in float32
    np.testing.assert_allclose(stored(z, tag + "/posebase_eval_y"), stored(z, tag + "/eval_y"), rtol=0, atol=2e-6)
    check(z, tag + "/posebase_eval_y", M.forward(p, x, cfg, training=False), rtol=5e-6, ntol=5e-6)
    ytr, cache = M.forward(p, x, cfg, training=True, want_cache=True)
    check(z, tag + "/posebase_train_y", ytr, rtol=5e-6, ntol=5e-6)
    mm = "linear_model/batch_normalization/moving_mean"
    np.testing.assert_allclose(z[tag + "/posebase_mm/moving_mean"], p[mm] * 0.99 + cache[0]["mean"] * 0.01, atol=1e-6)
    mv = "linear_model/batch_normalization/moving_variance"
    np.testing.assert_allclose(z[tag + "/posebase_mm/moving_variance"], p[mv] * 0.99 + cache[0]["var"] * 0.01, atol=1e-6)
