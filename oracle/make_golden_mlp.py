"""Generate tests/golden/mlp.npz by EXECUTING THE REFERENCE's own model code.

Run in the build container only (needs /root/reference):
    python oracle/make_golden_mlp.py

`/root/reference/src/linear_model.py` is imported UNMODIFIED; the `tensorflow` it imports is the op-level stand-in under
tests/tf_shim (torch-CPU autograd, float64).  `LinearModel.__init__` builds its graph, `LinearModel.step` runs it -
the wiring of the network, the loss, which variables train, the order bias -> BatchNorm -> ReLU -> dropout -> residual,
the control dependency of the train op on the BatchNorm update ops all come from the reference's lines.  The semantics
of the individual TensorFlow ops are restated in the shim from TensorFlow's sources (cited there); that part, and only
that part, of the MLP parity remains a restatement.

Second reading: `PoseBase` (src/top_vae_3d_pose/models.py:287-481, the TF2 twin with max_norm, BatchNorm and the
residual hard-wired) is cut out of its file by line number (the module as a whole needs yaml configs and argparse
state) and run eagerly on the same shim with the same variables.

Inputs and variables are seeded (oracle.synth / oracle.mlp_ref.init_params, rounded through float32 so that the CUDA
library can hold the very same values); dropout noise is injected as the documented Philox4x32-10 stream
(oracle.mlp_ref.dropout_mask_philox) that the CUDA kernels generate themselves.  Tensors of more than 256
entries are recorded as strided samples, norms and leading blocks, which keeps the fixture under 1 MB.
Nothing at test/bench time reads /root/reference.
"""
import os
import sys
import textwrap
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests", "tf_shim"))
for n in ["h5py", "matplotlib", "matplotlib.pyplot", "matplotlib.image", "mpl_toolkits", "mpl_toolkits.mplot3d", "viz"]:
    sys.modules[n] = types.ModuleType(n)
sys.modules["mpl_toolkits.mplot3d"].Axes3D = object
sys.path.insert(0, "/root/reference/src")

import tensorflow as tf               # noqa: E402  (tests/tf_shim)
assert tf.__version__.endswith("shim")
import linear_model as ref_lm         # noqa: E402  (/root/reference/src/linear_model.py, unmodified)
assert ref_lm.__file__.startswith("/root/reference/src/")

from oracle import mlp_ref as M       # noqa: E402
from oracle import synth              # noqa: E402

KEEP = 0.5
SEED = 1234                            # dropout stream seed (Philox key)


def f32(a):
    return np.asarray(a, np.float64).astype(np.float32).astype(np.float64)


def build(L, nl, residual, bn, max_norm, B, lr, predict_14=False):
    tf.reset_default_graph()
    tf.set_random_seed(11)
    model = ref_lm.LinearModel(L, nl, residual, bn, max_norm, B, lr, "/tmp/p3d_golden_summaries",
                               predict_14=predict_14, dtype=tf.float64)
    return model


def variables_by_name():
    return {v.name: v for v in tf.global_variables()}


def load_params(p):
    byname = variables_by_name()
    for k, v in p.items():
        byname[k].load(v)
    extra = set(byname) - set(p) - {"learning_rate", "global_step"}
    assert not extra, extra
    return byname


def sample(a):
    """What is stored of a tensor: everything (up to 256 entries), or a strided sample of 256 entries + the norm + the
    leading block (16 entries of a vector, 4 rows of an output, 2 rows x 48 columns of a wider matrix); the tests read
    it back with test_oracle_mlp_golden.strided_sample / head_of."""
    a = np.asarray(a, np.float64)
    if a.size <= 256:
        return {"": a}
    flat = a.reshape(-1)
    head = a[:16] if a.ndim == 1 else a[:(4 if a.shape[1] <= 48 else 2), :48]
    return {"@sample": flat[:: 16 * max(1, flat.size // 4093)][:256].copy(), "@norm": np.array(np.linalg.norm(flat)),
            "@head": head.copy()}


def put(out, key, a):
    for suf, v in sample(a).items():
        out[key + suf] = v


def run_case(out, tag, L, nl, residual, bn, max_norm, B, lr=1e-3, predict_14=False, steps=3, bn_init="trained", big=False,
             seed=3):
    osz = 42 if predict_14 else 48
    model = build(L, nl, residual, bn, max_norm, B, lr, predict_14)
    assert model.input_size == 32 and model.output_size == osz
    p = {k: f32(v) for k, v in M.init_params(L, nl, out_size=osz, seed=seed, batch_norm=bn, bn=bn_init).items()}
    if not big:
        p["linear_model/w4"] = f32(p["linear_model/w4"] * 0.01)     # ||w4|| < 1: the not-clipped branch of clip_by_norm
    byname = load_params(p)
    sess = tf.Session()
    sess.run(tf.global_variables_initializer())
    x, t = synth.mlp_inputs(B, out_size=osz, seed=5)
    x, t = x.astype(np.float64), t.astype(np.float64)
    out[tag + "/cfg"] = np.array([L, nl, int(residual), int(bn), int(max_norm), B, int(predict_14), steps, seed, int(big)])
    out[tag + "/lr0"] = np.array(lr)
    out[tag + "/bn_init"] = np.array(bn_init)
    n_hidden = 2 * nl + 1

    # ---- inference through LinearModel.step(isTraining=False): 3-tuple (linear_model.py:239-245)
    tf.set_dropout_masks(None)
    r = model.step(sess, x, t, 1.0, isTraining=False)
    assert len(r) == 3
    out[tag + "/eval_loss"] = np.array(r[0]); put(out, tag + "/eval_y", r[2])
    assert list(r[1].keys()) == ["loss/loss"] and r[1]["loss/loss"] == r[0]

    # ---- gradients of the first training step (opt.compute_gradients, :143-144), no update
    def masks_for(step):
        return [M.dropout_mask_philox(SEED, step, li, B, L, KEEP) for li in range(n_hidden)]
    tf.set_dropout_masks(masks_for(0))
    feed = {model.encoder_inputs: x, model.decoder_outputs: t, model.isTraining: True, model.dropout_keep_prob: KEEP}
    gv = [pair for pair in model.gradients if len(pair)]
    # compute_gradients is called inside `with tf.control_dependencies(update_ops)` (:140-143), so fetching a gradient
    # also runs the BatchNorm moving-average updates - as it would in TensorFlow.  Put the moving statistics back
    # afterwards so that what follows is exactly `steps` calls of LinearModel.step.
    moving = {n: v.eval() for n, v in byname.items() if n.endswith(("moving_mean", "moving_variance"))}
    gvals = sess.run([g for g, _ in gv], feed)
    if bn:
        assert any(np.abs(byname[n].eval() - m).max() > 0 for n, m in moving.items())
    for n, m in moving.items():
        byname[n].load(m)
    names = [v.name for _, v in gv]
    out[tag + "/grad_names"] = np.array(names)
    trainable = M.trainable_names(L, nl, batch_norm=bn)
    assert sorted(names) == sorted(trainable), (names, trainable)      # every W, b, gamma, beta; no moving statistics
    for nme, g in zip(names, gvals):
        put(out, tag + "/grad0/" + nme, g)

    # ---- training steps through LinearModel.step(isTraining=True): 4-tuple (:229-237)
    losses, lrs = [], []
    for s in range(steps):
        tf.set_dropout_masks(masks_for(s))
        r = model.step(sess, x, t, KEEP, isTraining=True)
        assert len(r) == 4
        losses.append(r[0]); lrs.append(r[2]["learning_rate/learning_rate"])
        put(out, tag + "/train_y%d" % s, r[3])
    out[tag + "/train_loss"] = np.array(losses)
    out[tag + "/train_lr"] = np.array(lrs)
    assert int(model.global_step.eval()) == steps
    for nme, v in byname.items():
        if nme in ("learning_rate", "global_step"):
            continue
        put(out, tag + "/final/" + nme, v.eval())

    # ---- inference after training (moving statistics now updated)
    tf.set_dropout_masks(None)
    r = model.step(sess, x, t, 1.0, isTraining=False)
    out[tag + "/eval2_loss"] = np.array(r[0]); put(out, tag + "/eval2_y", r[2])
    print("%-28s eval loss %.6f  train losses %s  lr %s" % (tag, out[tag + "/eval_loss"], np.round(losses, 6), lrs[-1]))
    return p, x


def posebase_case(out, tag, units, p, x):
    """The TF2 twin executed eagerly on the same variables: PoseBase.call(inputs, training=False/True)."""
    path = "/root/reference/src/top_vae_3d_pose/models.py"
    src = open(path).read().split("\n")
    assert src[93].startswith("def kaiming(shape, dtype=tf.float32"), src[93]
    assert src[286].startswith("class PoseBase(tf.keras.Model):"), src[286]
    assert src[480].strip() == "return y_out", src[480]
    tf.reset_default_graph()
    ns = {"tf": tf, "keras": tf.keras}
    exec(textwrap.dedent("\n".join(src[93:106])), ns)
    exec(textwrap.dedent("\n".join(src[286:481])), ns)
    m = ns["PoseBase"](units=units, input_size=32, output_size=48)
    y0 = m(x, training=False)          # builds the BatchNormalization variables
    _ = y0.numpy()
    byname = {v.name: v for v in tf.global_variables()}
    for k, v in p.items():
        byname[k].load(v)
    assert set(byname) == set(p), set(byname) ^ set(p)
    put(out, tag + "/posebase_eval_y", m(x, training=False).numpy())
    put(out, tag + "/posebase_train_y", m(x, training=True).numpy())       # batch statistics, no dropout
    for leaf in ("moving_mean", "moving_variance"):
        out[tag + "/posebase_mm/" + leaf] = byname["linear_model/batch_normalization/" + leaf].eval()


def main():
    out = {}
    small = [("s_res_bn_mn", 48, 2, True, True, True), ("s_res_bn", 48, 2, True, True, False),
             ("s_bn_mn_1", 40, 1, False, True, True), ("s_res_3", 32, 3, True, False, False),
             ("s_mn", 32, 2, False, False, True)]
    for tag, L, nl, res, bn, mn in small:
        run_case(out, tag, L, nl, res, bn, mn, B=24)
    run_case(out, "s_p14", 32, 2, True, True, True, B=24, predict_14=True)
    run_case(out, "s_lr1", 32, 2, True, True, True, B=24, lr=1.0)          # this fork's --learning_rate default
    p, x = run_case(out, "s_fresh", 32, 2, True, True, True, B=24, bn_init="fresh")
    # the headline model: linear_size 1024, 2 blocks, residual, batch norm, max norm, batch 64 (BASELINE configs[0,3])
    p, x = run_case(out, "h_1024_b64", 1024, 2, True, True, True, B=64, big=True, seed=1)
    posebase_case(out, "h_1024_b64", 1024, p, x)
    run_case(out, "h_1024_b64_nomn", 1024, 2, True, True, False, B=64, big=True, seed=1)
    run_case(out, "h_1024_b4096", 1024, 2, True, True, True, B=4096, big=True, seed=1, steps=2)
    path = os.path.join(ROOT, "tests", "golden", "mlp.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes,", len(out), "arrays")


if __name__ == "__main__":
    main()
