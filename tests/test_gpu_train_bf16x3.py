"""The bf16x3 training route (LinearModel(..., train_matmul="bf16x3"), P3D_TRAIN_MATMUL_BF16X3): every MatMul of the
step as three split-bf16 tcgen05 products, everything else as on the FFMA route of fp32 mode.

Held to (1) the fp32-mode golden training check on the fixture cases its CPU emulation passes
(tests/test_oracle_bf16x3_train.py), (2) that emulation - the oracle with the split products as its MatMuls: loss and
outputs within 1e-4, every gradient within 1e-3 relative L2 and, at batch <= 64, within 2e-4 of the tensor's max.  A
unit whose pre-activation lies within rounding of zero takes its ReLU decision from the summation order, which differs
between kernel and emulation (measured on a B200: one such unit moves a BN gradient by up to 3e-3 relative L2), so with
injected masks those units (|a| < 1e-4 rms, about one in ten thousand) are dropped on both sides; with generated
(Philox) masks the gradients are held to 1e-2 relative L2 - a wrong dropout counter costs O(1).  (3) The fp64 graph at
batch 4096 (gradients within 1e-2 relative L2; the emulation is at 2.5e-3).  Also: the default route is untouched
(bit-identical to fp32 mode), widths the tcgen05 GEMM does not tile stay on FFMA, train_epoch and graph replays,
inference on the trained weights, the refusals, two-rank data parallelism."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from helpers import rowwise_rel
from oracle import mlp_ref as M
from oracle import synth
from test_oracle_bf16x3_train import bn_fed_biases, split_matmul, split_operand

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def x3_model(cfg, seed=31, bn="trained", mode="bf16x3", lr=1e-3, batch_size=64, train_matmul="bf16x3"):
    from p3d import LinearModel
    p = M.init_params(cfg.linear_size, cfg.num_layers, out_size=cfg.out_size, seed=seed, batch_norm=cfg.batch_norm, bn=bn)
    m = LinearModel(cfg.linear_size, cfg.num_layers, cfg.residual, cfg.batch_norm, cfg.max_norm, batch_size, lr,
                    predict_14=(cfg.out_size == 42), mode=mode, seed=seed, train_matmul=train_matmul)
    p32 = {k: v.astype(np.float32) for k, v in p.items()}
    m.set_variables(p32)
    return m, {k: v.astype(np.float64) for k, v in p32.items()}


def emulated_step(p, x, t, cfg, keep, masks):
    y, cache = M.forward(p, x, cfg, training=True, keep_prob=keep, masks=masks, want_cache=True, quant=split_operand)
    g = M.backward(p, x, t, cfg, cache, y, quant=split_operand)
    for b in bn_fed_biases(cfg):
        g[b] = np.zeros_like(g[b])
    return M.loss_fn(y, t), y, g


def exclude_ambiguous_units(p, x, cfg, masks, keep, thr=1e-4):
    """Zero, in the injected keep-masks, every hidden unit whose emulated pre-ReLU value lies within thr * rms of zero
    (layer by layer: a mask changes what the next layer sees)."""
    names = M.layer_names(cfg.num_layers)
    for li in range(len(names) - 1):
        _, cache = M.forward(p, x, cfg, training=True, keep_prob=keep, masks=masks, want_cache=True, quant=split_operand)
        c = cache[li]
        if cfg.batch_norm:
            bns = names[li][2]
            a = c["xhat"] * p[bns + "/gamma"] + p[bns + "/beta"]
        else:
            a = split_matmul(c["h_in"], c["wc"]) * c["s"] + p[names[li][1]]
        masks[li] = np.where(np.abs(a) < thr * np.sqrt(np.mean(a * a)), 0, masks[li]).astype(np.uint8)
    return masks


def check_against(loss, y, got, rloss, ry, rg, B, l2_tol=1e-3, what=""):
    assert abs(float(loss) - rloss) <= 1e-4 * max(1.0, rloss), (what, float(loss), rloss)
    assert np.abs(y - ry).max() <= 1e-4 * max(np.abs(ry).max(), 1.0), (what, np.abs(y - ry).max())
    for name, g in rg.items():
        k = got[name].astype(np.float64)
        if np.abs(g).max() < 1e-12:
            assert np.abs(k).max() == 0.0, (what, name)          # bias in front of a BatchNorm: exactly zero
            continue
        rel = np.linalg.norm(k - g) / np.linalg.norm(g)
        assert rel <= l2_tol, (what, name, rel)
        if B <= 64:
            assert np.abs(k - g).max() <= 2e-4 * np.abs(g).max(), (what, name, np.abs(k - g).max() / np.abs(g).max())


# ---------------------------------------------------------------------------------------------- golden fixture

@pytest.mark.parametrize("tag,mode", [("s_res_bn_mn", "bf16x3"), ("s_p14", "bf16x3"), ("h_1024_b64", "bf16x3"),
                                      ("h_1024_b64", "fp32")])
def test_training_steps_match_reference_graph(tag, mode, monkeypatch):
    """The fp32-mode golden check (losses, outputs, learning rates, first-step gradients, final variables, an inference
    pass) on a model whose training MatMuls run as split products."""
    import test_gpu_mlp_golden as GG
    from p3d import LinearModel

    def model_for(cfg, p, B, lr0, _mode):
        m = LinearModel(cfg.linear_size, cfg.num_layers, cfg.residual, cfg.batch_norm, cfg.max_norm, B, lr0,
                        predict_14=(cfg.out_size == 42), mode=mode, seed=GG.SEED, train_matmul="bf16x3")
        m.set_variables({k: v.astype(np.float32) for k, v in p.items()})
        return m
    monkeypatch.setattr(GG, "model_for", model_for)
    GG.test_fp32_training_steps_match_reference_graph(np.load(GG.GOLD), tag)


# ---------------------------------------------------------------------------------------------- kernels vs emulation

EMU = [
    (M.Config(1024, 2, True, True, True), [64, 200, 1024, 4096]),
    (M.Config(1024, 2, True, True, False), [64, 1024]),
    (M.Config(256, 1, False, True, True), [200]),
    (M.Config(200, 2, True, True, True), [64, 200]),           # ragged width: a multiple of 8, not of 64
    (M.Config(64, 2, True, False, False), [64, 200]),          # no BatchNorm: dz split written by the activation pass
    (M.Config(256, 1, True, True, True, 42), [64, 1024]),      # predict_14: W4 / dy segments of 42 columns
]


@pytest.mark.parametrize("cfg,B", [(c, b) for c, bs in EMU for b in bs],
                         ids=[f"L{c.linear_size}n{c.num_layers}r{int(c.residual)}b{int(c.batch_norm)}m{int(c.max_norm)}o{c.out_size}-B{b}"
                              for c, bs in EMU for b in bs])
def test_step_matches_emulation_injected_masks(cfg, B):
    keep = 0.5
    m, p = x3_model(cfg)
    nh = 2 * cfg.num_layers + 1
    x, _ = synth.mlp_inputs(B, seed=77)
    t = np.random.RandomState(B).standard_normal((B, cfg.out_size)).astype(np.float32)
    masks = list((np.random.RandomState(4).uniform(size=(nh, B, cfg.linear_size)) < keep).astype(np.uint8))
    masks = exclude_ambiguous_units(p, x.astype(np.float64), cfg, masks, keep)
    loss, _, _, y = m.step(None, x, t, keep, isTraining=True, dropout_mask=np.stack(masks))
    got = m.get_gradients()
    m.close()
    rloss, ry, rg = emulated_step(p, x.astype(np.float64), t.astype(np.float64), cfg, keep, masks)
    check_against(loss, y, got, rloss, ry, rg, B, what="emulation")


def test_batch_4096_against_fp64_graph():
    cfg, B, keep = M.Config(1024, 2, True, True, True), 4096, 0.5
    m, p = x3_model(cfg)
    x, t = synth.mlp_inputs(B, seed=5)
    masks = (np.random.RandomState(9).uniform(size=(5, B, 1024)) < keep).astype(np.uint8)
    loss, _, _, y = m.step(None, x, t, keep, isTraining=True, dropout_mask=masks)
    got = m.get_gradients()
    m.close()
    x64, t64 = x.astype(np.float64), t.astype(np.float64)
    ry, cache = M.forward(p, x64, cfg, training=True, keep_prob=keep, masks=list(masks), want_cache=True)
    rg = M.backward(p, x64, t64, cfg, cache, ry)
    assert abs(float(loss) - M.loss_fn(ry, t64)) <= 1e-4 * M.loss_fn(ry, t64)
    for name in bn_fed_biases(cfg):
        assert np.abs(got[name]).max() == 0.0, name
        rg.pop(name)
    worst = max(np.linalg.norm(got[n].astype(np.float64) - g) / np.linalg.norm(g) for n, g in rg.items())
    assert worst <= 1e-2, worst


@pytest.mark.parametrize("B", [64, 1024])
def test_generated_dropout_feeds_the_same_philox_stream(B):
    """Without dropout_mask the step draws the documented Philox stream (M.dropout_mask_philox): the emulation run with
    those masks is the reference."""
    cfg, keep = M.Config(1024, 2, True, True, True), 0.5
    m, p = x3_model(cfg)
    x, t = synth.mlp_inputs(B, seed=3)
    loss, _, _, y = m.step(None, x, t, keep, isTraining=True)
    got, seed = m.get_gradients(), m._seed
    m.close()
    masks = [M.dropout_mask_philox(seed, 0, li, B, 1024, keep) for li in range(5)]
    rloss, ry, rg = emulated_step(p, x.astype(np.float64), t.astype(np.float64), cfg, keep, masks)
    check_against(loss, y, got, rloss, ry, rg, B=B + 64, l2_tol=1e-2, what="philox")      # no max-abs bound: see above


# ---------------------------------------------------------------------------------------------- replays, epochs

def test_train_epoch_equals_stepping_through_the_batches():
    cfg = M.Config(256, 1, True, True, True)
    n, B, keep = 1000, 64, 0.7
    x, t = synth.mlp_inputs(n, seed=12)
    perm = np.random.RandomState(3).permutation(n)
    ma, _ = x3_model(cfg, seed=5, bn="fresh")
    mb, _ = x3_model(cfg, seed=5, bn="fresh")
    losses, lr = ma.train_epoch(x, t, keep, perm=perm)
    assert losses.shape == (n // B,) and int(ma.global_step) == n // B
    ref = []
    for b in range(n // B):
        idx = perm[b * B:(b + 1) * B]
        loss, _, lrs, _ = mb.step(None, x[idx], t[idx], keep, isTraining=True)
        ref.append(float(loss))
    np.testing.assert_allclose(losses, np.array(ref), rtol=2e-4, atol=1e-6)
    assert abs(lr - float(lrs.value)) < 1e-9
    va, vb = ma.get_variables(), mb.get_variables()
    for k in va:
        assert np.abs(va[k] - vb[k]).max() <= 2e-3 * max(np.abs(vb[k]).max(), 1e-3), k
    ma.close(); mb.close()


def test_graph_replay_equals_the_eager_first_step():
    """The first step of a batch size runs directly, the second is captured, the third and later are replays.  At
    learning rate 0 and without dropout (generated masks are keyed by the global step) the variables do not move, so
    every step of the same batch computes the same thing: the replays must equal the eager first step (to the order of
    the split-K weight gradients' fp32 atomics).  Dropout under replays: test_train_epoch_equals_stepping_through_the_batches."""
    cfg, B = M.Config(1024, 2, True, True, True), 256
    m, _ = x3_model(cfg, seed=2, lr=0.0)
    x, t = synth.mlp_inputs(B, seed=40)
    runs = []
    for s in range(4):
        loss, _, _, y = m.step(None, x, t, 1.0, isTraining=True)
        runs.append((float(loss), y, m.get_gradients()))
    m.close()
    l0, y0, g0 = runs[0]
    for s, (l, y, g) in enumerate(runs[1:], 1):
        assert abs(l - l0) <= 1e-6 * l0, s
        assert rowwise_rel(y, y0.astype(np.float64)).max() <= 1e-6, s
        for k in g0:
            assert np.linalg.norm(g[k] - g0[k]) <= 1e-5 * max(np.linalg.norm(g0[k]), 1e-30), (s, k)


# ---------------------------------------------------------------------------------------------- the default and the edges

def _step_and_state(m, x, t, masks):
    m.step(None, x, t, 0.5, isTraining=True, dropout_mask=masks)
    return m.get_gradients(), m.get_variables(include_optimizer=True)


def _assert_bit_identical(a, b):
    (ga, va), (gb, vb) = a, b
    for k in gb:
        assert np.array_equal(ga[k], gb[k]), k
    for k in vb:
        assert np.array_equal(va[k], vb[k]), k


def test_default_route_is_unchanged():
    """A bf16x3 model without the keyword, and one set back to P3D_TRAIN_MATMUL_DEFAULT, train bit-identically to an
    fp32-mode model (the FFMA route)."""
    from p3d import _lib
    cfg, B = M.Config(256, 2, True, True, True), 64
    x, t = synth.mlp_inputs(B, seed=8)
    masks = (np.random.RandomState(1).uniform(size=(5, B, 256)) < 0.5).astype(np.uint8)
    ref_m, _ = x3_model(cfg, mode="fp32", train_matmul=None)
    ref = _step_and_state(ref_m, x, t, masks)
    plain, _ = x3_model(cfg, train_matmul=None)
    assert plain.train_matmul is None
    _assert_bit_identical(_step_and_state(plain, x, t, masks), ref)
    back, _ = x3_model(cfg)
    assert back.train_matmul == "bf16x3"
    _lib.check(_lib.lib.p3d_model_set_train_matmul(back._handle, _lib.TRAIN_MATMUL_DEFAULT))
    _assert_bit_identical(_step_and_state(back, x, t, masks), ref)
    for mm in (ref_m, plain, back):
        mm.close()


def test_ragged_width_keeps_the_ffma_route():
    cfg, B = M.Config(100, 2, True, True, True), 64
    x, t = synth.mlp_inputs(B, seed=9)
    masks = (np.random.RandomState(2).uniform(size=(5, B, 100)) < 0.5).astype(np.uint8)
    a, _ = x3_model(cfg, mode="fp32", train_matmul=None)
    b, _ = x3_model(cfg)
    _assert_bit_identical(_step_and_state(b, x, t, masks), _step_and_state(a, x, t, masks))
    a.close(); b.close()


def test_refusals():
    from p3d import LinearModel, _lib
    with pytest.raises(ValueError):
        LinearModel(256, 1, True, True, True, 64, 1e-3, mode="bf16", train_matmul="bf16x3")
    with pytest.raises(ValueError):
        LinearModel(256, 1, True, True, True, 64, 1e-3, mode="fp32", train_matmul="bf16x2")
    m = LinearModel(256, 1, True, True, True, 64, 1e-3, mode="bf16")
    for kind in (_lib.TRAIN_MATMUL_DEFAULT, _lib.TRAIN_MATMUL_BF16X3):
        assert _lib.lib.p3d_model_set_train_matmul(m._handle, kind) == -1       # P3D_ERR_ARG
    m.close()


def test_inference_after_training_meets_the_fp32_contract():
    """Trained by the split route, then served by bf16x3 inference: outputs within 1e-4 row-wise of the fp64 graph on
    the trained variables."""
    cfg = M.Config(1024, 2, True, True, True)
    m, _ = x3_model(cfg, seed=6, bn="fresh")
    for s in range(5):
        x, t = synth.mlp_inputs(512, seed=60 + s)
        m.step(None, x, t, 0.5, isTraining=True)
    p = {k: v.astype(np.float64) for k, v in m.get_variables().items()}
    x, t = synth.mlp_inputs(3000, seed=99)
    _, _, y = m.step(None, x, t, 1.0, isTraining=False)
    m.prepare_inference()
    _, _, y2 = m.step(None, x, t, 1.0, isTraining=False)
    m.close()
    ref = M.forward(p, x.astype(np.float64), cfg, training=False)
    assert rowwise_rel(y, ref).max() <= 1e-4 and np.array_equal(y, y2)


# ---------------------------------------------------------------------------------------------- data parallel

def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_rank_step_equals_single_device_global_batch():
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(ROOT, "tools", "dp_check_bf16x3.py")]
    r = subprocess.run(cmd, env=dict(os.environ, P3D_SYNC_TIMEOUT_S="60"), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "DP BF16X3 OK" in r.stdout, r.stdout[-3000:] + r.stderr[-3000:]
