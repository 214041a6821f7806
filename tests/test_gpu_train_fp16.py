"""The fp16 training route (LinearModel(..., train_matmul="fp16"), P3D_TRAIN_MATMUL_FP16): the bf16 tensor-core route's
kernels with fp16 in every 16-bit MatMul operand and the gradient operands scaled by 2^k, k = floor(log2(B * out)).

Held to (1) its NumPy emulation (tests/test_oracle_fp16_train.py) with the metric of the bf16 route's tests: units whose
ReLU derivative rounding decides are dropped through the injected masks on both sides, then loss within 1e-4, outputs
within 3e-3 of their max and every gradient within 5e-3 relative L2; with generated (Philox) masks nothing is excluded
and gradients are held to 5e-2.  Fused epilogues at 64 / 1024 / 4096 poses, the unfused route with P3D_TRAIN_FUSED=0
(and at 32768 poses in the accuracy claim); width 1024, 320 (fused, not a multiple of 256), 200 (unfused only),
predict_14, and residual / BN / max_norm switched off.  (2) The accuracy claim on the device: closer to the fp64 graph
than a bf16-route model holding the same weights.  (3) The golden training check of the bf16 route.  Also: train_epoch,
graph replays, switching back, the largest batch, inference after training, the refusals."""
import numpy as np
import pytest

from oracle import mlp_ref as M
from oracle import synth
from test_oracle_fp16_train import emulated_step, fp16_operand, weight_errors

pytestmark = pytest.mark.gpu
ERR_ARG = -1


def _cid(c):
    return f"L{c.linear_size}n{c.num_layers}r{int(c.residual)}b{int(c.batch_norm)}m{int(c.max_norm)}o{c.out_size}"


def fp16_model(cfg, seed=31, bn="trained", mode="bf16", lr=1e-3, train_matmul="fp16"):
    from p3d import LinearModel
    p = M.init_params(cfg.linear_size, cfg.num_layers, out_size=cfg.out_size, seed=seed, batch_norm=cfg.batch_norm, bn=bn)
    m = LinearModel(cfg.linear_size, cfg.num_layers, cfg.residual, cfg.batch_norm, cfg.max_norm, 64, lr,
                    predict_14=(cfg.out_size == 42), mode=mode, seed=seed, train_matmul=train_matmul)
    p32 = {k: v.astype(np.float32) for k, v in p.items()}
    m.set_variables(p32)
    return m, {k: v.astype(np.float64) for k, v in p32.items()}


def exclude_ambiguous_units(p, x, cfg, masks, keep, thr=2.0 ** -8):
    """Zero, in the injected keep-masks, every hidden unit whose emulated pre-ReLU value lies within thr * rms of zero
    (layer by layer: a mask changes what the next layer sees)."""
    names = M.layer_names(cfg.num_layers)
    for li in range(len(names) - 1):
        _, cache = M.forward(p, x, cfg, training=True, keep_prob=keep, masks=masks, want_cache=True, quant=fp16_operand)
        c = cache[li]
        if cfg.batch_norm:
            bns = names[li][2]
            a = c["xhat"] * p[bns + "/gamma"] + p[bns + "/beta"]
        else:
            a = (c["h_in"] @ c["wc"]) * c["s"] + p[names[li][1]]
        masks[li] = np.where(np.abs(a) < thr * np.sqrt(np.mean(a * a)), 0, masks[li]).astype(np.uint8)
    return masks


def check_against(loss, y, got, rloss, ry, rg, l2_tol, what=""):
    assert abs(float(loss) - rloss) <= 1e-4 * max(1.0, rloss), (what, float(loss), rloss)
    assert np.abs(y - ry).max() <= 3e-3 * max(np.abs(ry).max(), 1.0), (what, np.abs(y - ry).max())
    worst = {}
    for name, g in rg.items():
        k = got[name].astype(np.float64)
        if np.abs(g).max() < 1e-12:
            assert np.abs(k).max() == 0.0, (what, name)           # bias in front of a BatchNorm: exactly zero
            continue
        worst[name] = np.linalg.norm(k - g) / np.linalg.norm(g)
    bad = {k: v for k, v in worst.items() if v > l2_tol}
    assert not bad, (what, bad)


# ---------------------------------------------------------------------------------------------- kernels vs emulation

EMU = [
    (M.Config(1024, 2, True, True, True), [(64, "1"), (1024, "1"), (4096, "1"), (4096, "0")]),
    (M.Config(1024, 2, True, True, False), [(64, "1"), (1024, "0")]),
    (M.Config(320, 2, True, True, True), [(1024, "1"), (1024, "0")]),     # fused at a width that is not a multiple of 256
    (M.Config(200, 2, True, True, True), [(200, "1")]),                    # N % 32 != 0: the unfused route
    (M.Config(256, 2, False, False, False), [(64, "1"), (1024, "0")]),    # no residual / BN / max_norm: dz from the activation pass
    (M.Config(256, 1, True, True, True, 42), [(64, "1"), (1024, "0")]),  # predict_14
]


@pytest.mark.parametrize("cfg,B,fused", [(c, b, f) for c, bs in EMU for b, f in bs],
                         ids=[f"{_cid(c)}-B{b}-{'fused' if f == '1' else 'unfused'}" for c, bs in EMU for b, f in bs])
def test_step_matches_emulation_injected_masks(cfg, B, fused, monkeypatch):
    monkeypatch.setenv("P3D_TRAIN_FUSED", fused)
    keep = 0.5
    m, p = fp16_model(cfg)
    nh = 2 * cfg.num_layers + 1
    x, _ = synth.mlp_inputs(B, seed=77)
    t = np.random.RandomState(B).standard_normal((B, cfg.out_size)).astype(np.float32)
    x64, t64 = x.astype(np.float64), t.astype(np.float64)
    masks = [(np.random.RandomState(40 + li).uniform(size=(B, cfg.linear_size)) < keep).astype(np.uint8) for li in range(nh)]
    masks = exclude_ambiguous_units(p, x64, cfg, masks, keep)
    loss, _, _, y = m.step(None, x, t, keep, isTraining=True, dropout_mask=np.stack(masks))
    got = m.get_gradients()
    m.close()
    rloss, ry, rg, _ = emulated_step(p, x64, t64, cfg, keep, masks)
    check_against(loss, y, got, rloss, ry, rg, 5e-3, what="emulation")


@pytest.mark.parametrize("B,fused", [(64, "1"), (4096, "1"), (4096, "0")])
def test_generated_dropout_matches_emulation(B, fused, monkeypatch):
    """Without dropout_mask the step draws the documented Philox stream (M.dropout_mask_philox)."""
    monkeypatch.setenv("P3D_TRAIN_FUSED", fused)
    cfg, keep = M.Config(1024, 2, True, True, True), 0.5
    m, p = fp16_model(cfg)
    x, t = synth.mlp_inputs(B, seed=3)
    loss, _, _, y = m.step(None, x, t, keep, isTraining=True)
    got, seed = m.get_gradients(), m._seed
    m.close()
    masks = [M.dropout_mask_philox(seed, 0, li, B, 1024, keep) for li in range(5)]
    rloss, ry, rg, _ = emulated_step(p, x.astype(np.float64), t.astype(np.float64), cfg, keep, masks)
    check_against(loss, y, got, rloss, ry, rg, 5e-2, what="philox")


# ---------------------------------------------------------------------------------------------- the accuracy claim

@pytest.mark.parametrize("L,B", [(1024, 64), (1024, 4096), (256, 32768)])
def test_closer_to_the_fp64_graph_than_the_bf16_route(L, B):
    """Same weights, inputs and masks: the fp16 route's weight gradients at most half as far from the fp64 graph as the
    bf16 route's (worst tensor and median; the width-256 emulation gives 2.8-4.7x), its outputs at most a fifth as far.  32768
    poses take the unfused route, where an unscaled fp16 gradient would already lose to bf16."""
    cfg, keep = M.Config(L, 2, True, True, True), 0.5
    x, t = synth.mlp_inputs(B, seed=5)
    masks = (np.random.RandomState(9).uniform(size=(5, B, L)) < keep).astype(np.uint8)
    res = {}
    for tm in ("fp16", None):
        m, p = fp16_model(cfg, seed=5, train_matmul=tm)
        loss, _, _, y = m.step(None, x, t, keep, isTraining=True, dropout_mask=masks)
        res[tm] = (y.astype(np.float64), m.get_gradients())
        m.close()
    _, y64, g64, _ = emulated_step(p, x.astype(np.float64), t.astype(np.float64), cfg, keep, list(masks), "fp64")
    e16, eb = weight_errors(res["fp16"][1], g64), weight_errors(res[None][1], g64)
    assert e16.max() <= 0.5 * eb.max() and np.median(e16) <= 0.5 * np.median(eb), (e16, eb)
    assert np.abs(res["fp16"][0] - y64).max() <= 0.2 * np.abs(res[None][0] - y64).max()
    assert np.isfinite(res["fp16"][0]).all()


# ---------------------------------------------------------------------------------------------- golden fixture

@pytest.mark.parametrize("tag", ["h_1024_b64", "h_1024_b64_nomn", "h_1024_b4096", "s_res_bn_mn"])
@pytest.mark.parametrize("mode", ["bf16", "fp16"])
def test_golden_training_check_of_the_bf16_route(tag, mode, monkeypatch):
    import test_gpu_mlp_golden as GG
    from p3d import LinearModel

    def model_for(cfg, p, B, lr0, _mode):
        m = LinearModel(cfg.linear_size, cfg.num_layers, cfg.residual, cfg.batch_norm, cfg.max_norm, B, lr0,
                        predict_14=(cfg.out_size == 42), mode=mode, seed=GG.SEED, train_matmul="fp16")
        m.set_variables({k: v.astype(np.float32) for k, v in p.items()})
        return m
    monkeypatch.setattr(GG, "model_for", model_for)
    GG.test_bf16_training_steps_match_reference_graph(np.load(GG.GOLD), tag)


# ---------------------------------------------------------------------------------------------- routes and graphs

def test_train_epoch_equals_stepping_through_the_batches():
    cfg = M.Config(1024, 2, True, True, True)
    n, B, keep = 1024, 64, 0.7
    x, t = synth.mlp_inputs(n, seed=12)
    perm = np.random.RandomState(3).permutation(n)
    ma, _ = fp16_model(cfg, seed=5, bn="fresh")
    mb, _ = fp16_model(cfg, seed=5, bn="fresh")
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


@pytest.mark.parametrize("B", [256, 32768])
def test_graph_replay_equals_the_eager_first_step(B):
    """First step eager, second captured, later ones replayed; learning rate 0 and no dropout, so every step computes
    the same thing (to the order of the split-K weight gradients' fp32 atomics)."""
    from helpers import rowwise_rel
    cfg = M.Config(1024, 2, True, True, True)
    m, _ = fp16_model(cfg, seed=2, lr=0.0)
    x, t = synth.mlp_inputs(B, seed=40)
    runs = []
    for s in range(4):
        loss, _, _, y = m.step(None, x, t, 1.0, isTraining=True)
        runs.append((float(loss), y, m.get_gradients()))
    m.close()
    l0, y0, g0 = runs[0]
    assert np.isfinite(y0).all() and all(np.isfinite(g).all() for g in g0.values())
    for s, (l, y, g) in enumerate(runs[1:], 1):
        assert abs(l - l0) <= 1e-6 * l0, s
        assert rowwise_rel(y, y0.astype(np.float64)).max() <= 1e-6, s
        for k in g0:
            assert np.linalg.norm(g[k] - g0[k]) <= 1e-5 * max(np.linalg.norm(g0[k]), 1e-30), (s, k)


def test_switching_back_to_the_bf16_route():
    """A model stepped on the fp16 route and set back to P3D_TRAIN_MATMUL_BF16 trains like a bf16 model that never
    switched: steps with the same starting variables match it as closely as a second bf16 model does (the split-K fp32
    atomics make two bf16 runs differ in the last bits)."""
    from p3d import _lib
    cfg, B = M.Config(1024, 2, True, True, True), 512
    x, t = synth.mlp_inputs(B, seed=8)
    masks = (np.random.RandomState(1).uniform(size=(5, B, 1024)) < 0.5).astype(np.uint8)
    sw, p = fp16_model(cfg, seed=3)
    sw.step(None, x, t, 0.5, isTraining=True, dropout_mask=masks)           # compiles, allocates and captures on fp16
    sw.step(None, x, t, 0.5, isTraining=True)
    _lib.check(_lib.lib.p3d_model_set_train_matmul(sw._handle, _lib.TRAIN_MATMUL_BF16))
    start = sw.get_variables(include_optimizer=True)
    ref, _ = fp16_model(cfg, seed=3, train_matmul=None)
    ctl, _ = fp16_model(cfg, seed=3, train_matmul=None)
    for m in (ref, ctl):
        m.set_variables(start)
    outs = []
    for m in (sw, ref, ctl):
        for s in range(3):
            m.step(None, x, t, 0.5, isTraining=True)
        outs.append((m.get_gradients(), m.get_variables(include_optimizer=True)))
    (gs, vs), (gr, vr), (gc, vc) = outs
    for a, b, c in ((gs, gr, gc), (vs, vr, vc)):
        for k in b:
            d = np.linalg.norm(np.asarray(a[k], np.float64) - b[k])
            dc = np.linalg.norm(np.asarray(c[k], np.float64) - b[k])
            assert d <= 4 * dc + 1e-6 * np.linalg.norm(b[k]), (k, d, dc)
    for m in (sw, ref, ctl):
        m.close()


def test_largest_batch_stays_finite():
    cfg, B = M.Config(1024, 2, True, True, True), 65536
    m, _ = fp16_model(cfg, seed=4)
    x, t = synth.mlp_inputs(B, seed=6)
    for s in range(2):
        loss, _, _, y = m.step(None, x, t, 0.5, isTraining=True)
        assert np.isfinite(float(loss)) and np.isfinite(y).all()
    assert all(np.isfinite(v).all() for v in m.get_gradients().values())
    assert all(np.isfinite(v).all() for v in m.get_variables().values())
    m.close()


# ---------------------------------------------------------------------------------------------- inference, refusals

@pytest.mark.parametrize("mode", ["bf16", "fp16"])
def test_inference_after_training_follows_the_mode(mode):
    """Trained on the fp16 route, served by the model's own inference mode: bit-identical to a model of that mode that
    was handed the trained variables."""
    from helpers import make_model
    cfg = M.Config(1024, 2, True, True, True)
    m, _ = fp16_model(cfg, seed=6, bn="fresh", mode=mode)
    for s in range(3):
        x, t = synth.mlp_inputs(512, seed=60 + s)
        m.step(None, x, t, 0.5, isTraining=True)
    trained = m.get_variables()
    fresh, _ = make_model(cfg, seed=6, mode=mode)
    fresh.set_variables(trained)
    for B in (8, 64, 4096, 6144):
        x = synth.mlp_inputs(B, seed=90 + B)[0]
        _, _, y = m.step(None, x, np.zeros((B, 48), np.float32), 1.0, isTraining=False)
        _, _, yf = fresh.step(None, x, np.zeros((B, 48), np.float32), 1.0, isTraining=False)
        assert np.array_equal(y, yf), (mode, B)
    m.close(); fresh.close()


def test_refusals():
    from p3d import LinearModel, _lib
    for mode in ("fp32", "bf16x3"):
        with pytest.raises(ValueError):
            LinearModel(256, 1, True, True, True, 64, 1e-3, mode=mode, train_matmul="fp16")
        m = LinearModel(256, 1, True, True, True, 64, 1e-3, mode=mode)
        for kind in (_lib.TRAIN_MATMUL_FP16, _lib.TRAIN_MATMUL_BF16):
            assert _lib.lib.p3d_model_set_train_matmul(m._handle, kind) == ERR_ARG, (mode, kind)
        m.close()
    for mode in ("bf16", "fp16"):
        m = LinearModel(256, 1, True, True, True, 64, 1e-3, mode=mode, train_matmul="fp16")
        assert m.train_matmul == "fp16"
        for kind in (_lib.TRAIN_MATMUL_DEFAULT, _lib.TRAIN_MATMUL_BF16X3, 7):
            assert _lib.lib.p3d_model_set_train_matmul(m._handle, kind) == ERR_ARG, (mode, kind)
        for kind in (_lib.TRAIN_MATMUL_BF16, _lib.TRAIN_MATMUL_FP16):
            assert _lib.lib.p3d_model_set_train_matmul(m._handle, kind) == 0, (mode, kind)
        m.close()
    with pytest.raises(ValueError):
        LinearModel(256, 1, True, True, True, 64, 1e-3, mode="bf16", train_matmul="fp8")


def test_ragged_width_keeps_the_ffma_route():
    """linear_size % 8 != 0: the route changes nothing (bit-identical to a model without the keyword)."""
    cfg, B = M.Config(100, 2, True, True, True), 64
    x, t = synth.mlp_inputs(B, seed=9)
    masks = (np.random.RandomState(2).uniform(size=(5, B, 100)) < 0.5).astype(np.uint8)
    outs = []
    for tm in ("fp16", None):
        m, _ = fp16_model(cfg, train_matmul=tm)
        m.step(None, x, t, 0.5, isTraining=True, dropout_mask=masks)
        outs.append((m.get_gradients(), m.get_variables(include_optimizer=True)))
        m.close()
    for a, b in zip(*outs):
        for k in b:
            assert np.array_equal(a[k], b[k]), k
