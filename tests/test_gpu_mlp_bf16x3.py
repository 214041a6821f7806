"""The bf16x3 inference mode (P3D_MODE_BF16X3, LinearModel(mode="bf16x3")): three split-bf16 tcgen05 products per
MatMul, fp32 activations.  Held to the fp32 contract against the fp64 oracle (row-wise 1e-4, loss 1e-4 relative), to
its own rounding points (tests/test_oracle_bf16x3.py) at 3e-5 row-wise, and to the golden fixture.  The emulation bound
is not 1e-5: both sides accumulate in fp32 in different orders, and in the trained-BN models without max_norm that
order alone moves outputs by 5e-6 row-wise between two CPU summation orders (measured on a B200 at 1000 W: up to 1.3e-5
between kernel and emulation); a wrong segment pair or a dropped product costs ~4e-3.  Also covered: every way the
mode is reached - host and device buffers, row chunks, CUDA graphs, weight refresh, training (the FFMA route of fp32
mode), the realtime lifter, PoseBase and evaluate_batches."""
import numpy as np
import pytest

from helpers import make_model, rowwise_rel
from oracle import geometry_ref as G, mlp_ref as M, synth
from test_gpu_mlp import CFGS
from test_oracle_bf16x3 import emulate_bf16x3_forward

pytestmark = pytest.mark.gpu

CHUNK = 32768           # rows per chunk of the bf16x3 forward (kSplitChunk, csrc/mlp_layered.cu)
REPLAYS = 3


def _cid(c):
    return f"L{c.linear_size}n{c.num_layers}r{int(c.residual)}b{int(c.batch_norm)}m{int(c.max_norm)}o{c.out_size}"


PARITY = CFGS + [
    M.Config(200, 2, True, True, True),        # ragged K: a multiple of 8, not of 64
    M.Config(100, 2, True, True, True),        # linear_size % 8 != 0: the FFMA fallback
    M.Config(4096, 4, True, True, True),
    M.Config(1024, 2, True, True, True, 42),   # predict_14
]


def _rows(B, L):
    """Rows the oracle is evaluated on: all of a small batch, otherwise the first and last 128, every row within 2 of a
    chunk boundary and a seeded sample (rows are independent at inference)."""
    if B * L <= 6500 * 1024:
        return np.arange(B)
    near = np.array([r for c in range(CHUNK, B, CHUNK) for r in range(c - 2, c + 2) if r < B], dtype=np.int64)
    pick = np.random.RandomState(B).choice(B, 256, replace=False)
    return np.unique(np.concatenate([np.arange(128), np.arange(B - 128, B), near, pick]))


@pytest.mark.parametrize("cfg", PARITY, ids=_cid)
def test_matches_oracle_and_emulation(cfg):
    m, p = make_model(cfg, seed=11, bn="trained", mode="bf16x3", predict_14=(cfg.out_size == 42))
    sizes = [1, 7, 64, 65, 333, 6500]
    if cfg.linear_size == 1024 and cfg.num_layers == 2 and cfg.max_norm and cfg.out_size == 48:
        sizes += [CHUNK - 1, CHUNK, CHUNK + 1]
    for B in sizes:
        x, t = synth.mlp_inputs(B, out_size=cfg.out_size, seed=B)
        loss, _, y = m.step(None, x, t, 1.0, isTraining=False)
        assert y.shape == (B, cfg.out_size) and y.dtype == np.float32
        rows = _rows(B, cfg.linear_size)
        x64 = x[rows].astype(np.float64)
        ref = M.forward(p, x64, cfg, training=False)
        rel = rowwise_rel(y[rows], ref)
        assert rel.max() <= 1e-4, (B, rel.max())
        if cfg.linear_size % 8 == 0:                     # the split GEMMs (the fallback is the FFMA chain)
            emu = emulate_bf16x3_forward(p, x64, cfg)
            assert rowwise_rel(y[rows], emu).max() <= 3e-5, (B, rowwise_rel(y[rows], emu).max())
        if len(rows) == B:
            want = M.loss_fn(ref, t.astype(np.float64))
            assert abs(float(loss) - want) <= 1e-4 * want, (B, float(loss), want)
    m.close()


# ---------------------------------------------------------------------------------------------- golden fixture

@pytest.mark.parametrize("tag", ["s_res_bn_mn", "s_res_bn", "s_bn_mn_1", "s_res_3", "s_mn", "s_p14", "s_fresh",
                                 "h_1024_b64", "h_1024_b64_nomn", "h_1024_b4096"])
def test_inference_matches_reference_graph(tag):
    import test_gpu_mlp_golden as GG
    z = np.load(GG.GOLD)
    cfg, p, x, t, B, steps, big, lr0 = GG.case_setup(z, tag)
    m = GG.model_for(cfg, p, B, lr0, "bf16x3")
    loss, _, y = m.step(None, x, t, 1.0, isTraining=False)
    m.close()
    ref, got = GG.fetch(z, tag + "/eval_y", y)
    assert y.dtype == np.float32 and y.shape == (B, cfg.out_size)
    assert GG.rowrel(got, ref) <= 1e-4, (tag, GG.rowrel(got, ref))
    if tag + "/eval_y@norm" in z.files:
        nrm = float(z[tag + "/eval_y@norm"])
        assert abs(np.linalg.norm(y.astype(np.float64)) - nrm) <= 1e-4 * nrm, tag
    assert abs(float(loss) - float(z[tag + "/eval_loss"])) <= 1e-4 * float(z[tag + "/eval_loss"])


@pytest.mark.parametrize("tag", ["s_res_bn_mn", "s_p14", "h_1024_b64", "h_1024_b4096"])
def test_training_steps_match_reference_graph(tag, monkeypatch):
    """Training steps of a bf16x3 model are those of fp32 mode: the fp32-mode golden check, run on a bf16x3 model
    (losses, outputs, learning rates, gradients, final variables, and an inference pass on them)."""
    import test_gpu_mlp_golden as GG
    plain = GG.model_for
    monkeypatch.setattr(GG, "model_for", lambda cfg, p, B, lr0, mode: plain(cfg, p, B, lr0, "bf16x3"))
    GG.test_fp32_training_steps_match_reference_graph(np.load(GG.GOLD), tag)


# ---------------------------------------------------------------------------------------------- large batches, paths

@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


@pytest.fixture(scope="module")
def model1024():
    m, p = make_model(M.Config(1024, 2, True, True, True), seed=7, mode="bf16x3")
    yield m, p
    m.close()


def test_large_batch_deterministic_and_row_independent(torch, model1024):
    m, _ = model1024
    B = 1 << 20
    small, _ = synth.mlp_inputs(6300, seed=3)
    fixed = np.concatenate([np.arange(100), np.arange(B - 100, B), np.arange(CHUNK - 50, CHUNK + 50)])
    pos = np.concatenate([fixed, np.random.RandomState(4).choice(np.setdiff1d(np.arange(B), fixed), 6000, replace=False)])
    big = synth.mlp_inputs(B, seed=5)[0]
    big[pos] = small
    xb = torch.from_numpy(big).cuda()
    y1 = m.step(None, xb, None, 1.0, isTraining=False)[2].cpu().numpy()
    y2 = m.step(None, xb, None, 1.0, isTraining=False)[2].cpu().numpy()
    assert np.array_equal(y1, y2)
    ys = m.step(None, torch.from_numpy(small).cuda(), None, 1.0, isTraining=False)[2].cpu().numpy()
    assert rowwise_rel(y1[pos], ys.astype(np.float64)).max() <= 1e-6


def test_host_and_device_paths_agree(torch, model1024):
    m, _ = model1024
    x, t = synth.mlp_inputs(200000, seed=6)
    loss_h, _, y_h = m.step(None, x, t, 1.0, isTraining=False)           # host pipeline
    loss_d, _, y_d = m.step(None, torch.from_numpy(x).cuda(), torch.from_numpy(t).cuda(), 1.0, isTraining=False)
    assert np.array_equal(y_h, y_d.cpu().numpy())
    assert abs(float(loss_h) - float(loss_d)) <= 1e-6 * float(loss_h)


# ---------------------------------------------------------------------------------------------- CUDA graphs
# the capture helpers of tests/test_gpu_graphs.py

def _x(torch, B, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn((B, 32), generator=g, device="cuda", dtype=torch.float32)


def _t(torch, B, out, seed):
    g = torch.Generator(device="cuda").manual_seed(seed + 7777)
    return torch.randn((B, out), generator=g, device="cuda", dtype=torch.float32)


def _eager(model, x, t=None):
    loss, _, y = model.step(None, x, t, 1.0, isTraining=False)
    return loss.cpu().numpy(), y.cpu().numpy()


def _warm_and_capture(torch, model, B, seed, with_target=False):
    xs = _x(torch, B, seed)
    ts = _t(torch, B, model.output_size, seed) if with_target else None
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        model.step(None, xs, ts, 1.0, isTraining=False)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        loss, _, y = model.step(None, xs, ts, 1.0, isTraining=False)
    return g, xs, ts, loss, y


def _same_loss(a, b):
    a, b = np.float32(a), np.float32(b)
    return abs(float(a) - float(b)) <= float(np.spacing(np.abs(b)))


@pytest.mark.parametrize("with_target", [False, True], ids=["y", "y+loss"])
@pytest.mark.parametrize("B", [1, 64, 4096, CHUNK + 1])
def test_graph_replays_equal_eager(torch, model1024, B, with_target):
    m, _ = model1024
    g, xs, ts, loss, y = _warm_and_capture(torch, m, B, B, with_target)
    for i in range(REPLAYS):
        xi = _x(torch, B, B + 100 + i)
        xs.copy_(xi)
        ti = None
        if with_target:
            ti = _t(torch, B, 48, B + 100 + i)
            ts.copy_(ti)
        g.replay()
        got_y, got_loss = y.cpu().numpy(), loss.cpu().numpy()
        want_loss, want_y = _eager(m, xi.clone(), None if ti is None else ti.clone())
        assert np.array_equal(got_y, want_y), (B, i)
        if with_target:
            assert _same_loss(got_loss, want_loss), (B, i)
    del g


def test_capture_before_warm_up_is_refused(torch):
    from p3d._lib import P3DError
    m, _ = make_model(M.Config(1024, 2, True, True, True), seed=8, mode="bf16x3")
    xs = _x(torch, 300, 1)
    for expect in ("prepare_inference", "warm up"):     # stale fold, then scratch that does not exist yet
        g = torch.cuda.CUDAGraph()
        with pytest.raises(P3DError, match=expect):
            with torch.cuda.graph(g):
                m.step(None, xs, None, 1.0, isTraining=False)
        del g
        m.prepare_inference()
    _, ya = _eager(m, xs)
    assert np.isfinite(ya).all()
    m.close()


def test_new_weights_reach_eager_calls_and_graphs(torch):
    m, p = make_model(M.Config(1024, 2, True, True, True), seed=9, mode="bf16x3")
    cfg = M.Config(1024, 2, True, True, True)
    x = synth.mlp_inputs(64, seed=2)[0]
    y0 = m.step(None, x, None, 1.0, isTraining=False)[2]
    w4 = (np.random.RandomState(5).normal(size=(1024, 48)) * 0.01).astype(np.float32)
    m.set_variable("linear_model/w4", w4)                                # set_variable -> step
    y1 = m.step(None, x, None, 1.0, isTraining=False)[2]
    p2 = dict(p, **{"linear_model/w4": w4.astype(np.float64)})
    assert not np.array_equal(y0, y1)
    assert rowwise_rel(y1, M.forward(p2, x.astype(np.float64), cfg)).max() <= 1e-4
    g, xs, _, _, y = _warm_and_capture(torch, m, 64, seed=3)             # set_variable -> prepare_inference -> replay
    before = y.cpu().numpy()
    m.set_variable("linear_model/b4", np.full(48, 0.5, np.float32))
    m.prepare_inference()
    g.replay()
    after = y.cpu().numpy()
    assert not np.array_equal(after, before)
    assert np.array_equal(after, _eager(m, xs)[1])
    del g
    m.close()


# ---------------------------------------------------------------------------------------------- the public surface

def test_realtime_lifter(golden_dir):
    """The staged realtime route on a bf16x3 model, held to what fp32 mode is held to."""
    import os
    from p3d.realtime import RealtimeLifter, keypoints_to_xy
    gold = np.load(os.path.join(golden_dir, "realtime.npz"))
    cfg = M.Config(1024, 2, True, True, True)
    model, p = make_model(cfg, seed=3, mode="bf16x3")
    lifter = RealtimeLifter(model, gold["mean2d"], gold["std2d"], gold["use2d"], gold["mean3d"], gold["std3d"], gold["use3d"])
    m3, s3, ig3 = gold["mean3d"], gold["std3d"], gold["ignore3d"]
    for case in ["coco54", "tfpose36", "body25_75", "wide_87"]:
        for f in range(3):
            enc, y, pose = lifter.step(keypoints_to_xy(gold["%s_kp%d" % (case, f)].tolist()))
            assert np.array_equal(enc, gold["%s_enc%d" % (case, f)].astype(np.float32))
            ref = M.forward(p, enc.astype(np.float64), cfg, training=False)
            assert rowwise_rel(y, ref).max() <= 1e-4
            assert np.abs(pose - G.unnormalize(ref.astype(np.float32), m3, s3, ig3)).max() < 0.05
    kp = np.random.RandomState(1).uniform(50, 950, size=(300, 36))
    enc, y, pose = lifter.step_batch(kp)
    assert rowwise_rel(y, M.forward(p, enc.astype(np.float64), cfg, training=False)).max() <= 1e-4
    lifter.close()
    model.close()


def test_posebase_and_evaluate_batches():
    from p3d import evaluate
    from p3d.linear_model import PoseBase
    cfg = M.Config(1024, 2, True, True, True)
    p = {k: v.astype(np.float32) for k, v in M.init_params(1024, 2, seed=8, bn="trained").items()}
    p64 = {k: v.astype(np.float64) for k, v in p.items()}
    pb = PoseBase(units=1024, input_size=32, output_size=48, seed=1, mode="bf16x3")
    pb.load_weights(p)
    x = np.random.RandomState(0).normal(size=(33, 32))
    y = pb(x, training=False)
    assert rowwise_rel(y, M.forward(p64, x.astype(np.float32).astype(np.float64), cfg, training=False)).max() <= 1e-4
    pb.close()
    model, _ = make_model(cfg, seed=4, mode="bf16x3", batch_size=64)
    use3, ign3 = G.dims_to_use(3)
    use2, ign2 = G.dims_to_use(2)
    rng = np.random.RandomState(8)
    mean3, std3 = rng.normal(0, 50, 96), rng.uniform(50, 200, 96)
    mean3[:3] = 0
    mean2, std2 = rng.uniform(300, 700, 64), rng.uniform(50, 150, 64)
    enc = [rng.normal(size=(64, 32)) for _ in range(3)]
    dec = [0.3 * rng.normal(size=(64, 48)) for _ in range(3)]
    tot, joint, _, loss = evaluate.evaluate_batches(None, model, mean3, std3, use3, ign3, mean2, std2, use2, ign2, 0, enc, dec)
    ref_d = np.vstack([G.mpjpe(model.step(None, e, d, 1.0, isTraining=False)[2], d.astype(np.float32), mean3, std3, ign3, use3)
                       for e, d in zip(enc, dec)])
    assert abs(tot - ref_d.mean()) < 1e-3 and np.abs(joint - ref_d.mean(0)).max() < 1e-3
    model.close()
