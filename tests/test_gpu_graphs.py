"""Inference inside CUDA graphs (include/p3d.h, "CUDA graphs"): LinearModel.step(isTraining=False) and
RealtimeLifter.step_batch with torch CUDA tensors, captured with torch.cuda.graph and replayed.

Every case warms up eagerly, captures, then replays three times with new inputs copied into the static input tensor,
and compares each replay with an eager call on the same inputs BIT FOR BIT.  The one exception is the MSE loss: its
sum of squares is accumulated with double-precision atomics from many blocks, in whatever order they arrive, so two
runs can differ in the last bits of the double (relative ~1e-13); after the cast to float32 that is at most one
float32 ulp, which is the tolerance used for it."""
import numpy as np
import pytest

from helpers import make_model
from oracle import geometry_ref as G, mlp_ref as M

pytestmark = pytest.mark.gpu

REPLAYS = 3


@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


def _model(width, mode="bf16", predict_14=False, seed=11):
    return make_model(M.Config(width, 2, True, True, True), seed=seed, mode=mode, predict_14=predict_14)[0]


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
    """PyTorch's convention: one eager call of the same shape on a side stream, then the capture."""
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


def _replay_matches_eager(torch, model, B, seed, with_target=False):
    g, xs, ts, loss, y = _warm_and_capture(torch, model, B, seed, with_target)
    for i in range(REPLAYS):
        xi = _x(torch, B, seed + 100 + i)
        xs.copy_(xi)
        ti = None
        if with_target:
            ti = _t(torch, B, model.output_size, seed + 100 + i)
            ts.copy_(ti)
        g.replay()
        got_y, got_loss = y.cpu().numpy(), loss.cpu().numpy()
        want_loss, want_y = _eager(model, xi.clone(), None if ti is None else ti.clone())
        assert np.array_equal(got_y, want_y), (B, i, np.abs(got_y - want_y).max())
        if with_target:
            assert _same_loss(got_loss, want_loss), (B, i, float(got_loss), float(want_loss))
            assert float(got_loss) > 0.0
    del g


# ---------------------------------------------------------------------------------------------- every dispatch path

@pytest.fixture(scope="module")
def models():
    cache = {}

    def get(width, mode="bf16", predict_14=False):
        key = (width, mode, predict_14)
        if key not in cache:
            cache[key] = _model(width, mode, predict_14)
        return cache[key]
    yield get
    for m in cache.values():
        m.close()


# bf16 width 1024: whole-chip kernel (1-8 poses), whole-chip mma.sync kernel (9-64), per-layer GEMMs (65-6143), fused
# persistent kernel (6144 and up)
@pytest.mark.parametrize("B", [1, 2, 5, 8, 9, 33, 64, 65, 300, 6143, 6144, 20000])
def test_dispatch_bf16_1024(torch, models, B):
    _replay_matches_eager(torch, models(1024), B, seed=B)


@pytest.mark.parametrize("B", [1, 4096])
def test_dispatch_bf16_256(torch, models, B):
    _replay_matches_eager(torch, models(256), B, seed=B)


@pytest.mark.parametrize("B", [3, 200])
def test_dispatch_bf16_width_100(torch, models, B):
    """linear_size % 8 != 0: the per-layer SIMT kernels (<= 16 poses) and the fp32 SGEMM chain."""
    _replay_matches_eager(torch, models(100), B, seed=B)


@pytest.mark.parametrize("B", [1, 3, 16])
def test_width_100_small_batch_eager_matches_oracle(B):
    """The per-layer SIMT kernel at a width that is not a multiple of 8 (ragged last group of 8 weights), checked
    eagerly against the fp64 oracle and against the restated kernel arithmetic (bf16 weights, fp32 activations)."""
    from helpers import emulate_bf16_forward, rowwise_rel
    cfg = M.Config(100, 2, True, True, True)
    model, p = make_model(cfg, seed=31)
    x = np.random.RandomState(B).normal(size=(B, 32)).astype(np.float32)
    _, _, y = model.step(None, x, None, 1.0, isTraining=False)
    ref = M.forward(p, x.astype(np.float64), cfg, training=False)
    assert rowwise_rel(y, ref).max() <= 1e-2                    # bf16 tolerance used by the other parity tests
    emu = emulate_bf16_forward(p, x, cfg, small_batch=True)
    assert rowwise_rel(y, emu).max() <= 2e-3
    model.close()


@pytest.mark.parametrize("B", [1, 64, 5000])
def test_dispatch_fp32_1024(torch, models, B):
    _replay_matches_eager(torch, models(1024, "fp32"), B, seed=B)


def test_dispatch_predict_14(torch, models):
    _replay_matches_eager(torch, models(1024, predict_14=True), 64, seed=14)


@pytest.mark.parametrize("B", [64, 300])
def test_captured_step_loss(torch, models, B):
    _replay_matches_eager(torch, models(1024), B, seed=500 + B, with_target=True)


# ---------------------------------------------------------------------------------------------- protocol and buffers

def test_interleaved_graphs_and_eager_calls(torch):
    """Graphs of the whole-chip kernels replayed back to back, then alternately with eager calls in between: every
    launch needs an exchange tag no earlier launch used.  Replaying one graph several times in a row, with no other
    launch of the same kernel in between, is where a tag frozen into the graph at capture would let consumers accept
    the previous replay's words."""
    model = _model(1024, seed=21)
    g64, x64, _, _, y64 = _warm_and_capture(torch, model, 64, seed=1)
    g5, x5, _, _, y5 = _warm_and_capture(torch, model, 5, seed=2)
    g1, x1, _, _, y1 = _warm_and_capture(torch, model, 1, seed=3)
    # back to back: each graph REPLAYS times in a row with a new input, outputs cloned, no eager call in between
    for g, xs, y, B, seed in ((g64, x64, y64, 64, 200), (g5, x5, y5, 5, 300), (g1, x1, y1, 1, 400)):
        inputs, outputs = [], []
        for i in range(REPLAYS):
            xi = _x(torch, B, seed + i)
            xs.copy_(xi)
            g.replay()
            inputs.append(xi)
            outputs.append(y.clone())
        for i, (xi, yi) in enumerate(zip(inputs, outputs)):
            assert np.array_equal(yi.cpu().numpy(), _eager(model, xi)[1]), (B, i)
    del g1
    # alternating with eager calls of other batch sizes
    for i in range(REPLAYS):
        a, b = _x(torch, 64, 10 + i), _x(torch, 5, 20 + i)
        x64.copy_(a)
        g64.replay()
        got64 = y64.clone()
        model.step(None, _x(torch, 7, 30 + i), None, 1.0, isTraining=False)
        x5.copy_(b)
        g5.replay()
        got5 = y5.clone()
        model.step(None, _x(torch, 64, 40 + i), None, 1.0, isTraining=False)
        assert np.array_equal(got64.cpu().numpy(), _eager(model, a)[1]), i
        assert np.array_equal(got5.cpu().numpy(), _eager(model, b)[1]), i
    del g64, g5
    model.close()


def test_scratch_stays_put(torch):
    """Graphs keep addressing the scratch they were captured with after eager calls have grown it."""
    model = _model(1024, seed=22)
    g300, x300, _, _, y300 = _warm_and_capture(torch, model, 300, seed=3)
    g9k, x9k, _, _, y9k = _warm_and_capture(torch, model, 9000, seed=4)
    model.step(None, _x(torch, 70000, 5), None, 1.0, isTraining=False)        # grows the packed input
    model.step(None, _x(torch, 2000, 6), None, 1.0, isTraining=False)         # grows the layered activations
    torch.cuda.synchronize()
    for i in range(REPLAYS):
        a, b = _x(torch, 300, 50 + i), _x(torch, 9000, 60 + i)
        x300.copy_(a)
        x9k.copy_(b)
        g300.replay()
        g9k.replay()
        assert np.array_equal(y300.cpu().numpy(), _eager(model, a)[1]), i
        assert np.array_equal(y9k.cpu().numpy(), _eager(model, b)[1]), i
    del g300, g9k
    model.close()


def _lifter(model, seed=3):
    from p3d.realtime import RealtimeLifter
    use2, _ = G.dims_to_use(2)
    use3, _ = G.dims_to_use(3)
    rs = np.random.RandomState(seed)
    mu2, sd2 = rs.uniform(300, 700, 64), rs.uniform(50, 150, 64)
    mu3, sd3 = rs.normal(0, 200, 96), rs.uniform(50, 150, 96)
    return RealtimeLifter(model, mu2, sd2, use2, mu3, sd3, use3)


def test_replay_ordered_before_host_calls(torch):
    """A replay shares the forward scratch with the host-buffer step and the realtime host frame, which run on
    private streams: both must start behind it, without the caller synchronising."""
    model = _model(1024, seed=23)
    lifter = _lifter(model)
    B = 65536
    g, xs, ts, loss, y = _warm_and_capture(torch, model, B, seed=7, with_target=True)
    rs = np.random.RandomState(8)
    xn = rs.normal(size=(B, 32)).astype(np.float32)
    tn = rs.normal(size=(B, 48)).astype(np.float32)
    kp = rs.uniform(100, 900, 36).tolist()
    _, _, y_host0 = model.step(None, xn, tn, 1.0, isTraining=False)             # warms the host pipeline
    lifter.step(kp)
    for i in range(REPLAYS):
        xi, ti = _x(torch, B, 70 + i), _t(torch, B, 48, 70 + i)
        xs.copy_(xi)
        ts.copy_(ti)
        torch.cuda.synchronize()
        g.replay()                                                              # no synchronise after this
        l_host, _, y_host = model.step(None, xn, tn, 1.0, isTraining=False)
        enc, yrt, pose = lifter.step(kp)
        got_y, got_loss = y.cpu().numpy(), loss.cpu().numpy()
        want_loss, want_y = _eager(model, xi, ti)
        assert np.array_equal(got_y, want_y), i
        assert _same_loss(got_loss, want_loss), i
        torch.cuda.synchronize()
        l_host2, _, y_host2 = model.step(None, xn, tn, 1.0, isTraining=False)
        enc2, yrt2, pose2 = lifter.step(kp)
        assert np.array_equal(y_host, y_host2) and np.array_equal(y_host, y_host0), i
        assert _same_loss(l_host, l_host2), i
        assert np.array_equal(enc, enc2) and np.array_equal(yrt, yrt2) and np.array_equal(pose, pose2), i
    del g
    lifter.close()
    model.close()


# ---------------------------------------------------------------------------------------------- weights

def test_new_weights_reach_a_captured_graph(torch):
    from p3d._lib import P3DError
    model = _model(1024, seed=24)
    g, xs, _, _, y = _warm_and_capture(torch, model, 64, seed=9)
    xi = _x(torch, 64, 90)
    xs.copy_(xi)
    g.replay()
    before = y.cpu().numpy()
    # set_variable -> prepare_inference -> replay
    rs = np.random.RandomState(5)
    model.set_variable("linear_model/w4", (rs.normal(size=(1024, 48)) * 0.01).astype(np.float32))
    model.prepare_inference()
    g.replay()
    after = y.cpu().numpy()
    assert not np.array_equal(after, before)
    assert np.array_equal(after, _eager(model, xi)[1])
    # one training step -> prepare_inference -> replay
    xt, tt = _x(torch, 64, 91), _t(torch, 64, 48, 91)
    model.step(None, xt, tt, 1.0, isTraining=True)
    model.prepare_inference()
    g.replay()
    trained = y.cpu().numpy()
    assert not np.array_equal(trained, after)
    assert np.array_equal(trained, _eager(model, xi)[1])
    # a capture while the fold is stale is refused instead of capturing the fold
    model.set_variable("linear_model/b4", np.zeros(48, dtype=np.float32))
    g2 = torch.cuda.CUDAGraph()
    with pytest.raises(P3DError, match="prepare_inference"):
        with torch.cuda.graph(g2):
            model.step(None, xs, None, 1.0, isTraining=False)
    del g2
    # ... and the eager path still folds by itself
    y_eager = _eager(model, xi)[1]
    model.prepare_inference()
    g.replay()
    assert np.array_equal(y.cpu().numpy(), y_eager)
    del g
    model.close()


# ---------------------------------------------------------------------------------------------- refusals

def test_refusals_then_eager_calls_work(torch):
    from p3d._lib import P3DError
    model = _model(1024, seed=25)
    _warm_and_capture(torch, model, 64, seed=11)          # a warm model, but never at 300 poses
    xs = _x(torch, 300, 12)
    g = torch.cuda.CUDAGraph()
    with pytest.raises(P3DError, match="warm up"):
        with torch.cuda.graph(g):
            model.step(None, xs, None, 1.0, isTraining=False)
    del g
    xt, tt = _x(torch, 64, 13), _t(torch, 64, 48, 13)
    g = torch.cuda.CUDAGraph()
    with pytest.raises(P3DError, match="train_step"):
        with torch.cuda.graph(g):
            model.step(None, xt, tt, 1.0, isTraining=True)
    del g
    # eager calls behave normally afterwards, and the warm-up makes the capture at 300 poses possible
    assert int(model.global_step) == 0
    _, ya = _eager(model, xs)
    _, yb = _eager(model, xs.clone())
    assert np.array_equal(ya, yb) and np.isfinite(ya).all()
    model.step(None, xt, tt, 1.0, isTraining=True)
    assert int(model.global_step) == 1
    _replay_matches_eager(torch, model, 300, seed=14)
    model.close()


# ---------------------------------------------------------------------------------------------- realtime batches

@pytest.mark.parametrize("B", [1, 300])
def test_realtime_step_batch(torch, B):
    model = _model(1024, seed=26)
    lifter = _lifter(model)

    def kp(seed):
        g = torch.Generator(device="cuda").manual_seed(seed)
        return torch.rand((B, 36), generator=g, device="cuda", dtype=torch.float64) * 800 + 100

    ks = kp(1)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        lifter.step_batch(ks)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        enc, y, pose = lifter.step_batch(ks)
    for i in range(REPLAYS):
        ki = kp(10 + i)
        ks.copy_(ki)
        g.replay()
        got = [t.cpu().numpy() for t in (enc, y, pose)]
        want = [t.cpu().numpy() for t in lifter.step_batch(ki.clone())]
        for a, b in zip(got, want):
            assert np.array_equal(a, b), i
    del g
    lifter.close()
    model.close()
