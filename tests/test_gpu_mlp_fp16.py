"""The fp16 inference mode (P3D_MODE_FP16, LinearModel(mode="fp16")): bf16 mode's kernels on fp16 operands, the same
rounding points, fp32 accumulation.  Held to its contract (2e-3 row-wise against the fp64 oracle) and, through
assert_matches_emulation with the oracle as `ref`, to the accuracy of its own NumPy emulation
(test_oracle_fp16.emulate_fp16_forward: helpers.emulate_bf16_forward with fp16 rounding): a single stray bf16 rounding costs ~8x
and fails.  Every case proves which kernel ran: the fused kernel records p3d_profile events, the whole-chip kernels
are one launch, the layered path 1 + layers (input pack + one GEMM per layer).  Training takes the bf16 route and is
checked against a bf16 model."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from helpers import assert_matches_emulation, make_model, rowwise_rel
from oracle import geometry_ref as G, mlp_ref as M, synth
from test_gpu_mlp_widths import multi_round_batch, sample_rows
from test_oracle_fp16 import emulate_fp16_forward

pytestmark = pytest.mark.gpu
CONTRACT = 2e-3
ERR_ARG = -1            # P3D_ERR_ARG
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _cid(c):
    return f"L{c.linear_size}n{c.num_layers}r{int(c.residual)}b{int(c.batch_norm)}m{int(c.max_norm)}o{c.out_size}"


def run(m, x):
    """One p3d_model_forward of x (host rows, uploaded first); returns (y, fused-kernel launches, kernel launches)."""
    from p3d import _lib
    xd = torch.from_numpy(np.ascontiguousarray(x, np.float32)).cuda()
    y = torch.empty((xd.shape[0], m.output_size), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    ms, n = C.c_double(), C.c_int64()
    _lib.check(_lib.lib.p3d_profile_enable(1))
    try:
        l0 = _lib.lib.p3d_launch_count()
        _lib.check(_lib.lib.p3d_model_forward(m._handle, xd.data_ptr(), y.data_ptr(), xd.shape[0], _lib.current_stream()))
        launches = _lib.lib.p3d_launch_count() - l0
        _lib.check(_lib.lib.p3d_profile_read(C.byref(ms), C.byref(n)))
    finally:
        _lib.lib.p3d_profile_enable(0)
    return y.cpu().numpy(), n.value, launches


def expect_path(cfg, B, fused, launches):
    nl = 2 * cfg.num_layers + 2
    L = cfg.linear_size
    if L % 8:
        assert fused == 0
    elif L == 1024 and B <= 64:
        assert (fused, launches) == (0, 1), (B, fused, launches)              # whole-chip kernel
    elif L % 256 == 0 and B >= 6144:
        assert fused == 1, (B, fused)                                          # fused persistent kernel
    else:
        assert (fused, launches) == (0, 1 + nl), (B, fused, launches)         # layered: pack + one GEMM per layer


def check(y, x, p, cfg, B, tol=CONTRACT):
    """Kernel rows against the oracle (the contract) and the fp16 emulation; returns the oracle rows."""
    x64 = np.asarray(x, np.float64)
    ref = M.forward(p, x64, cfg, training=False)
    assert np.isfinite(y).all()
    rel = rowwise_rel(y, ref).max()
    assert rel <= tol, (B, rel)
    if cfg.linear_size % 8 == 0:
        small = cfg.linear_size == 1024 and B <= 8                             # fp32 activations, fp16 weights
        emu = emulate_fp16_forward(p, x, cfg, small_batch=small)
        assert_matches_emulation(y, emu, np.sqrt(np.mean(ref ** 2)), ref)
    return ref


@pytest.fixture(scope="module")
def models():
    made = {}

    def get(cfg, mode="fp16", seed=None):
        key = (_cid(cfg), mode, seed)
        if key not in made:
            made[key] = make_model(cfg, seed=seed or cfg.linear_size + cfg.num_layers, bn="trained", mode=mode,
                                   predict_14=(cfg.out_size == 42))
        return made[key]
    yield get
    for m, _ in made.values():
        m.close()


# ---------------------------------------------------------------------------------------------- every dispatch path

CFGS = [M.Config(1024, 2, True, True, True), M.Config(1024, 2, True, True, False), M.Config(1024, 2, False, False, False),
        M.Config(1024, 2, True, True, True, 42)]
BATCHES = [1, 2, 8, 9, 16, 17, 32, 33, 64, 65, 4096, 6144, "multi_round"]


@pytest.mark.parametrize("B", BATCHES, ids=str)
@pytest.mark.parametrize("cfg", CFGS, ids=_cid)
def test_every_path_width_1024(models, cfg, B):
    m, p = models(cfg)
    B = multi_round_batch() if B == "multi_round" else B
    x = synth.mlp_inputs(B, out_size=cfg.out_size, seed=B)[0]
    run(m, x[:1])                                                              # the fold happens outside the count
    y, fused, launches = run(m, x)
    expect_path(cfg, B, fused, launches)
    rows = sample_rows(B, 4096, B) if B > 6144 else np.arange(B)
    check(y[rows], x[rows], p, cfg, B)


WIDTHS = [(M.Config(256, 2, True, True, True), [6144]), (M.Config(4096, 4, True, True, True), [6144]),
          (M.Config(200, 2, True, True, True), [1, 64, 65, 6144]), (M.Config(520, 2, True, True, False), [9, 65, 6144]),
          (M.Config(100, 2, True, True, True), [1, 65, 6144])]


@pytest.mark.parametrize("cfg,sizes", WIDTHS, ids=[_cid(c) for c, _ in WIDTHS])
def test_widths(models, cfg, sizes):
    """256 and 4096 x 4 blocks: the fused kernel; 200 and 520: the layered path at every batch; 100: the FFMA chain,
    which meets the fp32 contract."""
    m, p = models(cfg)
    for B in sizes:
        x = synth.mlp_inputs(B, out_size=cfg.out_size, seed=B + 1)[0]
        run(m, x[:1])
        y, fused, launches = run(m, x)
        expect_path(cfg, B, fused, launches)
        rows = sample_rows(B, cfg.linear_size, B)
        check(y[rows], x[rows], p, cfg, B, tol=1e-4 if cfg.linear_size % 8 else CONTRACT)


def test_fp16_error_is_a_quarter_of_bf16(models):
    """The feature's claim on the GPU: the same model and rows, fp16 error <= 1/4 of bf16 error at q50 and q99, on the
    whole-chip, layered and fused paths (trained BN, no max_norm: the case where bf16 error is largest)."""
    cfg = M.Config(1024, 2, True, True, False)
    m16, p = models(cfg, "fp16", seed=5)
    mb, _ = models(cfg, "bf16", seed=5)
    for B in (8, 64, 4096, 6144):
        x = synth.mlp_inputs(B, seed=300 + B)[0]
        ref = M.forward(p, x.astype(np.float64), cfg, training=False)
        e16 = np.abs(run(m16, x)[0] - ref)
        eb = np.abs(run(mb, x)[0] - ref)
        for q in (0.5, 0.99):
            assert np.quantile(e16, q) <= 0.25 * np.quantile(eb, q), (B, q, np.quantile(e16, q), np.quantile(eb, q))


def test_fused_kernel_single_cta_tiles():
    """P3D_TC_CG=1 (read once per process): the single-CTA form of the fused kernel, in a process of its own."""
    code = (
        "import numpy as np, test_gpu_mlp_fp16 as T\n"
        "from helpers import make_model\n"
        "from oracle import mlp_ref as M, synth\n"
        "cfg = M.Config(1024, 2, True, True, True)\n"
        "m, p = make_model(cfg, seed=9, mode='fp16')\n"
        "x = synth.mlp_inputs(6144, seed=9)[0]\n"
        "T.run(m, x[:1]); y, fused, launches = T.run(m, x)\n"
        "assert fused == 1, fused\n"
        "T.check(y, x, p, cfg, 6144)\n"
        "m.close(); print('ok')\n")
    env = dict(os.environ, P3D_TC_CG="1")
    env["PYTHONPATH"] = os.pathsep.join([os.path.join(ROOT, "tests"), ROOT, os.path.join(ROOT, "3d-pose-baseline_b200")])
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


# ---------------------------------------------------------------------------------------------- golden fixture

@pytest.mark.parametrize("tag", ["s_res_bn_mn", "s_res_bn", "s_bn_mn_1", "s_res_3", "s_mn", "s_p14", "s_fresh",
                                 "h_1024_b64", "h_1024_b64_nomn", "h_1024_b4096"])
def test_inference_matches_reference_graph(tag):
    import test_gpu_mlp_golden as GG
    z = np.load(GG.GOLD)
    cfg, p, x, t, B, steps, big, lr0 = GG.case_setup(z, tag)
    m = GG.model_for(cfg, p, B, lr0, "fp16")
    loss, _, y = m.step(None, x, t, 1.0, isTraining=False)
    m.close()
    ref, got = GG.fetch(z, tag + "/eval_y", y)
    assert GG.rowrel(got, ref) <= CONTRACT, GG.rowrel(got, ref)
    gl = float(z[tag + "/eval_loss"])
    assert abs(float(loss) - gl) <= CONTRACT * gl, (float(loss), gl)


# ---------------------------------------------------------------------------------------------- training

def _variables(m):
    return m.get_variables(include_optimizer=True)


@pytest.mark.parametrize("cfg", [M.Config(1024, 2, True, True, True), M.Config(200, 1, True, True, False)], ids=_cid)
def test_training_is_the_bf16_route(cfg):
    """Same variables, seed and Philox masks: an fp16 model trains like a bf16 model.  The first steps give identical
    losses and outputs.  Two bf16 models do not stay bit-identical themselves (the weight-gradient GEMMs sum split-K
    partials with fp32 atomics, so the last bits of an update depend on arrival order, and over an epoch with dropout
    and Adam those bits grow), so a second bf16 model is the control: wherever it matches the first bit for bit, the
    fp16 model must too, and elsewhere the fp16 model may differ from the first bf16 model by no more than about what
    the control does.  Inference on the trained weights then meets the fp16 contract."""
    m16, p = make_model(cfg, seed=41, bn="trained", mode="fp16")
    mb, _ = make_model(cfg, seed=41, bn="trained", mode="bf16")
    mc, _ = make_model(cfg, seed=41, bn="trained", mode="bf16")
    for s in range(3):
        x, t = synth.mlp_inputs(256, seed=60 + s)
        a, b, _ = (m.step(None, x, t, 0.5, isTraining=True) for m in (m16, mb, mc))
        assert np.array_equal(np.asarray(a[0]), np.asarray(b[0])) and np.array_equal(a[-1], b[-1]), s
    X, T = synth.mlp_inputs(2048, seed=70)
    perm = np.random.RandomState(3).permutation(2048)
    (la, lra), (lb, lrb), (lc, _) = (m.train_epoch(X, T, 0.5, perm=perm) for m in (m16, mb, mc))
    assert lra == lrb

    def like_control(got, want, control, name):
        got, want, control = (np.asarray(v, np.float64) for v in (got, want, control))
        if np.array_equal(control, want):
            assert np.array_equal(got, want), name
        else:
            d, dc = np.linalg.norm(got - want), np.linalg.norm(control - want)
            assert d <= 4 * dc + 1e-6 * np.linalg.norm(want), (name, d, dc)
    like_control(la, lb, lc, "epoch losses")
    va, vb, vc = _variables(m16), _variables(mb), _variables(mc)
    assert va.keys() == vb.keys()
    for k in vb:
        like_control(va[k], vb[k], vc[k], k)
    trained = {k: v.astype(np.float64) for k, v in m16.get_variables().items()}
    for B in (8, 64, 4096):
        x = synth.mlp_inputs(B, seed=80 + B)[0]
        y, _, _ = run(m16, x)
        check(y, x, trained, cfg, B)
    for m in (m16, mb, mc):
        m.close()


def test_refusals():
    from p3d import LinearModel, _lib
    cfg = M.Config(1024, 2, True, True, True)
    with pytest.raises(ValueError):
        LinearModel(1024, 2, True, True, True, 64, 1e-3, mode="fp16", train_matmul="bf16x3")
    m, _ = make_model(cfg, mode="fp16")
    assert _lib.lib.p3d_model_set_train_matmul(m._handle, _lib.TRAIN_MATMUL_BF16X3) == ERR_ARG
    m.close()
    c = _lib.Cfg(1024, 2, 1, 1, 1, 0, 4, 0, 1e-3)
    h = C.c_void_p()
    assert _lib.lib.p3d_model_create(C.byref(c), C.byref(h)) == ERR_ARG
    assert b"unknown mode 4" in _lib.lib.p3d_last_error()


# ---------------------------------------------------------------------------------------------- graphs and host paths

@pytest.mark.parametrize("width,B", [(1024, 1), (1024, 8), (1024, 64), (1024, 4096), (1024, 6144), (200, 300), (100, 8)])
def test_graph_replays_equal_eager_calls(models, width, B):
    from test_gpu_graphs import _replay_matches_eager
    m, _ = models(M.Config(width, 2, True, True, True))
    _replay_matches_eager(torch, m, B, seed=B, with_target=True)


def test_prepare_inference_refreshes_captured_graphs(models):
    m, p = models(M.Config(1024, 2, True, True, True), seed=77)
    x = torch.from_numpy(synth.mlp_inputs(64, seed=1)[0]).cuda()
    m.step(None, x, None, 1.0, isTraining=False)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        _, _, y = m.step(None, x, None, 1.0, isTraining=False)
    b4 = np.full(48, 0.25, np.float32)
    m.set_variable("linear_model/b4", b4)
    m.prepare_inference()
    g.replay()
    p2 = dict(p, **{"linear_model/b4": b4.astype(np.float64)})
    check(y.cpu().numpy(), x.cpu().numpy(), p2, M.Config(1024, 2, True, True, True), 64)
    del g


@pytest.mark.parametrize("B", [1, 64, 4096, 6144])
def test_host_step_equals_device_path(models, B):
    """One pipeline chunk of the host-buffer step runs the kernel a device call of the same batch runs."""
    m, _ = models(M.Config(1024, 2, True, True, True))
    x, t = synth.mlp_inputs(B, seed=4)
    lh, _, yh = m.step(None, x, t, 1.0, isTraining=False)
    ld, _, yd = m.step(None, torch.from_numpy(x).cuda(), torch.from_numpy(t).cuda(), 1.0, isTraining=False)
    assert np.array_equal(yh, yd.cpu().numpy())
    assert abs(float(lh) - float(ld.cpu())) <= 1e-6 * float(lh)


# ---------------------------------------------------------------------------------------------- realtime

def test_realtime_frame(golden_dir):
    """A width-1024 frame is ONE launch (the 16-CTA cluster kernel on fp16 weights), bit exact around the lifter,
    within the contract and the weights-only emulation, < 0.5 mm after un-normalisation, equal to model.step."""
    from p3d import _lib
    from p3d.realtime import keypoints_to_xy
    from test_gpu_realtime import CASES, _lifter
    gold = np.load(os.path.join(golden_dir, "realtime.npz"))
    cfg = M.Config(1024, 2, True, True, True)
    model, p = make_model(cfg, seed=3, mode="fp16")
    lifter = _lifter(model, gold)
    m3, s3, ig3 = gold["mean3d"], gold["std3d"], gold["ignore3d"]
    lifter.step(keypoints_to_xy(gold["coco54_kp0"].tolist()))                # fold outside the count
    for case in CASES:
        for f in range(3):
            xy = keypoints_to_xy(gold["%s_kp%d" % (case, f)].tolist())
            l0 = _lib.lib.p3d_launch_count()
            enc, y, pose = lifter.step(xy)
            assert _lib.lib.p3d_launch_count() - l0 == 1
            assert np.array_equal(enc, gold["%s_enc%d" % (case, f)].astype(np.float32))
            assert np.array_equal(pose, G.unnormalize(y, m3, s3, ig3))
            ref = M.forward(p, enc.astype(np.float64), cfg, training=False)
            assert rowwise_rel(y, ref).max() <= CONTRACT
            emu = emulate_fp16_forward(p, enc, cfg, small_batch=True)
            assert rowwise_rel(y, emu).max() <= 3e-4
            assert np.abs(pose - G.unnormalize(ref.astype(np.float32), m3, s3, ig3)).max() < 0.5
            _, _, y2 = model.step(None, enc, np.zeros((1, 48)), 1.0, isTraining=False)
            assert np.array_equal(y, y2)
    lifter.close()
    model.close()
