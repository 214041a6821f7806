"""Parity of the CUDA LinearModel inference (tcgen05 bf16 path, fp32 path, small-batch path) with the
fp64 oracle (oracle/mlp_ref.py) on identical synthetic inputs and random-init weights.
All calls go through the Python mirror -> ctypes -> C ABI (libp3d.so).

Tolerances (BASELINE.json north_star): bf16 mode row-wise ||y-ref||2/||ref||2 <= 1e-2 ;
fp32 mode <= 1e-4.  In addition the bf16 kernels are held to a NumPy emulation of their own
rounding points (bf16 weights/activations, wide accumulation) at 2e-3 of the output rms - that
catches wrong tiles/columns/residuals that a loose relative bound could hide."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from oracle import mlp_ref as M
from oracle import synth
from helpers import assert_matches_emulation, bf16_round, emulate_bf16_forward, make_model, rowwise_rel

pytestmark = pytest.mark.gpu


def _bf16_bits(a):
    return (bf16_round(a).view(np.uint32) >> 16).astype(np.uint16)


@pytest.mark.parametrize("N,K", [(256, 64), (256, 128), (256, 1024), (48, 1024), (16, 64), (128, 256)])
def test_umma_gemm_selftest(N, K):
    """One-CTA TMA -> tcgen05.mma -> TMEM -> tcgen05.ld round trip against NumPy."""
    from p3d import _lib
    rng = np.random.RandomState(N + K)
    A = rng.standard_normal((128, K)).astype(np.float32)
    W = rng.standard_normal((N, K)).astype(np.float32)
    Ad = torch.from_numpy(_bf16_bits(A).view(np.int16)).cuda()
    Wd = torch.from_numpy(_bf16_bits(W).view(np.int16)).cuda()
    Cd = torch.zeros((128, N), dtype=torch.float32, device="cuda")
    _lib.check(_lib.lib.p3d_debug_umma_gemm(Ad.data_ptr(), Wd.data_ptr(), Cd.data_ptr(), N, K, None))
    torch.cuda.synchronize()
    ref = bf16_round(A).astype(np.float64) @ bf16_round(W).astype(np.float64).T
    got = Cd.cpu().numpy()
    assert np.abs(got - ref).max() <= 1e-4 * max(1.0, np.abs(ref).max()), np.abs(got - ref).max()


CFGS = [
    # linear_size, num_layers, residual, batch_norm, max_norm
    M.Config(1024, 2, True, True, True),
    M.Config(1024, 2, True, True, False),
    M.Config(256, 1, True, True, False),
    M.Config(512, 2, False, True, True),
    M.Config(256, 0, True, False, False),
    M.Config(1024, 1, True, False, False),
    M.Config(256, 3, True, True, False),
]


@pytest.mark.parametrize("cfg", CFGS, ids=lambda c: f"L{c.linear_size}n{c.num_layers}r{int(c.residual)}b{int(c.batch_norm)}m{int(c.max_norm)}")
@pytest.mark.parametrize("B", [128, 333, 1000, 6500])
def test_bf16_forward_matches_oracle(cfg, B):
    m, p = make_model(cfg, seed=11, bn="trained", mode="bf16")
    x, t = synth.mlp_inputs(B, seed=B)
    loss, _, y = m.step(None, x, t, 1.0, isTraining=False)
    ref = M.forward(p, x.astype(np.float64), cfg, training=False)
    emu = emulate_bf16_forward(p, x, cfg)
    assert y.shape == (B, 48) and y.dtype == np.float32
    rms = np.sqrt(np.mean(ref ** 2))
    assert_matches_emulation(y, emu, rms, ref)
    rel = rowwise_rel(y, ref)
    assert rel.max() <= 1e-2, rel.max()
    assert abs(float(loss) - M.loss_fn(y.astype(np.float64), t.astype(np.float64))) <= 1e-4 * max(1.0, float(loss))
    m.close()


@pytest.mark.parametrize("B", [1, 2, 3, 7, 8, 9, 10, 16, 17, 31, 32, 33, 48, 63, 64, 65, 127, 129, 4097, 6143, 6144, 6145, 7000])
def test_bf16_forward_ragged_batches(B):
    """Any B is accepted (placeholders [None,32], linear_model.py:96-97): the whole-chip latency kernel (B <= 8,
    fp32 activations), the whole-chip mma.sync kernel (9 <= B <= 64 when enabled: one or two row groups of 16 / 32
    poses, ragged last group), the layered per-layer GEMM path (up to 6143: partial tiles, tile+1 row) and the fused
    persistent kernel (B >= 6144), either side of the crossovers."""
    cfg = M.Config(1024, 2, True, True, True)
    m, p = make_model(cfg, seed=3, bn="trained", mode="bf16")
    x, t = synth.mlp_inputs(B, seed=100 + B)
    _, _, y = m.step(None, x, t, 1.0, isTraining=False)
    ref = M.forward(p, x.astype(np.float64), cfg, training=False)
    emu = emulate_bf16_forward(p, x, cfg, small_batch=(B <= 8))
    rms = np.sqrt(np.mean(ref ** 2))
    assert_matches_emulation(y, emu, rms, ref)
    assert rowwise_rel(y, ref).max() <= 1e-2
    m.close()


@pytest.mark.parametrize("cfg", [M.Config(1024, 1, True, False, False), M.Config(1024, 2, False, True, True),
                                 M.Config(1024, 2, True, True, False, out_size=42)],
                         ids=["L1024n1-nobn", "L1024n2-nores", "L1024n2-predict14"])
@pytest.mark.parametrize("B", [9, 40, 64])
def test_mid_batch_configs(cfg, B):
    """The 9 .. 64 pose range (the reference's batch_size flag is 64) on the other graphs a 1024-wide model can have:
    one residual block (2 hidden layers), no residual, 14-joint output (42 columns: a ragged last output group)."""
    m, p = make_model(cfg, seed=5, bn="trained", mode="bf16", predict_14=(cfg.out_size == 42))
    x, _ = synth.mlp_inputs(B, seed=7 + B)
    t = np.zeros((B, cfg.out_size), np.float32)
    _, _, y = m.step(None, x, t, 1.0, isTraining=False)
    ref = M.forward(p, x.astype(np.float64), cfg, training=False)
    emu = emulate_bf16_forward(p, x, cfg)
    assert y.shape == (B, cfg.out_size) and np.isfinite(y).all()
    assert_matches_emulation(y, emu, np.sqrt(np.mean(ref ** 2)), ref)
    assert rowwise_rel(y, ref).max() <= 1e-2
    # the same rows inside a larger batch go through another path (per-layer GEMMs): same rounding points
    xb, _ = synth.mlp_inputs(200, seed=99)
    xb[:B] = x
    _, _, yb = m.step(None, xb, np.zeros((200, cfg.out_size), np.float32), 1.0, isTraining=False)
    assert_matches_emulation(y, yb[:B].astype(np.float64), np.sqrt(np.mean(ref ** 2)))
    m.close()


def test_bf16_forward_without_max_norm_mm_error():
    """north_star: under 0.5 mm after un-normalise.  With sigma_3d = 100 mm and max_norm folded weights
    (the reference's training configuration) the bf16 path is far inside; without max_norm the outputs
    are O(1) normalised units and plain bf16 gives a few mm (SURVEY 7 'precision targets') - reported."""
    cfg = M.Config(1024, 2, True, True, True)
    m, p = make_model(cfg, seed=5, bn="fresh", mode="bf16")
    x, t = synth.mlp_inputs(4096, seed=9)
    _, _, y = m.step(None, x, t, 1.0, isTraining=False)
    ref = M.forward(p, x.astype(np.float64), cfg, training=False)
    assert np.abs(y - ref).max() * 100.0 < 0.5
    m.close()


def test_predict_14_and_empty_batch():
    cfg = M.Config(256, 1, True, True, False, out_size=42)
    m, p = make_model(cfg, seed=2, predict_14=True)
    x, _ = synth.mlp_inputs(200, seed=1)
    t = np.zeros((200, 42), np.float32)       # callers pass zeros for pure inference (sandbox_realtime.py:166)
    _, _, y = m.step(None, x, t, 1.0, isTraining=False)
    ref = M.forward(p, x.astype(np.float64), cfg, training=False)
    assert y.shape == (200, 42) and rowwise_rel(y, ref).max() <= 1e-2
    _, _, y0 = m.step(None, np.zeros((0, 32), np.float32), np.zeros((0, 42), np.float32), 1.0, isTraining=False)
    assert y0.shape == (0, 42)
    with pytest.raises(ValueError):
        m.step(None, np.zeros((4, 31), np.float32), np.zeros((4, 42), np.float32), 1.0, isTraining=False)
    m.close()


@pytest.mark.parametrize("cfg", [M.Config(1024, 2, True, True, True), M.Config(1024, 2, True, True, False),
                                 M.Config(64, 2, True, True, False), M.Config(100, 1, False, False, True)],
                         ids=["ref-maxnorm", "ref", "L64", "L100"])
def test_fp32_mode_matches_oracle(cfg):
    m, p = make_model(cfg, seed=7, bn="trained", mode="fp32")
    for B in (1, 64, 300):
        x, t = synth.mlp_inputs(B, seed=B)
        loss, _, y = m.step(None, x, t, 1.0, isTraining=False)
        ref = M.forward(p, x.astype(np.float64), cfg, training=False)
        assert rowwise_rel(y, ref).max() <= 1e-4, rowwise_rel(y, ref).max()
        assert abs(float(loss) - M.loss_fn(ref, t.astype(np.float64))) <= 1e-4 * max(1.0, float(loss))
    m.close()


def test_device_tensor_step_and_param_refresh():
    """torch CUDA tensors in -> torch out (no host copies); changing a variable re-folds the weights."""
    cfg = M.Config(256, 1, True, True, True)
    m, p = make_model(cfg, seed=4)
    x, t = synth.mlp_inputs(512, seed=2)
    xd, td = torch.from_numpy(x).cuda(), torch.from_numpy(t).cuda()
    loss, _, yd = m.step(None, xd, td, 1.0, isTraining=False)
    assert yd.is_cuda and yd.shape == (512, 48)
    ref = M.forward(p, x.astype(np.float64), cfg, training=False)
    assert rowwise_rel(yd.cpu().numpy(), ref).max() <= 1e-2
    assert abs(loss.item() - M.loss_fn(yd.cpu().numpy().astype(np.float64), t.astype(np.float64))) < 1e-4 * max(1, loss.item())
    p["linear_model/b4"] = p["linear_model/b4"] + 1.0
    m.set_variable("linear_model/b4", p["linear_model/b4"])
    _, _, yd2 = m.step(None, xd, td, 1.0, isTraining=False)
    assert np.allclose((yd2 - yd).cpu().numpy(), 1.0, atol=1e-3)
    got = m.get_variable("linear_model/w1")
    assert got.shape == (32, 256) and np.array_equal(got, p["linear_model/w1"].astype(np.float32))
    m.close()


def test_large_batch_properties():
    """At BASELINE's full size (2^20 poses) the oracle is too slow; use size-independent properties:
    row independence (every row equals the same row computed in a small batch) and determinism."""
    cfg = M.Config(1024, 2, True, True, True)
    m, p = make_model(cfg, seed=1, bn="trained")
    B = 1 << 20
    g = torch.Generator(device="cuda").manual_seed(0)
    xd = torch.randn((B, 32), device="cuda", generator=g)
    td = torch.zeros((B, 48), device="cuda")
    _, _, y1 = m.step(None, xd, td, 1.0, isTraining=False)
    _, _, y2 = m.step(None, xd, td, 1.0, isTraining=False)
    assert torch.equal(y1, y2)
    idx = torch.tensor([0, 1, 127, 128, 70000, 524287, 524288, B - 129, B - 1], device="cuda")
    rows = xd[idx].repeat(700, 1)                # 6300 rows -> the same fused kernel, other tiles
    _, _, ys = m.step(None, rows, torch.zeros((rows.shape[0], 48), device="cuda"), 1.0, isTraining=False)
    assert torch.allclose(ys[: idx.numel()], y1[idx], atol=1e-5, rtol=1e-5)
    # ... and the layered per-layer path (288 rows) rounds at the same points: it agrees up to the odd bf16-ulp flip
    _, _, yl = m.step(None, rows[:288].contiguous(), torch.zeros((288, 48), device="cuda"), 1.0, isTraining=False)
    dl = (yl[: idx.numel()] - y1[idx]).abs()
    assert dl.median() <= 1e-5 and dl.max() <= 2e-2 * y1[idx].abs().max()
    ref = M.forward(p, xd[idx].cpu().numpy().astype(np.float64), cfg, training=False)
    assert rowwise_rel(y1[idx].cpu().numpy(), ref).max() <= 1e-2
    assert torch.isfinite(y1).all()
    m.close()


def test_host_step_pinned_and_pageable_agree():
    from p3d import _lib
    cfg = M.Config(1024, 2, True, True, True)
    m, p = make_model(cfg, seed=8)
    B = 200000                                   # > one 65536-row pipeline chunk, ragged tail
    x, t = synth.mlp_inputs(B, seed=5)
    _, _, y_pageable = m.step(None, x, t, 1.0, isTraining=False)
    ptr = C.c_void_p()
    _lib.check(_lib.lib.p3d_host_alloc(C.byref(ptr), x.nbytes))
    xp = np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_float)), shape=x.shape)
    xp[:] = x
    loss, _, y_pinned = m.step(None, xp, t, 1.0, isTraining=False)
    assert np.array_equal(y_pageable, y_pinned)
    xd = torch.from_numpy(x).cuda()
    _, _, yd = m.step(None, xd, torch.from_numpy(t).cuda(), 1.0, isTraining=False)
    assert np.array_equal(yd.cpu().numpy(), y_pinned)
    assert abs(float(loss) - float(np.mean((y_pinned.astype(np.float64) - t) ** 2))) < 1e-4 * float(loss)
    del xp
    _lib.check(_lib.lib.p3d_host_free(ptr))
    m.close()


def test_width_4096_stress_config():
    """BASELINE configs[4]: linear_size=4096, num_layers=4 (134.6 M weights = 269 MB bf16 > L2) at 300 poses, which
    the layered path serves (one tcgen05 GEMM per layer, K = 4096).  The fused kernel at this width (16 chunks x 64
    K-slices per layer, 64 slab barriers) is checked in test_gpu_mlp_widths.py."""
    cfg = M.Config(4096, 4, True, True, True)
    m, p = make_model(cfg, seed=13, bn="trained", mode="bf16")
    x, t = synth.mlp_inputs(300, seed=3)
    _, _, y = m.step(None, x, t, 1.0, isTraining=False)
    ref = M.forward(p, x.astype(np.float64), cfg, training=False)
    emu = emulate_bf16_forward(p, x, cfg)
    assert_matches_emulation(y, emu, np.sqrt(np.mean(ref ** 2)), ref)
    assert rowwise_rel(y, ref).max() <= 1e-2
    m.close()


def test_step_without_target_is_an_extension_of_the_contract():
    """decoder_outputs=None (isTraining=False only): same predictions, loss 0, nothing uploaded for the target."""
    cfg = M.Config(1024, 2, True, True, True)
    m, p = make_model(cfg, seed=2)
    x, t = synth.mlp_inputs(700, seed=3)
    l0, _, y0 = m.step(None, x, t, 1.0, isTraining=False)
    l1, _, y1 = m.step(None, x, None, 1.0, isTraining=False)
    assert np.array_equal(y0, y1) and float(l1) == 0.0 and float(l0) > 0.0
    import torch
    xd = torch.from_numpy(x.astype(np.float32)).cuda()
    l2, _, y2 = m.step(None, xd, None, 1.0, isTraining=False)
    assert np.array_equal(y2.cpu().numpy(), y0) and float(l2) == 0.0
    with pytest.raises(ValueError):
        m.step(None, x, None, 0.5, isTraining=True)
    m.close()
