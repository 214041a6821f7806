"""The arithmetic of the fp16 inference mode (P3D_MODE_FP16), restated in NumPy at its rounding points, against the
fp64 oracle (oracle/mlp_ref.py) and the golden fixture.

fp16 mode rounds where bf16 mode rounds - folded weights, the input, every ReLU output and every residual sum - and
accumulates in fp32; only the 16-bit format differs (10 mantissa bits instead of 7).  So the emulation is
helpers.emulate_bf16_forward run with fp16 rounding (emulate_fp16_forward below).  The contract is 2e-3 row-wise, and on every case fp16 must be at
least 5x more accurate than bf16.  The GPU tests (tests/test_gpu_mlp_fp16.py) hold the kernels to this emulation."""
import numpy as np
import pytest

import helpers
from helpers import emulate_bf16_forward, rowwise_rel
from oracle import mlp_ref as M
from oracle import synth
from test_oracle_mlp_golden import GOLD, case_setup, head_of

CONTRACT = 2e-3


def fp16_round(a):
    """Round-to-nearest-even to IEEE half precision (subnormals kept), returned as float32 values."""
    return np.asarray(a, dtype=np.float32).astype(np.float16).astype(np.float32)


def emulate_fp16_forward(p, x, cfg, small_batch=False):
    """What the fp16-mode kernels compute: helpers.emulate_bf16_forward, whose every rounding point goes through its
    module's bf16_round, run with fp16_round in that place - the same rounding points, the fp16 format."""
    saved = helpers.bf16_round
    helpers.bf16_round = fp16_round
    try:
        return emulate_bf16_forward(p, x, cfg, small_batch=small_batch)
    finally:
        helpers.bf16_round = saved


def _case(L, nl, max_norm, bn="trained", rows=256, seed=21):
    cfg = M.Config(L, nl, True, True, max_norm)
    p = {k: v.astype(np.float32).astype(np.float64) for k, v in M.init_params(L, nl, seed=seed, bn=bn).items()}
    x = synth.mlp_inputs(rows, seed=seed)[0].astype(np.float64)
    return cfg, p, x, M.forward(p, x, cfg, training=False)


CASES = [(1024, 2, False, "trained"), (1024, 2, False, "fresh"), (1024, 2, True, "trained"), (4096, 4, True, "trained")]


@pytest.mark.parametrize("L,nl,max_norm,bn", CASES, ids=["L1024n2", "L1024n2fresh", "L1024n2mn", "L4096n4mn"])
def test_fp16_meets_contract_and_beats_bf16(L, nl, max_norm, bn):
    cfg, p, x, ref = _case(L, nl, max_norm, bn)
    e16 = rowwise_rel(emulate_fp16_forward(p, x, cfg), ref).max()
    eb = rowwise_rel(emulate_bf16_forward(p, x, cfg), ref).max()
    assert e16 <= CONTRACT, e16
    assert 5 * e16 <= eb, (e16, eb)


def test_fp16_round():
    """Round to nearest even at fp16's 10 mantissa bits; subnormals and the range limit are fp16's."""
    v = np.array([1 + 2 ** -11, 1 + 3 * 2 ** -11, 2 ** -24, 2 ** -25 * 1.5, 65504, 65520], np.float32)
    with np.errstate(over="ignore"):
        r = fp16_round(v)
    np.testing.assert_array_equal(r, np.array([1, 1 + 2 ** -9, 2 ** -24, 2 ** -24, 65504, np.inf], np.float32))


EVAL_TAGS = ["s_res_bn_mn", "s_res_bn", "s_bn_mn_1", "s_res_3", "s_mn", "s_p14", "s_fresh", "h_1024_b64",
             "h_1024_b64_nomn", "h_1024_b4096"]


@pytest.mark.parametrize("tag", EVAL_TAGS)
def test_golden_eval_cases(tag):
    """Every inference case of tests/golden/mlp.npz (the reference graph's own outputs): the contract, the loss, and
    at least 5x the accuracy of the bf16 emulation."""
    z = np.load(GOLD)
    cfg, p, x, t, B, steps, big, lr0 = case_setup(z, tag)
    key = tag + "/eval_y"
    ref = z[key] if key in z.files else z[key + "@head"]
    y = emulate_fp16_forward(p, x, cfg)
    e16 = rowwise_rel(head_of(y, ref), ref).max()
    eb = rowwise_rel(head_of(emulate_bf16_forward(p, x, cfg), ref), ref).max()
    assert e16 <= CONTRACT, e16
    assert 5 * e16 <= eb, (e16, eb)
    gl = float(z[tag + "/eval_loss"])
    assert abs(M.loss_fn(y, t) - gl) <= CONTRACT * gl, (M.loss_fn(y, t), gl)
