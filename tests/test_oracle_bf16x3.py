"""The arithmetic of the bf16x3 inference mode (P3D_MODE_BF16X3), restated in NumPy at its rounding points, against the
fp64 oracle (oracle/mlp_ref.py) and the golden fixture.

Every fp32 operand a is split into hi = bf16(a) and lo = bf16(a - hi); a MatMul is the sum of the three products
hi.hi + lo.hi + hi.lo (activation half first, weight half second) accumulated in fp32; bias, ReLU and the residual
add stay fp32, and so do the activations between layers.  The dropped lo.lo term is 2^-16 of the product, so three
products land far inside the fp32 contract (1e-4 row-wise), while any two of them leave a bf16-sized error behind -
which is why the mode pays for three.  The GPU tests (tests/test_gpu_mlp_bf16x3.py) hold the kernels to this
emulation."""
import numpy as np
import pytest

from helpers import bf16_round, rowwise_rel
from oracle import mlp_ref as M
from oracle import synth
from test_oracle_mlp_golden import GOLD, case_setup, head_of

THREE = ("hh", "lh", "hl")     # (activation half, weight half) of each product


def split(a):
    """fp32 a -> (hi, lo) as float32 arrays: hi = bf16(a), lo = bf16(a - hi) (the subtraction is exact in fp32)."""
    a32 = np.asarray(a, np.float32)
    hi = bf16_round(a32)
    return hi, bf16_round(a32 - hi)


def emulate_bf16x3_forward(p, x, cfg, products=THREE):
    """What the bf16x3 forward computes: folded weights held in fp32 and split, the input and every activation split
    as it enters a MatMul, the chosen products summed in fp32, bias / ReLU / residual in fp32.  Returns float64."""
    folded = M.fold_inference(p, cfg)
    h = np.asarray(x, np.float32)
    res = None
    last = len(folded) - 1
    for li, (w, b) in enumerate(folded):
        halves_a, halves_w = dict(zip("hl", split(h))), dict(zip("hl", split(w)))
        acc = np.zeros((h.shape[0], w.shape[1]), np.float32)
        for pa, pw in products:
            acc += halves_a[pa] @ halves_w[pw]
        z = acc + b.astype(np.float32)
        if li == last:
            return z.astype(np.float64)
        r = np.maximum(z, np.float32(0))
        if li == 0 or li % 2 == 1:
            h = r
        else:
            h = (r + res) if cfg.residual else r
        if li == 0 or li % 2 == 0:
            res = h


def _case(L, nl, max_norm, rows=256, seed=21):
    cfg = M.Config(L, nl, True, True, max_norm)
    p = {k: v.astype(np.float32).astype(np.float64) for k, v in M.init_params(L, nl, seed=seed, bn="trained").items()}
    x = synth.mlp_inputs(rows, seed=seed)[0].astype(np.float64)
    return cfg, p, x, M.forward(p, x, cfg, training=False)


CASES = [(1024, 2, False), (1024, 2, True), (4096, 4, True)]


@pytest.mark.parametrize("L,nl,max_norm", CASES, ids=["L1024n2", "L1024n2mn", "L4096n4mn"])
def test_three_products_meet_fp32_contract(L, nl, max_norm):
    cfg, p, x, ref = _case(L, nl, max_norm)
    y = emulate_bf16x3_forward(p, x, cfg)
    assert rowwise_rel(y, ref).max() <= 1e-4, rowwise_rel(y, ref).max()


@pytest.mark.parametrize("products", [("hh",), ("hh", "hl"), ("hh", "lh")], ids=["hh", "hh+hl", "hh+lh"])
def test_fewer_products_do_not(products):
    """Without max_norm the trained-BN model amplifies operand rounding to ~5e-3 row-wise; only the third product
    removes it."""
    cfg, p, x, ref = _case(1024, 2, False)
    y = emulate_bf16x3_forward(p, x, cfg, products)
    assert rowwise_rel(y, ref).max() > 1e-3, rowwise_rel(y, ref).max()


EVAL_TAGS = ["s_res_bn_mn", "s_res_bn", "s_bn_mn_1", "s_res_3", "s_mn", "s_p14", "s_fresh", "h_1024_b64",
             "h_1024_b64_nomn", "h_1024_b4096"]


@pytest.mark.parametrize("tag", EVAL_TAGS)
def test_golden_eval_cases(tag):
    """Every inference case of tests/golden/mlp.npz (the reference graph's own outputs), at the fp32 tolerance."""
    z = np.load(GOLD)
    cfg, p, x, t, B, steps, big, lr0 = case_setup(z, tag)
    y = emulate_bf16x3_forward(p, x, cfg)
    key = tag + "/eval_y"
    ref = z[key] if key in z.files else z[key + "@head"]
    got = head_of(y, ref)
    assert rowwise_rel(got, ref).max() <= 1e-4, rowwise_rel(got, ref).max()
    loss = M.loss_fn(y, t)
    assert abs(loss - float(z[tag + "/eval_loss"])) <= 1e-4 * float(z[tag + "/eval_loss"])
