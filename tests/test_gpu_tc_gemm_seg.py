"""The tcgen05 GEMM's segment schedule (csrc/tc_gemm.cu, SEG) on its own, through p3d_debug_tc_gemm_seg, for every
operand layout the bf16x3 training step uses, against a float64 sum of the three products of the bf16 halves:

    C[M,N] = alpha * (A.hi B.hi + A.lo B.hi + A.hi B.lo)^T-form  (+ res[m,n])

Every operand is a split pair: along its contiguous dimension (K for K-major, M or N for MN-major) the hi halves start at
column 0 and the lo halves at column `seg` (the width rounded up to 64), zeros in between.  The training step's shapes:
Z = H W (A K-major, B MN-major), dH = dZ W^T (both K-major, residual), dW = H^T dZ (both MN-major, K = batch rows,
split-K), with M = 32 (layer 0's weight gradient), N = 42 / 48 (the output layer) and K = 1, 63, 64, 65, 4096.  A lo
segment read from the wrong column or a K range walked by the wrong split costs ~2^-8 of the result; the bound is that
of tests/test_gpu_tc_gemm.py (fp32 accumulation in another order)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

CASES = [
    # every (a_mn, b_mn) layout, one tile and ragged
    dict(M=128, N=64, K=64, a_mn=0, b_mn=0),
    dict(M=128, N=64, K=64, a_mn=0, b_mn=1),
    dict(M=128, N=64, K=64, a_mn=1, b_mn=0),
    dict(M=128, N=64, K=64, a_mn=1, b_mn=1),
    dict(M=200, N=200, K=200, a_mn=1, b_mn=0),
    dict(M=200, N=200, K=200, a_mn=0, b_mn=1),
    # forward Z = H W and y = h W4
    dict(M=64, N=1024, K=32, a_mn=0, b_mn=1, seg_a=64, alpha=0.37),
    dict(M=4096, N=1024, K=1024, a_mn=0, b_mn=1),
    dict(M=1000, N=48, K=1024, a_mn=0, b_mn=1),
    dict(M=333, N=42, K=1024, a_mn=0, b_mn=1),
    # data gradient dH = dZ W^T (+ residual), and dh = dy W4^T (K = 48 / 42)
    dict(M=64, N=1024, K=1024, a_mn=0, b_mn=0, res=True, alpha=0.5),
    dict(M=4096, N=1024, K=1024, a_mn=0, b_mn=0, res=True),
    dict(M=4096, N=1024, K=48, a_mn=0, b_mn=0),
    dict(M=200, N=256, K=42, a_mn=0, b_mn=0),
    dict(M=300, N=1024, K=1, a_mn=0, b_mn=0),
    # weight gradients dW = H^T dZ: both MN-major, K = batch rows, split-K
    dict(M=1024, N=1024, K=4096, a_mn=1, b_mn=1, split_k=1),
    dict(M=1024, N=1024, K=64, a_mn=1, b_mn=1, split_k=1),
    dict(M=1024, N=1024, K=65, a_mn=1, b_mn=1, split_k=1),
    dict(M=32, N=1024, K=4096, a_mn=1, b_mn=1, split_k=1, seg_a=64),          # dW1: x split [B][128]
    dict(M=32, N=1024, K=63, a_mn=1, b_mn=1, split_k=1, seg_a=64),
    dict(M=1024, N=48, K=4096, a_mn=1, b_mn=1, split_k=1),                    # dW4
    dict(M=1024, N=42, K=1, a_mn=1, b_mn=1, split_k=1),
    dict(M=256, N=200, K=1000, a_mn=1, b_mn=1, split_k=1),
    dict(M=1024, N=1024, K=4096, a_mn=1, b_mn=1),                             # MN-major, unsplit
]


def _case_id(c):
    s = f"M{c['M']}N{c['N']}K{c['K']}a{c['a_mn']}b{c['b_mn']}"
    for k in ("split_k", "res"):
        if c.get(k):
            s += "-" + k
    return s


def _seg(n):
    return (n + 63) // 64 * 64


def split_pair(X, seg):
    """fp32 [rows][n] -> bf16 [rows][2 seg]: hi in columns 0..n-1, lo = bf16(X - hi) from column seg; and the halves."""
    rows, n = X.shape
    hi = X.to(torch.bfloat16)
    lo = (X - hi.float()).to(torch.bfloat16)
    buf = torch.zeros((rows, 2 * seg), dtype=torch.bfloat16, device=X.device)
    buf[:, :n] = hi
    buf[:, seg:seg + n] = lo
    return buf, hi.double().cpu().numpy(), lo.double().cpu().numpy()


@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_segment_schedule_matches_three_products(case):
    from p3d import _lib
    M, N, K, a_mn, b_mn = case["M"], case["N"], case["K"], case["a_mn"], case["b_mn"]
    split_k, alpha = case.get("split_k", 0), case.get("alpha", 1.0)
    g = torch.Generator(device="cuda").manual_seed(M * 7 + N * 3 + K)
    A = torch.randn((K, M) if a_mn else (M, K), generator=g, device="cuda")
    B = torch.randn((K, N) if b_mn else (N, K), generator=g, device="cuda")
    seg_a = case.get("seg_a", _seg(M if a_mn else K))
    seg_b = _seg(N if b_mn else K)
    As, ah, al = split_pair(A, seg_a)
    Bs, bh, bl = split_pair(B, seg_b)
    C = torch.zeros((M, N), device="cuda") if split_k else torch.full((M, N), float("nan"), device="cuda")
    res = torch.randn((M, N), generator=g, device="cuda") if case.get("res") else None
    _lib.check(_lib.lib.p3d_debug_tc_gemm_seg(As.data_ptr(), As.shape[1], a_mn, seg_a, Bs.data_ptr(), Bs.shape[1], b_mn, seg_b,
                                              C.data_ptr(), N, M, N, K, res.data_ptr() if res is not None else None, alpha,
                                              split_k, None))
    torch.cuda.synchronize()
    op_a = (lambda x: x.T) if a_mn else (lambda x: x)   # noqa: E731  -> [M][K]
    op_b = (lambda x: x) if b_mn else (lambda x: x.T)   # noqa: E731  -> [K][N]
    ref = alpha * (op_a(ah) @ op_b(bh) + op_a(al) @ op_b(bh) + op_a(ah) @ op_b(bl))
    if res is not None:
        ref += res.cpu().numpy().astype(np.float64)
    got = C.cpu().numpy().astype(np.float64)
    assert np.isfinite(got).all(), f"{int((~np.isfinite(got)).sum())} output elements not written"
    err = np.abs(got - ref).max() / np.abs(ref).max()
    assert err <= 2e-5 * max(1.0, (K / 64) ** 0.5) + (1e-5 if split_k else 1e-6), err
    # and the sum is the fp32-class product: what the dropped lo.lo term and the operand split leave is ~2^-16
    exact = alpha * (op_a(A.double().cpu().numpy()) @ op_b(B.double().cpu().numpy()))
    if res is not None:
        exact += res.cpu().numpy().astype(np.float64)
    assert np.abs(got - exact).max() / np.abs(exact).max() <= 1e-4
