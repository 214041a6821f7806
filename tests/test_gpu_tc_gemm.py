"""The generic tcgen05 GEMM (csrc/tc_gemm.cu, through p3d_debug_tc_gemm) on its own, against a float64 product of the
bf16-rounded operands with alpha, bias and residual applied:

    C[M,N] = alpha * A B^T (+ bias[n]) (+ res[m,n]),   colsum = column sums of C and of C^2

The training step and the layered inference path are built from this kernel; when one of them fails, these cases say
whether the GEMM itself is wrong.  The cases are those of tools/diag_tcgemm.py, which stays the localising diagnostic
(per-block errors, K-slice coefficients): every operand layout, each tile width pick_bn can choose, split-K with ragged
and short K, every epilogue input, ragged M, N and K.  C is prefilled with NaN when K is not split (a split GEMM
accumulates into a zeroed C), so every output element must have been written; one case has ldc > N and sentinel columns
[N, ldc) that must come back untouched.

Bounds (the diagnostic's): max |C - ref| <= (2e-5 * max(1, sqrt(K / 64)) + 1e-6) * max |ref|, + 1e-5 instead of 1e-6
when K is split (fp32 atomics in another order); column sums within 1e-4 of their largest."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

SENTINEL = -7.25

CASES = [
    # one tile, every (a_mn, b_mn) layout: K-major = [rows][K], MN-major = [K][rows]
    dict(M=128, N=64, K=64, a_mn=0, b_mn=0),
    dict(M=128, N=64, K=64, a_mn=0, b_mn=1),
    dict(M=128, N=64, K=64, a_mn=1, b_mn=0),
    dict(M=128, N=64, K=64, a_mn=1, b_mn=1),
    dict(M=128, N=256, K=256, a_mn=0, b_mn=1),
    dict(M=128, N=256, K=256, a_mn=1, b_mn=1),
    # the training step's shapes at batch 64
    dict(M=64, N=1024, K=32, a_mn=0, b_mn=1, bias=True, colsum=True, alpha=0.37),    # z0 = x W1
    dict(M=64, N=1024, K=1024, a_mn=0, b_mn=1, bias=True, colsum=True),              # z = h W
    dict(M=64, N=48, K=1024, a_mn=0, b_mn=1, bias=True),                             # y = h W4
    dict(M=64, N=1024, K=48, a_mn=0, b_mn=0),                                        # dh = dy W4^T
    dict(M=64, N=1024, K=1024, a_mn=0, b_mn=0, res=True),                            # dh = dz W^T + dres
    # split-K (weight gradients): K blocks <= 4 narrow the tile to 64, longer K keeps it wide
    dict(M=1024, N=1024, K=64, a_mn=1, b_mn=1, split_k=1),                           # dW = h^T dz
    dict(M=1024, N=48, K=64, a_mn=1, b_mn=1, split_k=1),                             # dW4
    dict(M=32, N=1024, K=64, a_mn=1, b_mn=1, split_k=1),                             # dW1
    dict(M=1024, N=1024, K=256, a_mn=1, b_mn=1, split_k=1),                          # 4 K blocks
    dict(M=384, N=1024, K=512, a_mn=1, b_mn=1, split_k=1),                           # BN = 256, 3 M tiles
    dict(M=1024, N=1024, K=1000, a_mn=1, b_mn=1, split_k=1),                         # ragged K
    dict(M=1000, N=96, K=1000, a_mn=1, b_mn=1, split_k=1),                           # ragged M, N and K
    # BN = 32: one M tile, N >= 256, N % 32 == 0, K-major B, no split (the layered inference layers)
    dict(M=1, N=1024, K=1024, a_mn=0, b_mn=0, bias=True),
    dict(M=2, N=1024, K=1024, a_mn=0, b_mn=0, bias=True),
    dict(M=7, N=256, K=1000, a_mn=0, b_mn=0, bias=True),
    dict(M=61, N=1024, K=1024, a_mn=0, b_mn=0, bias=True, res=True),
    dict(M=100, N=1024, K=64, a_mn=0, b_mn=0, bias=True),
    # BN = 64: N = 200 is not a multiple of 32, so a single M tile keeps 64-wide tiles
    dict(M=100, N=200, K=200, a_mn=0, b_mn=0, bias=True),
    dict(M=97, N=1024, K=64, a_mn=0, b_mn=1, bias=True, colsum=True, alpha=0.5),     # last quadrant holds one live row
    # BN = 128: 17 M tiles x 8
    dict(M=2176, N=1024, K=256, a_mn=0, b_mn=1, bias=True, colsum=True),
    dict(M=2100, N=1024, K=320, a_mn=0, b_mn=0, res=True),
    # BN = 256: 33 M tiles x 4
    dict(M=4224, N=1024, K=128, a_mn=0, b_mn=1),
    dict(M=4224, N=1024, K=1024, a_mn=0, b_mn=0, bias=True, res=True, colsum=True, alpha=0.75),
    # ragged M and N, K = 32 / 48
    dict(M=1000, N=1024, K=1024, a_mn=0, b_mn=1, bias=True, colsum=True),
    dict(M=1000, N=200, K=48, a_mn=0, b_mn=1, bias=True),
    dict(M=333, N=48, K=128, a_mn=0, b_mn=1, bias=True),                             # N ends inside a 32-column box
    dict(M=4096, N=48, K=1024, a_mn=0, b_mn=1, bias=True),                           # y = h W4 at batch 4096
    dict(M=4096, N=1024, K=48, a_mn=0, b_mn=0),                                      # dh = dy W4^T at batch 4096
    dict(M=1000, N=96, K=32, a_mn=0, b_mn=0, bias=True, colsum=True),
    # ldc > N: columns [N, ldc) of C (and of the residual, which shares the pitch) are not the GEMM's
    dict(M=333, N=48, K=128, a_mn=0, b_mn=1, bias=True, res=True, ldc=64),
    dict(M=1000, N=200, K=1000, a_mn=0, b_mn=0, bias=True, ldc=256),
]


def _case_id(c):
    s = f"M{c['M']}N{c['N']}K{c['K']}a{c['a_mn']}b{c['b_mn']}"
    for k in ("split_k", "bias", "res", "colsum"):
        if c.get(k):
            s += "-" + k
    if c.get("alpha", 1.0) != 1.0:
        s += f"-alpha{c['alpha']}"
    if c.get("ldc"):
        s += f"-ldc{c['ldc']}"
    return s


@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_tc_gemm_matches_fp64(case):
    from p3d import _lib
    M, N, K, a_mn, b_mn = case["M"], case["N"], case["K"], case["a_mn"], case["b_mn"]
    split_k, alpha = case.get("split_k", 0), case.get("alpha", 1.0)
    ldc = case.get("ldc", N)
    g = torch.Generator(device="cuda").manual_seed(M * 7 + N * 3 + K)
    A = torch.randn((K, M) if a_mn else (M, K), generator=g, device="cuda").to(torch.bfloat16)
    B = torch.randn((K, N) if b_mn else (N, K), generator=g, device="cuda").to(torch.bfloat16)
    C = torch.full((M, ldc), float("nan"), device="cuda")
    if split_k:
        C[:, :N] = 0.0
    C[:, N:] = SENTINEL
    bias = torch.randn(N, generator=g, device="cuda") if case.get("bias") else None
    res = torch.randn((M, ldc), generator=g, device="cuda") if case.get("res") else None
    colsum = torch.zeros(2 * N, dtype=torch.float64, device="cuda") if case.get("colsum") else None
    _lib.check(_lib.lib.p3d_debug_tc_gemm(A.data_ptr(), A.shape[1], a_mn, B.data_ptr(), B.shape[1], b_mn, C.data_ptr(), ldc,
                                          M, N, K, bias.data_ptr() if bias is not None else None,
                                          res.data_ptr() if res is not None else None, alpha, split_k,
                                          colsum.data_ptr() if colsum is not None else None, None))
    torch.cuda.synchronize()

    Af = A.float().cpu().numpy().astype(np.float64)
    Bf = B.float().cpu().numpy().astype(np.float64)
    ref = alpha * ((Af.T if a_mn else Af) @ (Bf if b_mn else Bf.T))
    if bias is not None:
        ref += bias.cpu().numpy().astype(np.float64)[None, :]
    if res is not None:
        ref += res[:, :N].cpu().numpy().astype(np.float64)
    got = C.cpu().numpy()
    assert np.all(got[:, N:] == SENTINEL), "columns past N were written"
    got = got[:, :N].astype(np.float64)
    assert np.isfinite(got).all(), f"{int((~np.isfinite(got)).sum())} output elements not written"
    scale = np.abs(ref).max()
    err = np.abs(got - ref).max() / scale
    assert err <= 2e-5 * max(1.0, (K / 64) ** 0.5) + (1e-5 if split_k else 1e-6), err
    if colsum is not None:
        cs = colsum.cpu().numpy()
        for got_s, ref_s in ((cs[:N], ref.sum(0)), (cs[N:], (ref * ref).sum(0))):
            assert np.abs(got_s - ref_s).max() <= 1e-4 * np.abs(ref_s).max(), np.abs(got_s - ref_s).max() / np.abs(ref_s).max()
