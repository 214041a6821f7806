"""bf16 inference at every width and tile edge the two tensor-core paths serve, against the fp64 oracle
(oracle/mlp_ref.py) and the NumPy emulation of the kernels' rounding points (helpers.emulate_bf16_forward).

- The fused persistent kernel (csrc/mlp_tc.cu: B >= 6144, linear_size % 256 == 0 up to 4096) at 1 to 16 column chunks
  of 256, 4 to 64 K-slabs of 64, with and without residual / BatchNorm / max_norm, 48 and 42 (predict_14) outputs, at a
  batch that ends in a one-row tile and at one where every CTA pair runs two rounds and pair 0 a third, ragged one.
- The layered path (csrc/mlp_layered.cu: one tcgen05 GEMM per layer) at widths that are a multiple of 8 but not of 256,
  which it serves at every batch size: K tails zero-filled by TMA, partial last N tiles, clipped bf16 epilogues.

Every case proves which kernel ran: only the fused kernel records p3d_profile events, one per launch.

Every output row depends on its input row alone, so beyond width 1280 the host-side references run on a sample of rows:
the tiles where the persistent schedule changes hands (both CTAs of pair 0, the last pair of round 1, pair 0's round-2
tiles, the final ragged tile) plus 256 random rows."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import mlp_ref as M
from oracle import synth
from helpers import assert_matches_emulation, emulate_bf16_forward, make_model, rowwise_rel

pytestmark = pytest.mark.gpu

TILE = 128          # rows per CTA of the fused kernel; a CTA pair takes 2 tiles per round


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def multi_round_batch():
    """Batch with 2 * (SMs / 2) + 1 pair tiles whose last tile is ragged (37925 on a 148-SM part): every CTA pair runs
    two rounds, pair 0 a third one that holds 37 rows in its first CTA and none in its second."""
    return 2 * (_sms() // 2) * 2 * TILE + 37


def sample_rows(B, L, seed):
    """Rows the host-side references check: all of them up to width 1280, beyond it the fused kernel's telling tiles
    plus 256 random rows."""
    if L <= 1280:
        return np.arange(B)
    pairs = _sms() // 2
    ntiles = -(-B // TILE)
    last_round1 = min(-(-ntiles // 2), pairs) - 1
    tiles = {0, 1, 2 * last_round1, 2 * last_round1 + 1, 2 * pairs, 2 * pairs + 1, ntiles - 1}
    rows = [np.arange(t * TILE, min(B, (t + 1) * TILE)) for t in sorted(tiles) if t * TILE < B]
    rows.append(np.random.RandomState(seed).randint(0, B, 256))
    return np.unique(np.concatenate(rows))


def forward(m, xd, y=None):
    """One p3d_model_forward of the device rows xd into y (allocated when None).  Returns (y, launches of the fused
    kernel): the fused kernel is the only one that records p3d_profile events."""
    from p3d import _lib
    B = int(xd.shape[0])
    if y is None:
        y = torch.empty((B, m.output_size), dtype=torch.float32, device="cuda")
    ms, n = C.c_double(), C.c_int64()
    _lib.check(_lib.lib.p3d_profile_enable(1))
    try:
        _lib.check(_lib.lib.p3d_model_forward(m._handle, xd.data_ptr(), y.data_ptr(), B, _lib.current_stream()))
        _lib.check(_lib.lib.p3d_profile_read(C.byref(ms), C.byref(n)))
    finally:
        _lib.lib.p3d_profile_enable(0)
    return y, n.value


def check_rows(y_rows, x_rows, p, cfg):
    """Kernel rows against the emulation and the oracle; returns (kernel error, emulation error) against the oracle
    in units of the output rms, at q50 / q90 / q99."""
    y_rows = np.asarray(y_rows, np.float64)
    ref = M.forward(p, x_rows.astype(np.float64), cfg, training=False)
    emu = emulate_bf16_forward(p, x_rows, cfg)
    assert y_rows.shape == ref.shape and np.isfinite(y_rows).all()
    rms = np.sqrt(np.mean(ref ** 2))
    assert_matches_emulation(y_rows, emu, rms, ref)
    assert rowwise_rel(y_rows, ref).max() <= 1e-2, rowwise_rel(y_rows, ref).max()
    q = (0.5, 0.9, 0.99)
    return np.quantile(np.abs(y_rows - ref), q) / rms, np.quantile(np.abs(emu - ref), q) / rms


def _cfg_id(c):
    return f"L{c.linear_size}n{c.num_layers}r{int(c.residual)}b{int(c.batch_norm)}m{int(c.max_norm)}o{c.out_size}"


@pytest.fixture(scope="module")
def models():
    """One model per configuration, shared by the batch sizes of the module (the width-4096 fold is slow on the host)."""
    made = {}

    def get(cfg):
        key = _cfg_id(cfg)
        if key not in made:
            made[key] = make_model(cfg, seed=cfg.linear_size + cfg.num_layers, bn="trained", predict_14=(cfg.out_size == 42))
        return made[key]
    yield get
    for m, _ in made.values():
        m.close()


FUSED = [
    # linear_size, num_layers, residual, batch_norm, max_norm, out_size
    M.Config(256, 1, True, True, False, out_size=42),     # predict_14 in the fused kernel, 1 chunk
    M.Config(768, 2, True, True, True),                   # 3 chunks (odd), 12 slabs
    M.Config(1024, 2, True, True, True, out_size=42),     # predict_14 at the reference width
    M.Config(1280, 1, False, True, False),                # 5 chunks, no residual
    M.Config(2048, 2, True, False, False),                # 32 slabs, no BatchNorm
    M.Config(4096, 4, True, True, True),                  # configs[4]: 64 slabs = MAX_SLABS, scratch not L2-persisting
]


@pytest.mark.parametrize("batch", ["one_row_tile", "multi_round"])
@pytest.mark.parametrize("cfg", FUSED, ids=_cfg_id)
def test_fused_forward_widths(models, cfg, batch):
    """B = 6145: 49 tiles, the last pair holds one row and a CTA without rows.  multi_round: see multi_round_batch.
    The first 4096 checked rows also go through the layered path, which rounds at the same points: the two agree up to
    the odd bf16-ulp flip."""
    m, p = models(cfg)
    B = 6145 if batch == "one_row_tile" else multi_round_batch()
    x, _ = synth.mlp_inputs(B, seed=B + cfg.linear_size)
    xd = torch.from_numpy(x).cuda()
    y, fused = forward(m, xd)
    assert fused == 1
    assert torch.isfinite(y).all()
    rows = sample_rows(B, cfg.linear_size, seed=B)
    idx = torch.from_numpy(rows).cuda()
    ek, ee = check_rows(y[idx].cpu().numpy(), x[rows], p, cfg)
    if cfg.linear_size == 4096:
        print(f"{_cfg_id(cfg)} B={B}: |y - oracle| / rms at q50/q90/q99 kernel {ek} emulation {ee}")
    n = min(4096, rows.size)
    yl, fused_l = forward(m, xd[idx[:n]])
    assert fused_l == 0
    dl = (yl - y[idx[:n]]).abs()
    assert dl.median() <= 1e-5 and dl.max() <= 2e-2 * y[idx[:n]].abs().max(), (dl.median().item(), dl.max().item())


def test_width_4096_bench_size(models):
    """The shape stress_width4096 times: 2^21 poses through one fused launch at width 4096 with 4 residual blocks
    (16384 tiles, ~110 rounds per CTA pair), device tensors in and out.  Sampled rows against the emulation and the
    oracle; two calls are bit-identical."""
    cfg = M.Config(4096, 4, True, True, True)
    m, p = models(cfg)
    B = 1 << 21
    g = torch.Generator(device="cuda").manual_seed(21)
    xd = torch.randn((B, 32), device="cuda", generator=g)
    y1, n1 = forward(m, xd)
    y2, n2 = forward(m, xd)
    assert n1 == 1 and n2 == 1
    assert torch.equal(y1, y2) and torch.isfinite(y1).all()
    rows = sample_rows(B, cfg.linear_size, seed=7)
    idx = torch.from_numpy(rows).cuda()
    ek, ee = check_rows(y1[idx].cpu().numpy(), xd[idx].cpu().numpy(), p, cfg)
    print(f"{_cfg_id(cfg)} B={B} ({rows.size} rows): |y - oracle| / rms at q50/q90/q99 kernel {ek} emulation {ee}")


LAYERED = [
    M.Config(24, 1, True, False, False),                  # narrower than one 32/64-wide tile
    M.Config(72, 2, True, True, True),                    # K tail of 8, kpad = 72
    M.Config(200, 2, False, True, False, out_size=42),    # N % 32 != 0 (no 32-wide tiles), predict_14
    M.Config(1000, 2, True, True, True),                  # near the reference width: K tail 40, partial last N tile
]


@pytest.mark.parametrize("B", [1, 2, 100, 129, 6144, 20000])
@pytest.mark.parametrize("cfg", LAYERED, ids=_cfg_id)
def test_layered_forward_widths(models, cfg, B):
    """Widths that are a multiple of 8 but not of 256 take the layered path at every batch size, 6144 and above too."""
    m, p = models(cfg)
    x, _ = synth.mlp_inputs(B, seed=3 * B + cfg.linear_size)
    y, fused = forward(m, torch.from_numpy(x).cuda())
    assert fused == 0
    check_rows(y.cpu().numpy(), x, p, cfg)


def test_layered_plan_cache():
    """The layered path caches its per-layer plans (tensor maps of the input, activations and y) by batch size, packed
    input buffer and y, and re-plans only what changed.  Changing the batch size, y or the input in turn must give, call
    for call, bit-identical results to the same call on a fresh model."""
    cfg = M.Config(1000, 2, True, True, True)
    m, _ = make_model(cfg, seed=17)
    xa, xb = (torch.from_numpy(synth.mlp_inputs(100, seed=s)[0]).cuda() for s in (1, 2))
    x3000 = torch.from_numpy(synth.mlp_inputs(3000, seed=3)[0]).cuda()
    y1, y2, y3000 = (torch.empty((B, 48), device="cuda") for B in (100, 100, 3000))
    calls = [(xa, y1), (x3000, y3000), (xa, y2), (xb, y2), (xa, y1)]   # the last one: same B and input, other y
    for i, (xd, y) in enumerate(calls):
        _, fused = forward(m, xd, y)
        assert fused == 0
        fresh, _ = make_model(cfg, seed=17)
        yf, _ = forward(fresh, xd)
        fresh.close()
        assert torch.equal(y, yf), i
    m.close()
