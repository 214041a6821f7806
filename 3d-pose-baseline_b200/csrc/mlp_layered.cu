// Layered inference forward for small and medium batches (2 <= B < ~6144) and for widths the fused
// persistent kernel does not tile (linear_size % 256 != 0): one tcgen05 GEMM per layer (tc_gemm.cu),
// bias + ReLU (+ residual) fused in the epilogue, bf16 activations ping-ponging between two L2-resident
// buffers.  Same graph as mlp_tc.cu (src/linear_model.py:102-125,154-201 at isTraining=False) and the same
// rounding points (relu(.) rounded to bf16, residual added and rounded again), so both paths agree.  P3D_MODE_FP16
// models run the same chain on fp16 operands and activations (GemmArgs::f16).
//
// Why: a single 128-pose tile walks the six layers of the persistent kernel in ~100 us - one SM (pair) has
// to stream all 8.6 MB of weights by itself.  Splitting every layer over N (L/64 CTAs) spreads the weight
// stream over 16+ SMs; the layers are separate launches whose plans (tensor maps + parameters) are cached
// per batch size, so a call costs 1 + nlayers back-to-back launches and no host-side encoding.  The plans are kernel
// parameters (tensor maps by value), so a captured graph keeps its own copy; the buffers they address are never freed
// while a graph may hold them (retire()).
#include "common.cuh"

namespace p3d {
namespace prep { int pack_input_split(const float*, __nv_bfloat16*, int64_t, cudaStream_t); }
namespace layered {

static int build_plans(p3d_model* m, const __nv_bfloat16* xb, float* y, int64_t B, bool only_last) {
  const int L = m->L, kpad = m->kpad;
  const int nlay = static_cast<int>(m->layers.size());
  __nv_bfloat16* P = m->lay_act;
  __nv_bfloat16* Q = m->lay_act + static_cast<size_t>(m->lay_cap) * L;
  m->lay_plans.resize(nlay);
  for (int l = only_last ? nlay - 1 : 0; l < nlay; ++l) {
    const Layer& ly = m->layers[l];
    const bool last = (l == nlay - 1);
    tcg::GemmArgs g;
    g.M = static_cast<int>(B); g.N = ly.N; g.K = (l == 0) ? 64 : L;
    if (l == 0) { g.A = xb; g.lda = 64; }
    else { g.A = (l & 1) ? P : Q; g.lda = L; }                       // odd layers read the block input P, even ones Q
    g.B = m->wt_bf16 + static_cast<size_t>(ly.row_off) * kpad; g.ldb = kpad;    // folded W'^T, K-major
    g.bias = m->bias_fold + ly.row_off;
    g.pdl = 1;                                       // layer l+1 starts (and prefetches its weights) while layer l drains
    g.f16 = m->cfg.mode == P3D_MODE_FP16 ? 1 : 0;
    if (last) {
      g.C = y; g.ldc = m->out_size;
    } else {
      const bool to_p = (l == 0) || ((l & 1) == 0);
      g.out_bf16 = to_p ? P : Q; g.ld_out_bf16 = L; g.relu = 1;
      if (m->cfg.residual && l >= 2 && (l & 1) == 0) { g.res_bf16 = P; g.ld_res_bf16 = L; }   // P = relu(.) + P, in place
    }
    P3D_TRY(tcg::plan(g, &m->lay_plans[l]));
  }
  return P3D_OK;
}

int forward(p3d_model* m, const __nv_bfloat16* xb, float* y, int64_t B, cudaStream_t st) {
  const int L = m->L;
  P3D_REQUIRE((L % 8) == 0, "layered bf16 / fp16 path needs linear_size %% 8 == 0 (got %d)", L);
  P3D_REQUIRE(B <= 0x7fffffff, "layered path: batch too large");
  bool rebuild = (m->lay_B != B) || (m->lay_x != xb) || m->lay_plans.empty();
  if (m->lay_cap < B) {
    P3D_TRY(refuse_in_capture(st, "forward: growing the layered path's activation buffers"));
    const int64_t cap = grown_cap(m, m->lay_cap, B < 1024 ? 1024 : B);
    retire(m, m->lay_act);
    m->lay_act = nullptr; m->lay_cap = 0;
    P3D_CUDA(cudaMalloc(&m->lay_act, sizeof(__nv_bfloat16) * 2ull * cap * L));
    m->lay_cap = cap;
    rebuild = true;
  }
  if (rebuild) P3D_TRY(build_plans(m, xb, y, B, false));
  else if (m->lay_y != y) P3D_TRY(build_plans(m, xb, y, B, true));
  m->lay_B = B; m->lay_x = xb; m->lay_y = y;
  for (const auto& pl : m->lay_plans) P3D_TRY(tcg::launch(pl, st));
  return P3D_OK;
}

// ----------------------------------------------------------------------------- bf16x3 (split precision)
// The same chain for P3D_MODE_BF16X3: every operand is a split pair (hi = bf16(a), lo = bf16(a - hi)) and every layer
// one GEMM with the segment schedule, A.hi B.hi + A.lo B.hi + A.hi B.lo accumulated in fp32 in TMEM.  Activations stay
// fp32: each hidden epilogue stores the split pair of relu(.) (+ residual) for the next layer, and the fp32 value itself
// where a later block adds it (the residual stream, in place).  Rows go in chunks of kSplitChunk, so the scratch is
// bounded whatever the batch (unchunked, 2^20 poses at width 4096 would need ~50 GB); a chunk of 32768 rows still
// gives every layer 256 M tiles.
constexpr int64_t kSplitChunk = 32768;

static int build_split_plans(p3d_model* m, p3d_model::X3Plans& ps, int64_t rows, float* y, bool only_last) {
  const int L = m->L, seg = m->x3_seg, ld = 2 * seg;
  const int nlay = static_cast<int>(m->layers.size());
  __nv_bfloat16* P = m->x3_act;
  __nv_bfloat16* Q = m->x3_act + static_cast<size_t>(m->x3_cap) * ld;
  ps.pl.resize(nlay);
  for (int l = only_last ? nlay - 1 : 0; l < nlay; ++l) {
    const Layer& ly = m->layers[l];
    tcg::GemmArgs g;
    g.M = static_cast<int>(rows); g.N = ly.N; g.K = ly.K;
    if (l == 0) { g.A = m->x3_in; g.lda = 128; g.seg_a = 64; }
    else { g.A = (l & 1) ? P : Q; g.lda = ld; g.seg_a = seg; }       // same wiring as build_plans
    g.B = m->wt_x3 + static_cast<size_t>(ly.row_off) * ld; g.ldb = ld; g.seg_b = seg;
    g.bias = m->bias_fold + ly.row_off;
    g.pdl = 1;
    if (l == nlay - 1) {
      g.C = y; g.ldc = m->out_size;
    } else {
      const bool to_p = (l == 0) || ((l & 1) == 0);
      g.out_bf16 = to_p ? P : Q; g.ld_out_bf16 = ld; g.out_lo = seg; g.relu = 1;
      if (m->cfg.residual && to_p) {
        g.C = m->x3_res; g.ldc = L;                                       // the block output a later block adds
        if (l >= 2) { g.res = m->x3_res; g.ldres = L; }                   // x3_res = relu(.) + x3_res, in place
      }
    }
    P3D_TRY(tcg::plan(g, &ps.pl[l]));
  }
  return P3D_OK;
}

int forward_split(p3d_model* m, const float* x, float* y, int64_t B, cudaStream_t st) {
  const int L = m->L, ld = 2 * m->x3_seg;
  P3D_REQUIRE((L % 8) == 0 && m->wt_x3, "bf16x3 path needs a bf16x3 model with linear_size %% 8 == 0 (got %d)", L);
  const int64_t need = B < kSplitChunk ? B : kSplitChunk;
  if (m->x3_cap < need) {
    P3D_TRY(refuse_in_capture(st, "forward: growing the bf16x3 path's activation buffers"));
    int64_t cap = grown_cap(m, m->x3_cap, need < 1024 ? 1024 : need);
    if (cap > kSplitChunk) cap = kSplitChunk;
    retire(m, m->x3_in); retire(m, m->x3_act); retire(m, m->x3_res);
    m->x3_in = nullptr; m->x3_act = nullptr; m->x3_res = nullptr; m->x3_cap = 0;
    P3D_CUDA(cudaMalloc(&m->x3_in, sizeof(__nv_bfloat16) * 128ull * cap));
    P3D_CUDA(cudaMalloc(&m->x3_act, sizeof(__nv_bfloat16) * 2ull * cap * ld));
    P3D_CUDA(cudaMemsetAsync(m->x3_act, 0, sizeof(__nv_bfloat16) * 2ull * cap * ld, st));   // padding columns stay zero
    if (m->cfg.residual) P3D_CUDA(cudaMalloc(&m->x3_res, sizeof(float) * static_cast<size_t>(cap) * L));
    m->x3_cap = cap;
    for (auto& ps : m->x3_plans) ps.rows = -1;
  }
  for (int64_t r0 = 0; r0 < B; r0 += kSplitChunk) {
    const int64_t n = (B - r0 < kSplitChunk) ? B - r0 : kSplitChunk;
    float* yc = y + r0 * m->out_size;
    p3d_model::X3Plans& ps = m->x3_plans[n == kSplitChunk ? 0 : 1];
    if (ps.rows != n) P3D_TRY(build_split_plans(m, ps, n, yc, false));
    else if (ps.y != yc) P3D_TRY(build_split_plans(m, ps, n, yc, true));
    ps.rows = n; ps.y = yc;
    P3D_TRY(prep::pack_input_split(x + r0 * kIn, m->x3_in, n, st));
    for (const auto& pl : ps.pl) P3D_TRY(tcg::launch(pl, st));
  }
  return P3D_OK;
}

}  // namespace layered
}  // namespace p3d
