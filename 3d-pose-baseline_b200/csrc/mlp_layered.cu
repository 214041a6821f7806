// Layered inference forward for small and medium batches (2 <= B < ~6144) and for widths the fused
// persistent kernel does not tile (linear_size % 256 != 0): one tcgen05 GEMM per layer (tc_gemm.cu),
// bias + ReLU (+ residual) fused in the epilogue, bf16 activations ping-ponging between two L2-resident
// buffers.  Same graph as mlp_tc.cu (src/linear_model.py:102-125,154-201 at isTraining=False) and the same
// rounding points (relu(.) rounded to bf16, residual added and rounded again), so both paths agree.
//
// Why: a single 128-pose tile walks the six layers of the persistent kernel in ~100 us - one SM (pair) has
// to stream all 8.6 MB of weights by itself.  Splitting every layer over N (L/64 CTAs) spreads the weight
// stream over 16+ SMs; the layers are separate launches whose plans (tensor maps + parameters) are cached
// per batch size, so a call costs 1 + nlayers back-to-back launches and no host-side encoding.  The plans are kernel
// parameters (tensor maps by value), so a captured graph keeps its own copy; the buffers they address are never freed
// while a graph may hold them (retire()).
#include "common.cuh"

namespace p3d {
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
  P3D_REQUIRE((L % 8) == 0, "layered bf16 path needs linear_size %% 8 == 0 (got %d)", L);
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

}  // namespace layered
}  // namespace p3d
