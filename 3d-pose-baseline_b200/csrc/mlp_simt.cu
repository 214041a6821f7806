// FP32 (FFMA) kernels: the "fp32 mode" forward (<=1e-4 of the fp64 oracle), the small-batch
// (latency) forward and the generic SGEMM the training step is built from.
// Same graph as mlp_tc.cu: src/linear_model.py:102-125,154-201.
#include <cstdlib>

#include "common.cuh"
#include "math_hd.h"

namespace p3d {
namespace simt {

constexpr int TM = 64, TN = 64, TK = 16;


// C[M,N] = epi(alpha * op(A)[M,K] op(B)[K,N]);  op(A)[m,k] = TA ? A[k*lda+m] : A[m*lda+k],
// op(B)[k,n] = TB ? B[n*ldb+k] : B[k*ldb+n].  256 threads, 64x64 tile, 4x4 per thread.
template <bool TA, bool TB>
__global__ void __launch_bounds__(256) sgemm_kernel(int M, int N, int K, const float* __restrict__ A, int lda,
                                                    const float* __restrict__ B, int ldb, float* __restrict__ C,
                                                    int ldc, const Epilogue e) {
  __shared__ float As[TK][TM + 4];
  __shared__ float Bs[TK][TN + 4];
  const int tid = threadIdx.x;
  const long long m0 = static_cast<long long>(blockIdx.y) * TM;
  const int n0 = blockIdx.x * TN;
  const int tx = tid & 15, ty = tid >> 4;   // 16 x 16 threads, each a 4x4 micro tile
  float acc[4][4] = {};
  for (int k0 = 0; k0 < K; k0 += TK) {
    // ---- A tile -> As[k][m]
    if (!TA) {
      const int mm = tid >> 2, kk = (tid & 3) * 4;
      const long long m = m0 + mm;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int k = k0 + kk + j;
        As[kk + j][mm] = (m < M && k < K) ? A[m * lda + k] : 0.f;
      }
    } else {
      const int kk = tid >> 4, mm = (tid & 15) * 4;
      const int k = k0 + kk;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const long long m = m0 + mm + j;
        As[kk][mm + j] = (m < M && k < K) ? A[static_cast<long long>(k) * lda + m] : 0.f;
      }
    }
    // ---- B tile -> Bs[k][n]
    if (!TB) {
      const int kk = tid >> 4, nn = (tid & 15) * 4;
      const int k = k0 + kk;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int n = n0 + nn + j;
        Bs[kk][nn + j] = (n < N && k < K) ? B[static_cast<long long>(k) * ldb + n] : 0.f;
      }
    } else {
      const int nn = tid >> 2, kk = (tid & 3) * 4;
      const int n = n0 + nn;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int k = k0 + kk + j;
        Bs[kk + j][nn] = (n < N && k < K) ? B[static_cast<long long>(n) * ldb + k] : 0.f;
      }
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < TK; ++k) {
      const float4 a4 = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
      const float4 b4 = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
      const float a[4] = {a4.x, a4.y, a4.z, a4.w};
      const float b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
  const float alpha = e.alpha * (e.alpha_dev ? *e.alpha_dev : 1.f);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long long m = m0 + ty * 4 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= N) continue;
      float v = alpha * acc[i][j];
      if (e.beta != 0.f) v += e.beta * C[m * ldc + n];
      if (e.bias) v += e.bias[n];
      if (e.relu) v = fmaxf(v, 0.f);
      if (e.res) v += e.res[m * ldc + n];
      C[m * ldc + n] = v;
    }
  }
}

int sgemm(bool ta, bool tb, int64_t M, int N, int K, const float* A, int lda, const float* B, int ldb, float* C,
          int ldc, const Epilogue& e, cudaStream_t st) {
  if (M == 0 || N == 0) return P3D_OK;
  dim3 grid((N + TN - 1) / TN, static_cast<unsigned>((M + TM - 1) / TM));
  P3D_REQUIRE(grid.y <= 65535u || true, "sgemm: M too large");
  // gridDim.y is limited to 65535: process in slabs of rows
  const int64_t slab = 65535ll * TM;
  for (int64_t r0 = 0; r0 < M; r0 += slab) {
    const int64_t mr = (M - r0 < slab) ? (M - r0) : slab;
    dim3 g((N + TN - 1) / TN, static_cast<unsigned>((mr + TM - 1) / TM));
    const float* Ar = ta ? A + r0 : A + r0 * lda;
    float* Cr = C + r0 * ldc;
    Epilogue er = e;
    if (er.res) er.res = e.res + r0 * ldc;
    if (!ta && !tb) sgemm_kernel<false, false><<<g, 256, 0, st>>>((int)mr, N, K, Ar, lda, B, ldb, Cr, ldc, er);
    else if (!ta && tb) sgemm_kernel<false, true><<<g, 256, 0, st>>>((int)mr, N, K, Ar, lda, B, ldb, Cr, ldc, er);
    else if (ta && !tb) sgemm_kernel<true, false><<<g, 256, 0, st>>>((int)mr, N, K, Ar, lda, B, ldb, Cr, ldc, er);
    else sgemm_kernel<true, true><<<g, 256, 0, st>>>((int)mr, N, K, Ar, lda, B, ldb, Cr, ldc, er);
    P3D_LAUNCH_CHECK();
  }
  return P3D_OK;
}

// fp32 activations P | Q of at least `rows` rows each (m->f32_a, [2][f32_cap][L])
static int ensure_f32(p3d_model* m, int64_t rows, cudaStream_t st) {
  if (m->f32_cap >= rows) return P3D_OK;
  P3D_TRY(refuse_in_capture(st, "forward: growing the fp32 activation buffers"));
  const int64_t cap = grown_cap(m, m->f32_cap, rows);
  retire(m, m->f32_a);
  m->f32_a = nullptr; m->f32_cap = 0;
  P3D_CUDA(cudaMalloc(&m->f32_a, sizeof(float) * 2ull * cap * m->L));
  m->f32_cap = cap;
  return P3D_OK;
}

// fp32-mode inference through the folded fp32 weights; activations in two [cap,L] fp32 buffers
int forward_fp32(p3d_model* m, const float* x, float* y, int64_t B, cudaStream_t st) {
  const int L = m->L;
  P3D_TRY(ensure_f32(m, B, st));
  float* P = m->f32_a;
  float* Q = m->f32_a + static_cast<size_t>(m->f32_cap) * L;
  const int nl = static_cast<int>(m->layers.size());
  for (int l = 0; l < nl; ++l) {
    const Layer& ly = m->layers[l];
    Epilogue e;
    e.bias = m->bias_fold + ly.row_off;
    const float* W = m->wfold + ly.off_wfold;
    if (l == nl - 1) {
      P3D_TRY(sgemm(false, false, B, ly.N, ly.K, P, L, W, ly.N, y, ly.N, e, st));
    } else if (l == 0) {
      e.relu = 1;
      P3D_TRY(sgemm(false, false, B, ly.N, ly.K, x, kIn, W, ly.N, P, L, e, st));
    } else if (l & 1) {
      e.relu = 1;
      P3D_TRY(sgemm(false, false, B, ly.N, ly.K, P, L, W, ly.N, Q, L, e, st));
    } else {
      e.relu = 1;
      if (m->cfg.residual) e.res = P;       // in-place: each element is read (res) then written by one thread
      P3D_TRY(sgemm(false, false, B, ly.N, ly.K, Q, L, W, ly.N, P, L, e, st));
    }
  }
  return P3D_OK;
}

// ----------------------------------------------------------------------------- small batch
// Latency path (the batch-1 loop of src/openpose_3dpose_sandbox_realtime.py:50-168): one launch per
// layer, one warp per output feature, bf16 K-major weights streamed once, fp32 activations.
// Handles up to SB_ROWS rows per launch.
constexpr int SB_ROWS = 8;

template <int ROWS>
__global__ void __launch_bounds__(256) small_batch_layer_kernel(const float* __restrict__ hin, int ldin, int K,
                                                                const __nv_bfloat16* __restrict__ wt, int kpad,
                                                                const float* __restrict__ bias, int N, int relu,
                                                                const float* res, float* hout, int ldout, int rows) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= N) return;
  const __nv_bfloat16* wrow = wt + static_cast<size_t>(warp) * kpad;
  float acc[ROWS];
#pragma unroll
  for (int r = 0; r < ROWS; ++r) acc[r] = 0.f;
  for (int k = lane * 8; k < K; k += 256) {
    if (k + 8 > K) {       // the ragged tail of a width that is not a multiple of 8 (kpad is): element by element
#pragma unroll
      for (int r = 0; r < ROWS; ++r)
        if (r < rows)
          for (int i = 0; i < K - k; ++i) acc[r] = fmaf(hin[static_cast<size_t>(r) * ldin + k + i], __bfloat162float(wrow[k + i]), acc[r]);
      continue;
    }
    const uint4 wv = __ldg(reinterpret_cast<const uint4*>(wrow + k));
    const __nv_bfloat162* w2 = reinterpret_cast<const __nv_bfloat162*>(&wv);
    float w[8];
#pragma unroll
    for (int i = 0; i < 4; ++i) { w[2 * i] = __low2float(w2[i]); w[2 * i + 1] = __high2float(w2[i]); }
#pragma unroll
    for (int r = 0; r < ROWS; ++r) {
      if (r < rows) {
        const float4 a = *reinterpret_cast<const float4*>(hin + static_cast<size_t>(r) * ldin + k);
        const float4 b = *reinterpret_cast<const float4*>(hin + static_cast<size_t>(r) * ldin + k + 4);
        acc[r] = fmaf(a.x, w[0], acc[r]); acc[r] = fmaf(a.y, w[1], acc[r]);
        acc[r] = fmaf(a.z, w[2], acc[r]); acc[r] = fmaf(a.w, w[3], acc[r]);
        acc[r] = fmaf(b.x, w[4], acc[r]); acc[r] = fmaf(b.y, w[5], acc[r]);
        acc[r] = fmaf(b.z, w[6], acc[r]); acc[r] = fmaf(b.w, w[7], acc[r]);
      }
    }
  }
#pragma unroll
  for (int r = 0; r < ROWS; ++r) {
    float v = acc[r];
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0 && r < rows) {
      v += bias[warp];
      if (relu) v = fmaxf(v, 0.f);
      if (res) v += res[static_cast<size_t>(r) * ldout + warp];
      hout[static_cast<size_t>(r) * ldout + warp] = v;
    }
  }
}

// Latency path, one launch: a cooperative persistent kernel walks all layers; the grid synchronises between
// layers with a monotonic global counter (no reset needed: the host passes a per-launch epoch).  The bf16
// weight row of the NEXT layer is prefetched into registers before the barrier, so a layer costs one barrier
// plus one L2 round trip for the activations.
struct LatArgs {
  const float* x; float* y; const __nv_bfloat16* wt; const float* bias; float* hP; float* hQ;
  unsigned long long* counter; unsigned long long base;   // barrier counter value at kernel entry
  unsigned long long* stamps;                              // optional [16] globaltimer stamps (debug)
  int rows, L, nlayers, out, kpad, residual;
  rt::Fused rt;                                            // realtime front-end / back-end fused into the cluster kernel
};

__device__ __forceinline__ void grid_barrier(unsigned long long* counter, unsigned long long target) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    atomicAdd(counter, 1ull);
    unsigned spins = 0;
    while (*reinterpret_cast<volatile unsigned long long*>(counter) < target) {
      if (++spins > (1u << 26)) { printf("p3d: grid barrier timeout block=%d\n", (int)blockIdx.x); __trap(); }
    }
    __threadfence();
  }
  __syncthreads();
}

template <int ROWS, int KW, int NT>   // KW = uint4 weight words per lane = K / 256, NT = threads per block
__global__ void __launch_bounds__(NT) latency_forward_kernel(const LatArgs a) {
  const int lane = threadIdx.x & 31;
  const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
  const int L = a.L;
  uint4 wreg[KW];
  // layer 0 weights (K = 32 -> lanes 0..3)
  {
    const int n = gw;
    if (n < L && lane < 4) wreg[0] = __ldg(reinterpret_cast<const uint4*>(a.wt + static_cast<size_t>(n) * a.kpad + lane * 8));
  }
  unsigned long long target = a.base;
  int row_off = 0;
  for (int l = 0; l < a.nlayers; ++l) {
    const bool first = (l == 0), last = (l == a.nlayers - 1);
    const int K = first ? kIn : L, N = last ? a.out : L;
    const float* hin = first ? a.x : ((l & 1) ? a.hP : a.hQ);
    const int ldin = first ? kIn : L;
    float* hout = last ? a.y : ((first || !(l & 1)) ? a.hP : a.hQ);
    const int ldout = last ? a.out : L;
    const float* res = (!last && a.residual && l >= 2 && !(l & 1)) ? a.hP : nullptr;
    for (int n = gw; n < N; n += nw) {
      if (n != gw) {       // rows beyond the prefetched one (only when N > number of warps)
        const __nv_bfloat16* wrow = a.wt + static_cast<size_t>(row_off + n) * a.kpad;
#pragma unroll
        for (int i = 0; i < KW; ++i) if (lane * 8 + i * 256 < K) wreg[i] = __ldg(reinterpret_cast<const uint4*>(wrow + lane * 8 + i * 256));
      }
      float acc[ROWS];
#pragma unroll
      for (int r = 0; r < ROWS; ++r) acc[r] = 0.f;
#pragma unroll
      for (int i = 0; i < KW; ++i) {
        const int k = lane * 8 + i * 256;
        if (k < K) {
          const __nv_bfloat162* w2 = reinterpret_cast<const __nv_bfloat162*>(&wreg[i]);
          float w[8];
#pragma unroll
          for (int j = 0; j < 4; ++j) { w[2 * j] = __low2float(w2[j]); w[2 * j + 1] = __high2float(w2[j]); }
#pragma unroll
          for (int r = 0; r < ROWS; ++r) {
            if (r < a.rows) {
              const float4 u = __ldcg(reinterpret_cast<const float4*>(hin + static_cast<size_t>(r) * ldin + k));
              const float4 v = __ldcg(reinterpret_cast<const float4*>(hin + static_cast<size_t>(r) * ldin + k + 4));
              acc[r] = fmaf(u.x, w[0], acc[r]); acc[r] = fmaf(u.y, w[1], acc[r]); acc[r] = fmaf(u.z, w[2], acc[r]); acc[r] = fmaf(u.w, w[3], acc[r]);
              acc[r] = fmaf(v.x, w[4], acc[r]); acc[r] = fmaf(v.y, w[5], acc[r]); acc[r] = fmaf(v.z, w[6], acc[r]); acc[r] = fmaf(v.w, w[7], acc[r]);
            }
          }
        }
      }
#pragma unroll
      for (int r = 0; r < ROWS; ++r) {
        float v = acc[r];
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0 && r < a.rows) {
          v += __ldg(a.bias + row_off + n);
          if (!last) v = fmaxf(v, 0.f);
          if (res) v += __ldcg(res + static_cast<size_t>(r) * ldout + n);
          __stcg(hout + static_cast<size_t>(r) * ldout + n, v);
        }
      }
    }
    row_off += N;
    if (last) break;
    // prefetch my first weight row of the next layer, then synchronise the grid
    {
      const int Nn = (l + 1 == a.nlayers - 1) ? a.out : L;
      if (gw < Nn) {
        const __nv_bfloat16* wrow = a.wt + static_cast<size_t>(row_off + gw) * a.kpad;
#pragma unroll
        for (int i = 0; i < KW; ++i) wreg[i] = __ldg(reinterpret_cast<const uint4*>(wrow + lane * 8 + i * 256));
      }
    }
    target += gridDim.x;
    grid_barrier(a.counter, target);
  }
}

template <int ROWS, int KW, int NT>
static int launch_latency(p3d_model* m, LatArgs& a, cudaStream_t st) {
  static int grid = 0, coop = 1;
  if (!grid) {
    int per_sm = 0;
    P3D_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, latency_forward_kernel<ROWS, KW, NT>, NT, 0));
    P3D_REQUIRE(per_sm >= 1, "latency kernel does not fit on an SM");
    // enough warps for one output feature each (L warps), never more blocks than SMs (all must be co-resident)
    grid = (a.L * 32 + NT - 1) / NT;
    if (grid > m->num_sms) grid = m->num_sms;
    if (const char* e = getenv("P3D_LAT_GRID")) { const int g = atoi(e); if (g >= 1 && g <= m->num_sms) grid = g; }
    if (const char* e = getenv("P3D_LAT_COOP")) coop = atoi(e);
  }
  a.base = m->lat_base;
  m->lat_base += static_cast<unsigned long long>(grid) * (a.nlayers - 1);
  if (coop) {
    void* params[] = {&a};
    P3D_CUDA(cudaLaunchCooperativeKernel(reinterpret_cast<void*>(latency_forward_kernel<ROWS, KW, NT>), dim3(grid), dim3(NT), params, 0, st));
  } else {
    latency_forward_kernel<ROWS, KW, NT><<<grid, NT, 0, st>>>(a);
  }
  P3D_LAUNCH_CHECK();
  return P3D_OK;
}

int forward_latency(p3d_model* m, const float* x, float* y, int64_t B, cudaStream_t st) {
  const int L = m->L;
  P3D_TRY(ensure_f32(m, SB_ROWS, st));
  for (int64_t r0 = 0; r0 < B; r0 += SB_ROWS) {
    LatArgs a;
    a.rows = static_cast<int>(B - r0 < SB_ROWS ? B - r0 : SB_ROWS);
    a.x = x + r0 * kIn; a.y = y + r0 * m->out_size; a.wt = m->wt_bf16; a.bias = m->bias_fold;
    a.hP = m->f32_a; a.hQ = m->f32_a + static_cast<size_t>(m->f32_cap) * L;
    a.counter = m->lat_counter; a.stamps = nullptr; a.L = L; a.nlayers = static_cast<int>(m->layers.size()); a.out = m->out_size;
    a.kpad = m->kpad; a.residual = m->cfg.residual;
    static int nt = 0;
    if (!nt) { const char* e = getenv("P3D_LAT_THREADS"); nt = e ? atoi(e) : 1024; }
    if (a.rows == 1) {
      if (nt == 256) P3D_TRY((launch_latency<1, 4, 256>(m, a, st)));
      else if (nt == 512) P3D_TRY((launch_latency<1, 4, 512>(m, a, st)));
      else P3D_TRY((launch_latency<1, 4, 1024>(m, a, st)));
    } else {
      if (nt == 256) P3D_TRY((launch_latency<SB_ROWS, 4, 256>(m, a, st)));
      else P3D_TRY((launch_latency<SB_ROWS, 4, 512>(m, a, st)));
    }
  }
  return P3D_OK;
}

// ----------------------------------------------------------------------------- batch-1 cluster kernel
// One 16-CTA thread-block cluster (non-portable size) serves a single pose: every CTA owns 1/16 of each
// layer's output features, keeps the FULL activation vector in its own shared memory and pushes its 64 results
// into all 16 CTAs' shared memory (st.shared::cluster), followed by a hardware cluster barrier (~0.3 us instead
// of ~3 us of L2 round trips for a grid-wide barrier).
// Weights: the CTA's slice of a hidden layer is 64 rows x 2 KB = two contiguous 64 KB halves (one output per
// warp each).  They are streamed by TMA bulk copies (cp.async.bulk) into a 3-slot shared-memory ring that is
// kept full from the first instruction on, so the 512 KB per CTA cross L2->SM exactly once at the SM's full
// ingest rate, off the critical path of the layer chain.  L = 1024 only.
constexpr int LC = 16;            // cluster size
constexpr int LNT = 512;          // threads per CTA (16 warps, 4 output features per warp and layer)
constexpr int LNW = LNT / 32;
constexpr int LOPW = 64 / LNW;    // outputs per warp per layer
constexpr int LSLOTS = 6;
constexpr int LPART_BYTES = LNW * 1024 * 2;    // one ring slot: LNW rows x 1024 bf16 = 32 KB
constexpr int LAT_SMEM = LSLOTS * LPART_BYTES + 1024;

__device__ __forceinline__ uint32_t cl_rank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cl_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void st_cluster_f32(float* local, uint32_t cta, float v) {
  const uint32_t la = static_cast<uint32_t>(__cvta_generic_to_shared(local));
  asm volatile("{\n\t.reg .b32 ra;\n\tmapa.shared::cluster.u32 ra, %0, %1;\n\tst.shared::cluster.f32 [ra], %2;\n\t}"
               ::"r"(la), "r"(cta), "f"(v) : "memory");
}
__device__ __forceinline__ uint32_t sm_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void lat_mbar_init(uint64_t* b, uint32_t n) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(sm_u32(b)), "r"(n) : "memory"); }
__device__ __forceinline__ void lat_mbar_arrive(uint64_t* b) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(sm_u32(b)) : "memory"); }
__device__ __forceinline__ void lat_mbar_wait(uint64_t* b, uint32_t parity) {
  uint32_t ok = 0, spins = 0;
  while (!ok) {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(sm_u32(b)), "r"(parity) : "memory");
    if (!ok && ++spins > (1u << 26)) { printf("p3d: latency kernel mbarrier timeout\n"); __trap(); }
  }
}
// 1D bulk copy global -> shared, completion (bytes) signalled on an mbarrier.  The copy is issued as `pieces`
// independent bulk operations: one operation has a small window of outstanding L2 requests (measured ~30 GB/s
// per SM for a single 64 KB copy), many in flight reach the SM's ingest rate.
__device__ __forceinline__ void bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar, int pieces = 16) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(sm_u32(bar)), "r"(bytes) : "memory");
  const uint32_t pb = bytes / pieces;
  for (int i = 0; i < pieces; ++i)
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(sm_u32(dst) + i * pb), "l"(reinterpret_cast<const uint8_t*>(src) + static_cast<size_t>(i) * pb), "r"(pb), "r"(sm_u32(bar)) : "memory");
}

__device__ __forceinline__ unsigned long long gtimer() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
#define LAT_STAMP(i) do { if (a.stamps && threadIdx.x == 0 && rank == 0) a.stamps[i] = gtimer(); } while (0)

template <bool F16 = false>     // F16: fp16 weights (P3D_MODE_FP16)
__global__ void __launch_bounds__(LNT, 1) latency_cluster_kernel(const LatArgs a) {
  using O = Op16<F16>;
  constexpr int L = 1024;
  extern __shared__ __align__(128) uint8_t lat_smem[];
  __shared__ __align__(16) float sP[L];
  __shared__ __align__(16) float sQ[L];
  __shared__ uint64_t wfull[LSLOTS], wfree[LSLOTS];
  uint8_t* ring = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(lat_smem) + 127) & ~uintptr_t(127));
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t rank = cl_rank();
  LAT_STAMP(0);
  const int nhid = a.nlayers - 2;                 // hidden layers with L x L weights (layers 1 .. nlayers-2)
  const int nparts = LOPW * nhid;                 // part p = (layer 1 + p/LOPW, o = p%LOPW); rows n = rank*64 + o*LNW + warp
  auto part_src = [&](int p) {
    const int l = 1 + p / LOPW, o = p % LOPW;
    return a.wt + (static_cast<size_t>(l) * L + rank * 64 + o * LNW) * a.kpad;
  };
  if (threadIdx.x == 0) {
    for (int s = 0; s < LSLOTS; ++s) { lat_mbar_init(&wfull[s], 1); lat_mbar_init(&wfree[s], LNW); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    for (int p = 0; p < LSLOTS && p < nparts; ++p) bulk_load(ring + p * LPART_BYTES, part_src(p), LPART_BYTES, &wfull[p], 4);
  }
  // x -> sQ[0..31] (layer 0 reads "Q"); layer 0 weights (K = 32: lanes 0..7, 4 bf16 each) straight from L2
  if (a.rt.tab == nullptr) {
    if (threadIdx.x < kIn) sQ[threadIdx.x] = __ldg(a.x + threadIdx.x);
  } else {
    // realtime step: keypoints (one coalesced read of 36 doubles per CTA, possibly across PCIe from mapped host
    // memory) -> H3.6M order, synthesised hip / neck / thorax, (x - mu) / sigma in fp64, fp32 feed
    double* skp = reinterpret_cast<double*>(sQ + 64);      // scratch no other CTA writes before the first cluster barrier
    if (threadIdx.x < 36) skp[threadIdx.x] = *reinterpret_cast<const volatile double*>(a.rt.kp + threadIdx.x);
    __syncthreads();
    if (threadIdx.x < kIn) {
      const rt::Tables* tb = a.rt.tab;
      const double v = (openpose_h36m_coord(skp, tb->use2[threadIdx.x]) - tb->mu2[threadIdx.x]) / tb->sd2[threadIdx.x];
      const float vf = static_cast<float>(v);
      sQ[threadIdx.x] = vf;
      if (rank == 0 && a.rt.enc) a.rt.enc[threadIdx.x] = vf;
    }
  }
  uint2 w0[LOPW]; float b0[LOPW];
#pragma unroll
  for (int o = 0; o < LOPW; ++o) {
    const int n = static_cast<int>(rank) * 64 + o * LNW + warp;
    w0[o] = make_uint2(0, 0);
    if (lane < 8) w0[o] = __ldg(reinterpret_cast<const uint2*>(a.wt + static_cast<size_t>(n) * a.kpad + lane * 4));
    b0[o] = __ldg(a.bias + n);
  }
  float bias_next[LOPW];       // biases of the next hidden layer, fetched a layer ahead
#pragma unroll
  for (int o = 0; o < LOPW; ++o) bias_next[o] = (nhid > 0) ? __ldg(a.bias + L + rank * 64 + o * LNW + warp) : 0.f;
  __syncthreads();

  // ---- layer 0 (reads x in sQ, writes sP)
  {
    float hv4[4] = {0.f, 0.f, 0.f, 0.f};
    if (lane < 8) { const float4 h = *reinterpret_cast<const float4*>(sQ + lane * 4); hv4[0] = h.x; hv4[1] = h.y; hv4[2] = h.z; hv4[3] = h.w; }
#pragma unroll
    for (int o = 0; o < LOPW; ++o) {
      const typename O::T2* w2 = reinterpret_cast<const typename O::T2*>(&w0[o]);
      float acc = hv4[0] * O::lo(w2[0]) + hv4[1] * O::hi(w2[0]) + hv4[2] * O::lo(w2[1]) + hv4[3] * O::hi(w2[1]);
      for (int s = 16; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
      const float v = fmaxf(acc + b0[o], 0.f);
      if (lane < LC) st_cluster_f32(sP + rank * 64 + o * LNW + warp, static_cast<uint32_t>(lane), v);
    }
    cl_sync();
  }
  LAT_STAMP(1);
  // ---- hidden layers: activations in registers for the whole layer, weights from the smem ring
  int p = 0;
  for (int l = 1; l <= nhid; ++l) {
    const float* src = (l & 1) ? sP : sQ;
    float* dst = (l & 1) ? sQ : sP;
    const bool add_res = a.residual && l >= 2 && !(l & 1);
    float4 hreg[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) hreg[i] = *reinterpret_cast<const float4*>(src + i * 128 + lane * 4);
    float bias[LOPW];
#pragma unroll
    for (int o = 0; o < LOPW; ++o) bias[o] = bias_next[o];
    if (l < nhid) {
#pragma unroll
      for (int o = 0; o < LOPW; ++o) bias_next[o] = __ldg(a.bias + (l + 1) * L + rank * 64 + o * LNW + warp);
    }
#pragma unroll 1
    for (int o = 0; o < LOPW; ++o, ++p) {
      const int slot = p % LSLOTS;
      const int n = static_cast<int>(rank) * 64 + o * LNW + warp;
      lat_mbar_wait(&wfull[slot], (p / LSLOTS) & 1);
      const uint2* wrow = reinterpret_cast<const uint2*>(ring + slot * LPART_BYTES + warp * 2048);
      float acc0 = 0.f, acc1 = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const uint2 wv = wrow[i * 32 + lane];                         // k = i*128 + lane*4 .. +3 : conflict-free
        const typename O::T2* w2 = reinterpret_cast<const typename O::T2*>(&wv);
        acc0 = fmaf(hreg[i].x, O::lo(w2[0]), acc0); acc1 = fmaf(hreg[i].y, O::hi(w2[0]), acc1);
        acc0 = fmaf(hreg[i].z, O::lo(w2[1]), acc0); acc1 = fmaf(hreg[i].w, O::hi(w2[1]), acc1);
      }
      __syncwarp();
      if (lane == 0) lat_mbar_arrive(&wfree[slot]);                   // this warp is done with the slot
      float acc = acc0 + acc1;
      for (int s = 16; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
      float v = fmaxf(acc + (o == 0 ? bias[0] : o == 1 ? bias[1] : o == 2 ? bias[2] : bias[3]), 0.f);
      if (add_res) v += sP[n];
      if (lane < LC) st_cluster_f32(dst + n, static_cast<uint32_t>(lane), v);
      // refill the slot with part p+LSLOTS as soon as all warps have released it
      if (threadIdx.x == 0 && p + LSLOTS < nparts) {
        lat_mbar_wait(&wfree[slot], (p / LSLOTS) & 1);
        bulk_load(ring + slot * LPART_BYTES, part_src(p + LSLOTS), LPART_BYTES, &wfull[slot], 4);
      }
      __syncwarp();
    }
    cl_sync();                                                        // layer complete everywhere
    LAT_STAMP(1 + l);
  }
  // ---- output layer: feature g = rank*LNW + warp < out, weights straight from L2
  {
    const int l = a.nlayers - 1;
    const int g = static_cast<int>(rank) * LNW + warp;
    if (g < a.out) {
      const float* src = (l & 1) ? sP : sQ;
      const __nv_bfloat16* wrow = a.wt + (static_cast<size_t>(l) * L + g) * a.kpad;
      float acc = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const uint2 wv = __ldg(reinterpret_cast<const uint2*>(wrow + i * 128 + lane * 4));
        const float4 hv = *reinterpret_cast<const float4*>(src + i * 128 + lane * 4);
        const typename O::T2* w2 = reinterpret_cast<const typename O::T2*>(&wv);
        acc = fmaf(hv.x, O::lo(w2[0]), acc); acc = fmaf(hv.y, O::hi(w2[0]), acc);
        acc = fmaf(hv.z, O::lo(w2[1]), acc); acc = fmaf(hv.w, O::hi(w2[1]), acc);
      }
      for (int s = 16; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
      if (lane == 0) {
        const float yv = acc + __ldg(a.bias + l * L + g);
        a.y[g] = yv;
        if (a.rt.tab) {                                    // data_utils.unNormalizeData (:299-311): fp32 value, fp64 scale
          const int j = a.rt.tab->use3[g];
          a.rt.pose[j] = __dadd_rn(__dmul_rn(static_cast<double>(yv), a.rt.tab->sd3[j]), a.rt.tab->mu3[j]);
        }
      }
    }
  }
  if (a.rt.flag) {
    // every output store is ordered before the cluster barrier (release) and the flag store after it (acquire +
    // system-scope release): a host that polls the mapped flag sees complete outputs without a stream synchronise
    cl_sync();
    if (rank == 0 && threadIdx.x == 0)
      asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(a.rt.flag), "l"(a.rt.seq) : "memory");
  }
  LAT_STAMP(a.nlayers);
}

static int launch_latency_cluster(p3d_model* m, const float* x, float* y, const rt::Fused* f, cudaStream_t st) {
  // per device: the attributes live in the device's context and the cluster may be schedulable on one GPU only
  static int ok_dev[64] = {0};                      // 0 = not probed yet, 1 = usable, 2 = not usable
  int& okd = ok_dev[m->cfg.device & 63];
  int ok = okd == 1 ? 1 : (okd == 2 ? 0 : -1);
  if (ok < 0) {
    P3D_TRY(refuse_in_capture(st, "forward: probing the 16-CTA cluster kernel"));
    ok = 0;
    if (cudaFuncSetAttribute(latency_cluster_kernel<false>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess &&
        cudaFuncSetAttribute(latency_cluster_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, LAT_SMEM) == cudaSuccess &&
        cudaFuncSetAttribute(latency_cluster_kernel<true>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess &&
        cudaFuncSetAttribute(latency_cluster_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, LAT_SMEM) == cudaSuccess) {
      cudaLaunchConfig_t cfg{};
      cfg.gridDim = dim3(LC); cfg.blockDim = dim3(LNT); cfg.dynamicSmemBytes = LAT_SMEM;
      cudaLaunchAttribute attr[1];
      attr[0].id = cudaLaunchAttributeClusterDimension; attr[0].val.clusterDim.x = LC; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
      cfg.attrs = attr; cfg.numAttrs = 1;
      int nclusters = 0;
      if (cudaOccupancyMaxActiveClusters(&nclusters, latency_cluster_kernel<false>, &cfg) == cudaSuccess && nclusters >= 1) ok = 1;
    }
    cudaGetLastError();
    if (const char* e = getenv("P3D_LAT_CLUSTER")) ok = ok && atoi(e);
    okd = ok ? 1 : 2;
  }
  if (!ok || m->layers.size() < 3) return 1;       // caller falls back to the per-layer kernels
  LatArgs a;
  if (f) a.rt = *f;
  a.rows = 1; a.x = x; a.y = y; a.wt = m->wt_bf16; a.bias = m->bias_fold; a.hP = a.hQ = nullptr; a.counter = nullptr; a.base = 0;
  a.stamps = getenv("P3D_LAT_STAMPS") ? m->lat_counter + 8 : nullptr;
  a.L = m->L; a.nlayers = static_cast<int>(m->layers.size()); a.out = m->out_size; a.kpad = m->kpad; a.residual = m->cfg.residual;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(LC); cfg.blockDim = dim3(LNT); cfg.dynamicSmemBytes = LAT_SMEM; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension; attr[0].val.clusterDim.x = LC; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  if (m->cfg.mode == P3D_MODE_FP16) P3D_CUDA(cudaLaunchKernelEx(&cfg, latency_cluster_kernel<true>, a));
  else P3D_CUDA(cudaLaunchKernelEx(&cfg, latency_cluster_kernel<false>, a));
  P3D_LAUNCH_CHECK();
  return P3D_OK;
}


// ----------------------------------------------------------------------------- batch-1 whole-chip kernel
// The 16-CTA cluster kernel above streams 512 KB of weights per SM; it is bound by what ONE SM can ingest (measured:
// 3.2-4.1 us per hidden layer = ~37 GB/s per SM, 19 us in the kernel, 16 of 148 SMs busy).  Here 128 CTAs (cooperative
// launch: all resident) own 8 output features of every layer each: a CTA's whole share of the weights is 64 KB and is
// requested in the first instructions (the chip pulls the 8.56 MB in parallel, ~2 us), so what remains is the layer
// chain itself.  Activations travel between the layers through a global buffer of self-validating words {fp32 value,
// launch tag}: a producer stores its feature with one 8-byte store, every consumer polls the words it needs until they
// carry this launch's tag - no counter, no fence, no barrier: one L2 write + read per layer (~1 us) instead of the
// ~3 us round trips of a grid-wide barrier.  The tag comes from the model's epoch word in device memory (xchg_tag in
// common.cuh), which every launch advances on its way out, so the buffer is never cleared and a launch captured into a
// CUDA graph gets a fresh tag on every replay.
constexpr int GLC = 128;          // CTAs
constexpr int GLT = 256;          // threads: 8 warps, one output feature per warp and layer
constexpr int GLF = GLT / 32;     // features per CTA and layer
struct GridLatArgs {
  const float* x; float* y; const __nv_bfloat16* wt; const float* bias;
  uint2* act;                     // [nlayers - 1][8 poses][1024] {value bits, tag}
  unsigned* xchg;                 // epoch + arrival counter (p3d_model::xchg)
  int nlayers, out, kpad, residual, rows, backoff_ns;
  unsigned long long* stamps;
};
__device__ __forceinline__ void st_ll(uint2* p, float v, unsigned tag) {
  asm volatile("st.volatile.global.v2.u32 [%0], {%1, %2};" ::"l"(p), "r"(__float_as_uint(v)), "r"(tag) : "memory");
}
__device__ __forceinline__ uint4 ld_ll2(const uint2* p) {
  uint4 v;
  asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
  return v;
}
#define GLAT_STAMP(i) do { if (a.stamps && threadIdx.x == 0 && blockIdx.x == 0) a.stamps[i] = gtimer(); } while (0)

template <int ROWS, bool F16 = false>      // poses served by one launch (1, 2, 4 or 8; a.rows <= ROWS of them are live); F16: fp16 weights
__global__ void __launch_bounds__(GLT, 1) latency_grid_kernel(const GridLatArgs a) {
  using O = Op16<F16>;
  constexpr int L = 1024;
  extern __shared__ __align__(128) uint8_t glat_smem[];
  const int c = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nhid = a.nlayers - 2;
  uint8_t* wsm = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(glat_smem) + 127) & ~uintptr_t(127));
  uint8_t* wout = wsm + nhid * (GLF * 2048);                        // this CTA's row of the output layer (c < out)
  float* sP = reinterpret_cast<float*>(wout + 2048);                // [ROWS][L]
  float* sQ = sP + ROWS * L;
  uint64_t* wbar = reinterpret_cast<uint64_t*>(sQ + ROWS * L);     // [nhid + 1]
  GLAT_STAMP(0);
  const unsigned tag = xchg_tag(a.xchg);                            // in flight with the weight copies; first used by layer 0's publish
  unsigned arrived = 0;                                             // thread 0: CTAs that arrived before this one
  if (threadIdx.x == 0) {
    for (int l = 0; l <= nhid; ++l) lat_mbar_init(&wbar[l], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    // the CTA's 8 rows of a hidden layer are contiguous in the packed weights: 16 KB per layer, everything requested now
    for (int l = 0; l < nhid; ++l)
      bulk_load(wsm + l * (GLF * 2048), a.wt + (static_cast<size_t>(1 + l) * L + c * GLF) * a.kpad, GLF * 2048, &wbar[l], 4);
    if (c < a.out) bulk_load(wout, a.wt + (static_cast<size_t>(a.nlayers - 1) * L + c) * a.kpad, 2048, &wbar[nhid], 1);
  }
  const int n = c * GLF + warp;                                     // this warp's feature of every hidden layer
  // Layer l's outputs of pose r live in ONE shared copy that every CTA polls (pull).  Measured alternatives: a private inbox
  // per consumer CTA that the producers write to (push: 128 scattered 8-byte stores per feature) was slower (23 us per
  // call against 13-18); so were 8-byte stores from eight different warps into the shared copy - partial-sector writes into
  // lines that 512 threads are polling.  A CTA therefore collects its eight features in shared memory and publishes them
  // as ONE 64-byte row of four 16-byte stores (two whole sectors).
  auto word = [&](int l, int r) { return a.act + (static_cast<size_t>(l) * 8 + r) * L; };
  __shared__ float spub[ROWS][GLF];
  auto publish_cta = [&](int l) {                                 // after a block barrier: spub holds the CTA's features
    if (threadIdx.x < 4 * ROWS) {
      const int r = threadIdx.x >> 2, q = threadIdx.x & 3;
      if (r < a.rows) {
        uint2* dst = word(l, r) + c * GLF + 2 * q;
        asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "r"(__float_as_uint(spub[r][2 * q])), "r"(tag),
                     "r"(__float_as_uint(spub[r][2 * q + 1])), "r"(tag) : "memory");
      }
    }
  };
  // ---- layer 0 (K = 32): weights and x straight from L2
  {
    uint2 wv = make_uint2(0, 0);
    if (lane < 8) wv = __ldg(reinterpret_cast<const uint2*>(a.wt + static_cast<size_t>(n) * a.kpad + lane * 4));
    const typename O::T2* w2 = reinterpret_cast<const typename O::T2*>(&wv);
    const float b = __ldg(a.bias + n);
#pragma unroll
    for (int r = 0; r < ROWS; ++r) {
      float acc = 0.f;
      if (lane < 8 && r < a.rows) {
        const float4 h = __ldg(reinterpret_cast<const float4*>(a.x + r * kIn + lane * 4));
        acc = h.x * O::lo(w2[0]) + h.y * O::hi(w2[0]) + h.z * O::lo(w2[1]) + h.w * O::hi(w2[1]);
      }
      for (int s = 16; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
      if (lane == 0) spub[r][warp] = fmaxf(acc + b, 0.f);
    }
    __syncthreads();
    publish_cta(0);
  }
  GLAT_STAMP(1);
  // all of layer `lp`'s outputs -> dst (shared): every thread polls its own four words per pose until they carry the tag
  auto gather = [&](int lp, float* dst) {
    // the words of ALL poses are requested together and the batch is re-polled until every word carries the tag: one L2
    // round trip per poll (pose after pose, eight poses cost eight round trips per layer: 5.7 us)
    uint4 u[ROWS], v[ROWS];
    unsigned spins = 0;
    for (;;) {
      bool ok = true;
#pragma unroll
      for (int r = 0; r < ROWS; ++r) {
        const uint2* src = word(lp, r < a.rows ? r : 0) + threadIdx.x * 4;
        u[r] = ld_ll2(src); v[r] = ld_ll2(src + 2);
      }
#pragma unroll
      for (int r = 0; r < ROWS; ++r) ok = ok && u[r].y == tag && u[r].w == tag && v[r].y == tag && v[r].w == tag;
      if (ok) break;
      if (++spins > (1u << 24)) { printf("p3d: batch-1 kernel: layer %d never arrived (block %d)\n", lp, (int)blockIdx.x); __trap(); }
      // back off between polls: 32 K threads re-reading the same 8 KB as fast as they can keep the L2 slices that hold it
      // busy, and the producers' stores queue up behind the reads (per-layer times of 2-4.5 us instead of 1.5)
      if (a.backoff_ns > 0) __nanosleep(static_cast<unsigned>(a.backoff_ns));
    }
#pragma unroll
    for (int r = 0; r < ROWS; ++r)
      *reinterpret_cast<float4*>(dst + r * L + threadIdx.x * 4) =
          make_float4(__uint_as_float(u[r].x), __uint_as_float(u[r].z), __uint_as_float(v[r].x), __uint_as_float(v[r].z));
  };
  // ---- hidden layers: layer 0 and the even layers leave their outputs in P, the odd ones in Q (the residual of an even
  // layer is the block input, still in P when the layer computes)
  for (int l = 1; l <= nhid; ++l) {
    float* src = (l & 1) ? sP : sQ;
    const bool add_res = a.residual && l >= 2 && !(l & 1);
    const float bias = __ldg(a.bias + l * L + n);
    // every thread of the CTA has compared its tag in the first gather: arrive, while the outputs of layer 1 are on their way
    if (l == 2 && threadIdx.x == 0) arrived = xchg_arrive(a.xchg);
    gather(l - 1, src);
    __syncthreads();
    lat_mbar_wait(&wbar[l - 1], 0);
    const uint2* wrow = reinterpret_cast<const uint2*>(wsm + (l - 1) * (GLF * 2048) + warp * 2048);
    float acc0[ROWS], acc1[ROWS];
#pragma unroll
    for (int r = 0; r < ROWS; ++r) { acc0[r] = 0.f; acc1[r] = 0.f; }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const uint2 wv = wrow[i * 32 + lane];                         // k = i*128 + lane*4 .. +3 : conflict-free
      const typename O::T2* w2 = reinterpret_cast<const typename O::T2*>(&wv);
      const float w0 = O::lo(w2[0]), w1 = O::hi(w2[0]), w2f = O::lo(w2[1]), w3 = O::hi(w2[1]);
#pragma unroll
      for (int r = 0; r < ROWS; ++r) {
        const float4 h = *reinterpret_cast<const float4*>(src + r * L + i * 128 + lane * 4);
        acc0[r] = fmaf(h.x, w0, acc0[r]); acc1[r] = fmaf(h.y, w1, acc1[r]);
        acc0[r] = fmaf(h.z, w2f, acc0[r]); acc1[r] = fmaf(h.w, w3, acc1[r]);
      }
    }
#pragma unroll
    for (int r = 0; r < ROWS; ++r) {
      float acc = acc0[r] + acc1[r];
      for (int s = 16; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
      if (lane == 0) {
        float v = fmaxf(acc + bias, 0.f);
        if (add_res) v += sP[r * L + n];
        spub[r][warp] = v;
      }
    }
    __syncthreads();                                               // the next gather overwrites what this layer still reads
    publish_cta(l);
    GLAT_STAMP(1 + l);
  }
  // ---- output layer: CTA c < out computes feature c from its row in shared memory
  if (nhid < 2 && threadIdx.x == 0) arrived = xchg_arrive(a.xchg);
  if (c < a.out) {
    const int l = a.nlayers - 1;
    float* src = (l & 1) ? sP : sQ;
    gather(l - 1, src);
    __syncthreads();
    if (warp < ROWS && warp < a.rows) {                            // one pose per warp
      lat_mbar_wait(&wbar[nhid], 0);
      const uint2* wrow = reinterpret_cast<const uint2*>(wout);
      float acc = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const uint2 wv = wrow[i * 32 + lane];
        const float4 hv = *reinterpret_cast<const float4*>(src + warp * L + i * 128 + lane * 4);
        const typename O::T2* w2 = reinterpret_cast<const typename O::T2*>(&wv);
        acc = fmaf(hv.x, O::lo(w2[0]), acc); acc = fmaf(hv.y, O::hi(w2[0]), acc);
        acc = fmaf(hv.z, O::lo(w2[1]), acc); acc = fmaf(hv.w, O::hi(w2[1]), acc);
      }
      for (int s = 16; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
      if (lane == 0) a.y[warp * a.out + c] = acc + __ldg(a.bias + l * L + c);
    }
  }
  if (threadIdx.x == 0 && arrived == gridDim.x - 1) xchg_advance(a.xchg, tag);
  GLAT_STAMP(a.nlayers);
}

// returns 1 when the kernel cannot serve this model / device (the caller takes another path)
static int launch_latency_grid(p3d_model* m, const float* x, float* y, int rows, cudaStream_t st) {
  static const bool on = [] { const char* e = getenv("P3D_LAT_GRIDLL"); return !(e && e[0] == '0'); }();
  const int nlayers = static_cast<int>(m->layers.size()), nhid = nlayers - 2;
  if (!on || m->L != 1024 || nhid < 1 || nhid > 6 || m->out_size > GLC || m->num_sms < GLC || m->kpad != 1024 || rows < 1 || rows > 8) return 1;
  static const int rmin = [] { const char* e = getenv("P3D_LAT_RMIN"); return e ? atoi(e) : 1; }();      // diagnostics
  int R = rows == 1 ? 1 : (rows == 2 ? 2 : (rows <= 4 ? 4 : 8));
  if (R < rmin) R = rmin;
  const int smem = 128 + nhid * (GLF * 2048) + 2048 + 2 * R * 1024 * 4 + 8 * (nhid + 1) + 64;
  using K = void (*)(const GridLatArgs);
  const bool f16 = m->cfg.mode == P3D_MODE_FP16;
  const K fn = f16 ? (R == 1 ? latency_grid_kernel<1, true> : (R == 2 ? latency_grid_kernel<2, true> : (R == 4 ? latency_grid_kernel<4, true> : latency_grid_kernel<8, true>)))
                   : (R == 1 ? latency_grid_kernel<1> : (R == 2 ? latency_grid_kernel<2> : (R == 4 ? latency_grid_kernel<4> : latency_grid_kernel<8>)));
  if (!m->lat_act) return 1;                           // allocated (8 MB, zero) by p3d_model_create for width 1024 / bf16 / fp16
  static PerDeviceOnce attr;
  if (attr.needed()) {
    P3D_TRY(refuse_in_capture(st, "forward: first use of the whole-chip kernel on this device"));
    const int cap = 128 + 6 * (GLF * 2048) + 2048 + 2 * 8 * 1024 * 4 + 256;
    for (K k : {static_cast<K>(latency_grid_kernel<1>), static_cast<K>(latency_grid_kernel<2>), static_cast<K>(latency_grid_kernel<4>), static_cast<K>(latency_grid_kernel<8>),
                static_cast<K>(latency_grid_kernel<1, true>), static_cast<K>(latency_grid_kernel<2, true>), static_cast<K>(latency_grid_kernel<4, true>), static_cast<K>(latency_grid_kernel<8, true>)})
      P3D_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, cap));
    attr.mark();
  }
  GridLatArgs a;
  a.x = x; a.y = y; a.wt = m->wt_bf16; a.bias = m->bias_fold; a.act = static_cast<uint2*>(m->lat_act); a.xchg = m->xchg;
  a.nlayers = nlayers; a.out = m->out_size; a.kpad = m->kpad; a.residual = m->cfg.residual; a.rows = rows;
  static const int backoff = [] { const char* e = getenv("P3D_LAT_BACKOFF_NS"); return e ? atoi(e) : 0; }();
  a.backoff_ns = backoff;
  a.stamps = getenv("P3D_LAT_STAMPS") ? m->lat_counter + 8 : nullptr;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(GLC); cfg.blockDim = dim3(GLT); cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeCooperative; at[0].val.cooperative = 1;     // every CTA polls what the others produce
  cfg.attrs = at; cfg.numAttrs = 1;
  P3D_CUDA(cudaLaunchKernelEx(&cfg, fn, a));
  P3D_LAUNCH_CHECK();
  return P3D_OK;
}
// 2 .. 8 poses through the same kernel (fp32 activations, bf16 weights; 1 = not applicable here)
int forward_latency_grid(p3d_model* m, const float* x, float* y, int rows, cudaStream_t st) { return launch_latency_grid(m, x, y, rows, st); }

int forward_latency_cluster(p3d_model* m, const float* x, float* y, cudaStream_t st) {
  const int rc = launch_latency_grid(m, x, y, 1, st);       // the whole chip; 1 = not applicable here
  if (rc != 1) return rc;
  return launch_latency_cluster(m, x, y, nullptr, st);
}
// the same launch running the whole realtime step (keypoints -> normalised input -> lifter -> un-normalised pose).  It stays on
// the 16-CTA cluster kernel: fused into the whole-chip kernel (128 CTAs reading the keypoints from mapped host memory, 48
// output CTAs writing y / pose there behind system-scope fences and counting themselves) a frame took 181 us instead of 49.
int forward_latency_cluster_rt(p3d_model* m, const rt::Fused& f, float* y, cudaStream_t st) {
  if (m->L != 1024 || (m->cfg.mode != P3D_MODE_BF16 && m->cfg.mode != P3D_MODE_FP16)) return 1;
  return launch_latency_cluster(m, nullptr, y, &f, st);
}

int forward_small(p3d_model* m, const float* x, float* y, int64_t B, cudaStream_t st) {
  const int L = m->L;
  P3D_TRY(ensure_f32(m, SB_ROWS, st));
  float* P = m->f32_a;
  float* Q = m->f32_a + static_cast<size_t>(m->f32_cap) * L;
  const int nl = static_cast<int>(m->layers.size());
  for (int64_t r0 = 0; r0 < B; r0 += SB_ROWS) {
    const int rows = static_cast<int>(B - r0 < SB_ROWS ? B - r0 : SB_ROWS);
    for (int l = 0; l < nl; ++l) {
      const Layer& ly = m->layers[l];
      const __nv_bfloat16* wt = m->wt_bf16 + static_cast<size_t>(ly.row_off) * m->kpad;
      const float* bias = m->bias_fold + ly.row_off;
      const float* hin; int ldin; float* hout; int ldout; const float* res = nullptr; int relu = 1;
      if (l == 0) { hin = x + r0 * kIn; ldin = kIn; hout = P; ldout = L; }
      else if (l == nl - 1) { hin = P; ldin = L; hout = y + r0 * m->out_size; ldout = m->out_size; relu = 0; }
      else if (l & 1) { hin = P; ldin = L; hout = Q; ldout = L; }
      else { hin = Q; ldin = L; hout = P; ldout = L; if (m->cfg.residual) res = P; }
      const int blocks = (ly.N * 32 + 255) / 256;
      if (rows == 1)
        small_batch_layer_kernel<1><<<blocks, 256, 0, st>>>(hin, ldin, ly.K, wt, m->kpad, bias, ly.N, relu, res, hout, ldout, rows);
      else
        small_batch_layer_kernel<SB_ROWS><<<blocks, 256, 0, st>>>(hin, ldin, ly.K, wt, m->kpad, bias, ly.N, relu, res, hout, ldout, rows);
      P3D_LAUNCH_CHECK();
    }
  }
  return P3D_OK;
}

}  // namespace simt
}  // namespace p3d
