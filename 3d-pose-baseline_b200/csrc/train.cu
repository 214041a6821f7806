// Training step: model.step(..., isTraining=True)  (src/linear_model.py:129-145,203-235).
//   forward with BATCH statistics (tf.layers.batch_normalization(training=True): momentum .99, eps 1e-3,
//   biased variance, moving averages updated with the step) and TF1 dropout  y/keep * floor(keep+U),
//   loss = mean((y-t)^2) over B*out, backward through clip_by_norm / BN / ReLU / dropout / residual,
//   TF-flavoured Adam with lr = lr0 * 0.96^(global_step/100000).
// P3D_MODE_BF16: every MatMul of the step (forward, tf.gradients wrt activations, weight gradients) runs on the
// tcgen05 tensor cores (tc_gemm.cu) with bf16 operands, fp32 accumulation and fp32 master weights; H, dZ and W
// are consumed in their natural row-major layouts (MN-major UMMA descriptors where the reduction dimension is
// the row index), the forward GEMM's epilogue also produces the BatchNorm column sums.  P3D_MODE_FP32: FFMA GEMMs.
// P3D_TRAIN_MATMUL_BF16X3 (fp32 / bf16x3 models, opt-in): the FFMA route's kernels, with every GEMM replaced by three
// split-bf16 tcgen05 products (tc_gemm.cu segment schedule) on split-pair copies of x, h, dz, dy and W.
// Data parallel (one process per GPU): rows are sharded, BN statistics and their backward sums are
// all-reduced (SyncBN - required for parity with the single-device reference), and the flat gradient
// buffer is all-reduced once with NCCL before the (replicated) Adam update.
#include <dlfcn.h>
#include <nccl.h>

#include <cmath>
#include <cstring>

#include "common.cuh"
#include "train_common.cuh"

namespace p3d {
namespace prep { int pack_input_split(const float*, __nv_bfloat16*, int64_t, cudaStream_t); }

namespace train {

// ------------------------------------------------------------------ NCCL through dlopen
struct NcclApi {
  void* lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
};
static NcclApi* nccl() {
  static NcclApi api;
  if (api.lib) return &api;
  const char* names[] = {"libnccl.so.2", "libnccl.so"};
  for (const char* n : names) { api.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL); if (api.lib) break; }
  if (!api.lib) { set_error("libnccl.so.2 not found: %s", dlerror()); return nullptr; }
  api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(dlsym(api.lib, "ncclGetUniqueId"));
  api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(dlsym(api.lib, "ncclCommInitRank"));
  api.AllReduce = reinterpret_cast<decltype(api.AllReduce)>(dlsym(api.lib, "ncclAllReduce"));
  api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(dlsym(api.lib, "ncclCommDestroy"));
  api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(dlsym(api.lib, "ncclGetErrorString"));
  if (!api.GetUniqueId || !api.CommInitRank || !api.AllReduce || !api.CommDestroy) {
    set_error("libnccl is missing required symbols");
    api.lib = nullptr;
    return nullptr;
  }
  return &api;
}
#define P3D_NCCL(expr)                                                                         \
  do {                                                                                         \
    ncclResult_t r__ = (expr);                                                                 \
    if (r__ != ncclSuccess) {                                                                  \
      set_error("%s failed: %s", #expr, ::p3d::train::nccl()->GetErrorString ? ::p3d::train::nccl()->GetErrorString(r__) : "?"); \
      return P3D_ERR_NCCL;                                                                     \
    }                                                                                          \
  } while (0)

static int allreduce(p3d_model* m, void* buf, size_t n, ncclDataType_t dt, cudaStream_t st) {
  if (m->world <= 1) return P3D_OK;
  // the latency-bound reductions (SyncBN sums, loss) go over NVLink peer memory in one kernel each (p2p.cu)
  if (dt == ncclDouble && n <= 8192 && p2p::ready(m)) return p2p::allreduce_small(m, static_cast<double*>(buf), n, st);
  // the flat gradient: pulled, summed in rank order and pushed back over peer memory (one kernel)
  if (dt == ncclFloat && buf == m->grad && p2p::grad_ready(m)) {
    // the step's outputs ride along: after this kernel every rank holds the global batch's outputs
    const bool gy = m->dp_y != nullptr && m->dp_Bg * m->out_size <= p2p::YMAX;
    return p2p::allreduce_grad(m, n, gy ? m->dp_y : nullptr, m->dp_rows, m->dp_row0, m->out_size, st);
  }
  P3D_NCCL(nccl()->AllReduce(buf, buf, n, dt, ncclSum, static_cast<ncclComm_t>(m->nccl_comm), st));
  return P3D_OK;
}

// ------------------------------------------------------------------ kernels
constexpr int RCH = 256;   // rows per block in the column-reduction kernels (block = 32 cols x 8 row lanes)
constexpr int RCH4 = 64;   // rows per block of the float4 column-reduction kernels (block = 32 x 4 cols, 8 row lanes)

__global__ void set_scalars_kernel(StepScalars* dst, const StepScalars v) { *dst = v; }

// per-layer table for the kernels that sweep all weight matrices in one launch (gridDim.y = layer)
struct LayerTabEntry { long long off_w, off_wb, off_ws; int K, N, ldwb, seg; };

// bf16x3 split pair of 4 consecutive values: hi = bf16(v) at p[0..3], lo = bf16(v - hi) at p[lo..lo+3] (v - hi is exact)
__device__ __forceinline__ void store_split4(__nv_bfloat16* p, int lo, const float (&v)[4]) {
  __nv_bfloat16 h[4], l[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) { h[j] = __float2bfloat16_rn(v[j]); l[j] = __float2bfloat16_rn(v[j] - __bfloat162float(h[j])); }
  uint2 qh, ql;
  memcpy(&qh, h, 8); memcpy(&ql, l, 8);
  *reinterpret_cast<uint2*>(p) = qh;
  *reinterpret_cast<uint2*>(p + lo) = ql;
}

// W -> bf16 operand copy (row pitch ldwb >= N) and ||W||_F^2, every layer in ONE launch; ws: the split pair of W instead
// (bf16x3 training route, rows [hi | lo] of pitch 2 seg at off_ws).  The norm is summed in the same order either way.
__global__ void wprep_kernel(const float* __restrict__ theta, const LayerTabEntry* __restrict__ tab, __nv_bfloat16* __restrict__ wb,
                             double* __restrict__ norm2, __nv_bfloat16* __restrict__ ws) {
  const LayerTabEntry e = tab[blockIdx.y];
  const long long n = static_cast<long long>(e.K) * e.N;
  const float* w = theta + e.off_w;
  double acc = 0.0;
  if (e.ldwb == e.N && (n & 3) == 0) {
    for (long long i = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) * 4; i < n;
         i += static_cast<long long>(gridDim.x) * blockDim.x * 4) {
      const float4 v = *reinterpret_cast<const float4*>(w + i);
      acc += static_cast<double>(v.x) * v.x + static_cast<double>(v.y) * v.y + static_cast<double>(v.z) * v.z + static_cast<double>(v.w) * v.w;
      if (wb) {
        __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
        uint2 pk; pk.x = *reinterpret_cast<uint32_t*>(&lo); pk.y = *reinterpret_cast<uint32_t*>(&hi);
        *reinterpret_cast<uint2*>(wb + e.off_wb + i) = pk;
      }
      if (ws) {      // N % 4 == 0 here (hidden widths, and the output layer only when N == its 48-column pitch)
        const long long r = i / e.N;
        const float vv[4] = {v.x, v.y, v.z, v.w};
        store_split4(ws + e.off_ws + r * 2 * e.seg + (i - r * e.N), e.seg, vv);
      }
    }
  } else {
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n; i += static_cast<long long>(gridDim.x) * blockDim.x) {
      const float v = w[i];
      acc += static_cast<double>(v) * v;
      if (wb) { const long long r = i / e.N; wb[e.off_wb + r * e.ldwb + (i - r * e.N)] = __float2bfloat16_rn(v); }
      if (ws) {
        const long long r = i / e.N;
        __nv_bfloat16* row = ws + e.off_ws + r * 2 * e.seg + (i - r * e.N);
        const __nv_bfloat16 h = __float2bfloat16_rn(v);
        row[0] = h; row[e.seg] = __float2bfloat16_rn(v - __bfloat162float(h));
      }
    }
  }
  if (norm2) {
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    __shared__ double part[8];
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
      double tot = 0;
      for (int q = 0; q < (int)(blockDim.x >> 5); ++q) tot += part[q];
      atomicAdd(norm2 + blockIdx.y, tot);
    }
  }
}

// <W_l, grad_l> for every layer in one launch (the clip_by_norm pull-back needs it)
__global__ void clipdot_kernel(const float* __restrict__ theta, const float* __restrict__ grad, const LayerTabEntry* __restrict__ tab,
                               double* __restrict__ dots) {
  const LayerTabEntry e = tab[blockIdx.y];
  const long long n = static_cast<long long>(e.K) * e.N;
  const float* w = theta + e.off_w;
  const float* g = grad + e.off_w;
  double acc = 0.0;
  if ((n & 3) == 0 && (e.off_w & 3) == 0) {
    for (long long i = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) * 4; i < n; i += static_cast<long long>(gridDim.x) * blockDim.x * 4) {
      const float4 a = *reinterpret_cast<const float4*>(w + i), b = *reinterpret_cast<const float4*>(g + i);
      acc += static_cast<double>(a.x) * b.x + static_cast<double>(a.y) * b.y + static_cast<double>(a.z) * b.z + static_cast<double>(a.w) * b.w;
    }
  } else {
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n; i += static_cast<long long>(gridDim.x) * blockDim.x)
      acc += static_cast<double>(w[i]) * g[i];
  }
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  __shared__ double part[8];
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double tot = 0;
    for (int q = 0; q < (int)(blockDim.x >> 5); ++q) tot += part[q];
    atomicAdd(dots + blockIdx.y, tot);
  }
}

__global__ void clip_scale_kernel(const double* norm2, float* scale, int n) {
  const int i = threadIdx.x;
  if (i < n) scale[i] = 1.f / fmaxf(static_cast<float>(sqrt(norm2[i])), 1.f);
}

__global__ void colstats_kernel(const float* __restrict__ z, long long B, int L, double* __restrict__ out) {
  __shared__ double s1[8][33], s2[8][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const long long r0 = static_cast<long long>(blockIdx.y) * RCH;
  const long long r1 = (r0 + RCH < B) ? r0 + RCH : B;
  double a = 0, b = 0;
  if (c < L)
    for (long long r = r0 + threadIdx.y; r < r1; r += 8) { const double v = z[r * L + c]; a += v; b += v * v; }
  s1[threadIdx.y][threadIdx.x] = a; s2[threadIdx.y][threadIdx.x] = b;
  __syncthreads();
  if (threadIdx.y == 0 && c < L) {
    for (int i = 1; i < 8; ++i) { a += s1[i][threadIdx.x]; b += s2[i][threadIdx.x]; }
    atomicAdd(out + c, a);
    atomicAdd(out + L + c, b);
  }
}

// mean / biased variance from (sum, sumsq) over the GLOBAL batch; moving averages (momentum .99)
__global__ void bn_finalize_kernel(const double* __restrict__ stats, double invB, int L, float* __restrict__ mean,
                                   float* __restrict__ rstd, float* __restrict__ mm, float* __restrict__ mv) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= L) return;
  const double mu = stats[c] * invB;
  double var = stats[L + c] * invB - mu * mu;
  if (var < 0) var = 0;
  mean[c] = static_cast<float>(mu);
  rstd[c] = static_cast<float>(1.0 / sqrt(var + static_cast<double>(kBnEps)));
  mm[c] = mm[c] * kBnMomentum + static_cast<float>(mu) * (1.f - kBnMomentum);
  mv[c] = mv[c] * kBnMomentum + static_cast<float>(var) * (1.f - kBnMomentum);
}

struct ActArgs {
  const float* z; const float* mean; const float* rstd; const float* gamma; const float* beta;
  const float* res; float* h; __nv_bfloat16* hb; uint8_t* mask; const uint8_t* mask_in;
  const StepScalars* sc; unsigned layer; long long row0, B; int L; int has_bn; int dropout;
  __nv_bfloat16* hs; int seg;     // bf16x3 training route: split pair of h, rows [hi | lo] of pitch 2 seg (else null)
};

// h = dropout(relu(bn(z))) (+res); one thread per 4 columns; also materialises the keep-mask
__global__ void fwd_act_kernel(const ActArgs a) {
  const int L4 = a.L / 4;
  const long long total = a.B * L4;
  const float keep = a.sc->keep, inv_keep = a.sc->inv_keep;
  const unsigned long long seed = a.sc->seed;
  const unsigned step = a.sc->step;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = i / L4;
    const int c4 = static_cast<int>(i - r * L4), c = c4 * 4;
    const float4 zz = *reinterpret_cast<const float4*>(a.z + r * a.L + c);
    float v[4] = {zz.x, zz.y, zz.z, zz.w};
    if (a.has_bn) {
#pragma unroll
      for (int j = 0; j < 4; ++j) v[j] = a.gamma[c + j] * ((v[j] - a.mean[c + j]) * a.rstd[c + j]) + a.beta[c + j];
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] = fmaxf(v[j], 0.f);
    if (a.dropout) {
      uint8_t kb[4];
      if (a.mask_in) {
        const uchar4 mi = *reinterpret_cast<const uchar4*>(a.mask_in + r * a.L + c);
        kb[0] = mi.x; kb[1] = mi.y; kb[2] = mi.z; kb[3] = mi.w;
      } else {
        const uint4 w = dropout_words(seed, step, a.layer, static_cast<uint32_t>(a.row0 + r), static_cast<uint32_t>(c4));
        kb[0] = keep_bit(w.x, keep); kb[1] = keep_bit(w.y, keep); kb[2] = keep_bit(w.z, keep); kb[3] = keep_bit(w.w, keep);
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) v[j] = kb[j] ? v[j] * inv_keep : 0.f;
      *reinterpret_cast<uchar4*>(a.mask + r * a.L + c) = make_uchar4(kb[0], kb[1], kb[2], kb[3]);
    }
    if (a.res) {
      const float4 rr = *reinterpret_cast<const float4*>(a.res + r * a.L + c);
      v[0] += rr.x; v[1] += rr.y; v[2] += rr.z; v[3] += rr.w;
    }
    if (a.h) *reinterpret_cast<float4*>(a.h + r * a.L + c) = make_float4(v[0], v[1], v[2], v[3]);
    if (a.hb) {      // operand of the next layer's tcgen05 GEMMs (forward and weight gradient)
      __nv_bfloat162 lo = __floats2bfloat162_rn(v[0], v[1]), hi = __floats2bfloat162_rn(v[2], v[3]);
      uint2 pk; pk.x = *reinterpret_cast<uint32_t*>(&lo); pk.y = *reinterpret_cast<uint32_t*>(&hi);
      *reinterpret_cast<uint2*>(a.hb + r * a.L + c) = pk;
    }
    if (a.hs) store_split4(a.hs + r * 2 * a.seg + c, a.seg, v);     // operand of the next layer's bf16x3 GEMMs
  }
}

// fp32 -> bf16 with a (possibly wider) destination pitch; pad columns are left untouched (zero)
__global__ void to_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, long long rows, int cols, int ld_dst) {
  const long long total = rows * cols;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = i / cols;
    const int c = static_cast<int>(i - r * cols);
    dst[r * ld_dst + c] = __float2bfloat16_rn(src[i]);
  }
}

// dy = 2 (y - t) / (Bg*out), loss accumulator += sum (y-t)^2
// dyb: bf16 operand copy of dy with row pitch ld_b; lo_b > 0: the split pair instead, lo half at column lo_b + c
__global__ void loss_dy_kernel(const float* __restrict__ y, const float* __restrict__ t, size_t n, float scale,
                               float* __restrict__ dy, double* __restrict__ acc, __nv_bfloat16* __restrict__ dyb, int out, int ld_b,
                               int lo_b) {
  double s = 0;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const float d = y[i] - t[i];
    dy[i] = scale * d;
    if (dyb) {
      const size_t r = i / out;
      const float v = scale * d;
      const __nv_bfloat16 h = __float2bfloat16_rn(v);
      dyb[r * ld_b + (i - r * out)] = h;
      if (lo_b) dyb[r * ld_b + lo_b + (i - r * out)] = __float2bfloat16_rn(v - __bfloat162float(h));
    }
    s += static_cast<double>(d) * d;
  }
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  __shared__ double part[8];
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double tot = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += part[w];
    atomicAdd(acc, tot);
  }
}
__global__ void finish_step_scalars_kernel(const double* acc, double denom, const StepScalars* sc, float* loss, float* lr_out) {
  if (loss) *loss = static_cast<float>(*acc / denom);
  if (lr_out) *lr_out = sc->lr_t;
}

struct BwdArgs {
  const float* dh; const float* z; const float* mean; const float* rstd; const float* gamma; const float* beta;
  const uint8_t* mask; float* dz; __nv_bfloat16* dzb; double* sums; const StepScalars* sc; long long B; int L; int has_bn; int dropout;
  __nv_bfloat16* dzs; int seg;    // bf16x3 training route, layers without BN: split pair of dz (else null)
};

// pass A: da = dh * dropout * relu'(a); column sums of da and da*xhat (for BN backward / dgamma, dbeta).
// Block = 32 x 8 threads, every thread owns 4 consecutive columns (float4) of RCH4 / 8 rows.
__global__ void __launch_bounds__(256) bwd_act_kernel(const BwdArgs a) {
  __shared__ double s1[8][33][4], s2[8][33][4];
  const int c = (blockIdx.x * 32 + threadIdx.x) * 4;
  const long long r0 = static_cast<long long>(blockIdx.y) * RCH4;
  const long long r1 = (r0 + RCH4 < a.B) ? r0 + RCH4 : a.B;
  const float inv_keep = a.sc->inv_keep;
  double p[4] = {0, 0, 0, 0}, q[4] = {0, 0, 0, 0};
  if (c < a.L) {
    float mu[4] = {0, 0, 0, 0}, rs[4] = {1, 1, 1, 1}, g[4] = {1, 1, 1, 1}, be[4] = {0, 0, 0, 0};
    if (a.has_bn) {
      const float4 m4 = *reinterpret_cast<const float4*>(a.mean + c), r4 = *reinterpret_cast<const float4*>(a.rstd + c);
      const float4 g4 = *reinterpret_cast<const float4*>(a.gamma + c), b4 = *reinterpret_cast<const float4*>(a.beta + c);
      mu[0] = m4.x; mu[1] = m4.y; mu[2] = m4.z; mu[3] = m4.w; rs[0] = r4.x; rs[1] = r4.y; rs[2] = r4.z; rs[3] = r4.w;
      g[0] = g4.x; g[1] = g4.y; g[2] = g4.z; g[3] = g4.w; be[0] = b4.x; be[1] = b4.y; be[2] = b4.z; be[3] = b4.w;
    }
    for (long long r = r0 + threadIdx.y; r < r1; r += 8) {
      const size_t o = static_cast<size_t>(r) * a.L + c;
      const float4 z4 = *reinterpret_cast<const float4*>(a.z + o);
      const float4 d4 = *reinterpret_cast<const float4*>(a.dh + o);
      uchar4 mk = make_uchar4(1, 1, 1, 1);
      if (a.dropout) mk = *reinterpret_cast<const uchar4*>(a.mask + o);
      const float zz[4] = {z4.x, z4.y, z4.z, z4.w};
      const float dd[4] = {d4.x, d4.y, d4.z, d4.w};
      const unsigned char kk[4] = {mk.x, mk.y, mk.z, mk.w};
      float da[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float xh = a.has_bn ? (zz[j] - mu[j]) * rs[j] : 0.f;
        const float act = a.has_bn ? g[j] * xh + be[j] : zz[j];
        float gr = dd[j];
        if (a.dropout) gr = kk[j] ? gr * inv_keep : 0.f;
        da[j] = act > 0.f ? gr : 0.f;
        p[j] += da[j]; q[j] += static_cast<double>(da[j]) * xh;
      }
      if (a.dz) *reinterpret_cast<float4*>(a.dz + o) = make_float4(da[0], da[1], da[2], da[3]);
      if (a.dzb) {       // final dz only when the layer has no BN
        __nv_bfloat162 lo = __floats2bfloat162_rn(da[0], da[1]), hi = __floats2bfloat162_rn(da[2], da[3]);
        uint2 pk; pk.x = *reinterpret_cast<uint32_t*>(&lo); pk.y = *reinterpret_cast<uint32_t*>(&hi);
        *reinterpret_cast<uint2*>(a.dzb + o) = pk;
      }
      if (a.dzs) store_split4(a.dzs + static_cast<size_t>(r) * 2 * a.seg + c, a.seg, da);
    }
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) { s1[threadIdx.y][threadIdx.x][j] = p[j]; s2[threadIdx.y][threadIdx.x][j] = q[j]; }
  __syncthreads();
  if (threadIdx.y == 0 && c < a.L) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      double pp = p[j], qq = q[j];
      for (int i = 1; i < 8; ++i) { pp += s1[i][threadIdx.x][j]; qq += s2[i][threadIdx.x][j]; }
      atomicAdd(a.sums + c + j, pp);
      if (a.has_bn) atomicAdd(a.sums + a.L + c + j, qq);
    }
  }
}

// pass B (BN layers): dz = gamma * rstd * (da - mean(da) - xhat * mean(da*xhat)), means over the GLOBAL batch;
// also writes dgamma / dbeta (pre-divided by the world size: the flat gradient all-reduce restores them).
__global__ void bwd_bn_kernel(float* __restrict__ dz, const float* __restrict__ z, const float* __restrict__ mean,
                              const float* __restrict__ rstd, const float* __restrict__ gamma,
                              const double* __restrict__ sums, float invB, long long B, int L, __nv_bfloat16* __restrict__ dzb,
                              int write_f32, double pg_scale, float* __restrict__ ggamma, float* __restrict__ gbeta,
                              const float* __restrict__ dh, const uint8_t* __restrict__ mask, const float* __restrict__ beta,
                              const StepScalars* __restrict__ sc, __nv_bfloat16* __restrict__ dzs, int seg) {
  // dzs: the split pair of dz (bf16x3 training route), rows [hi | lo] of pitch 2 seg
  // dh != null: da is recomputed from (dh, z, mask) instead of being read back - pass A then never stores it
  const int L4 = L / 4;
  const long long total = B * L4;
  const float inv_keep = sc->inv_keep;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = i / L4;
    const int c = static_cast<int>(i - r * L4) * 4;
    const size_t o = static_cast<size_t>(r) * L + c;
    const float4 z4 = *reinterpret_cast<const float4*>(z + o);
    const float4 d4 = *reinterpret_cast<const float4*>((dh ? dh : dz) + o);
    const float4 m4 = *reinterpret_cast<const float4*>(mean + c), r4 = *reinterpret_cast<const float4*>(rstd + c);
    const float4 g4 = *reinterpret_cast<const float4*>(gamma + c);
    const float zz[4] = {z4.x, z4.y, z4.z, z4.w};
    float dd[4] = {d4.x, d4.y, d4.z, d4.w};
    const float mu[4] = {m4.x, m4.y, m4.z, m4.w}, rs[4] = {r4.x, r4.y, r4.z, r4.w}, gg[4] = {g4.x, g4.y, g4.z, g4.w};
    float xh[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) xh[j] = (zz[j] - mu[j]) * rs[j];
    if (dh) {
      const float4 b4 = *reinterpret_cast<const float4*>(beta + c);
      const float be[4] = {b4.x, b4.y, b4.z, b4.w};
      uchar4 mk = make_uchar4(1, 1, 1, 1);
      if (mask) mk = *reinterpret_cast<const uchar4*>(mask + o);
      const unsigned char kk[4] = {mk.x, mk.y, mk.z, mk.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float gr = dd[j];
        if (mask) gr = kk[j] ? gr * inv_keep : 0.f;
        dd[j] = (gg[j] * xh[j] + be[j] > 0.f) ? gr : 0.f;
      }
    }
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float m1 = static_cast<float>(sums[c + j]) * invB, m2 = static_cast<float>(sums[L + c + j]) * invB;
      v[j] = gg[j] * rs[j] * (dd[j] - m1 - xh[j] * m2);
    }
    if (write_f32) *reinterpret_cast<float4*>(dz + o) = make_float4(v[0], v[1], v[2], v[3]);
    if (dzb) {
      __nv_bfloat162 lo = __floats2bfloat162_rn(v[0], v[1]), hi = __floats2bfloat162_rn(v[2], v[3]);
      uint2 pk; pk.x = *reinterpret_cast<uint32_t*>(&lo); pk.y = *reinterpret_cast<uint32_t*>(&hi);
      *reinterpret_cast<uint2*>(dzb + o) = pk;
    }
    if (dzs) store_split4(dzs + static_cast<size_t>(r) * 2 * seg + c, seg, v);
    if (r == 0) {
#pragma unroll
      for (int j = 0; j < 4; ++j) { gbeta[c + j] = static_cast<float>(sums[c + j] * pg_scale); ggamma[c + j] = static_cast<float>(sums[L + c + j] * pg_scale); }
    }
  }
}

__global__ void colsum_kernel(const float* __restrict__ a, long long B, int N, float* __restrict__ out) {
  __shared__ float s1[8][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const long long r0 = static_cast<long long>(blockIdx.y) * RCH;
  const long long r1 = (r0 + RCH < B) ? r0 + RCH : B;
  float p = 0;
  if (c < N)
    for (long long r = r0 + threadIdx.y; r < r1; r += 8) p += a[r * N + c];
  s1[threadIdx.y][threadIdx.x] = p;
  __syncthreads();
  if (threadIdx.y == 0 && c < N) {
    for (int i = 1; i < 8; ++i) p += s1[i][threadIdx.x];
    atomicAdd(out + c, p);
  }
}

// Pull the gradient wrt the clipped weight back through tf.clip_by_norm (src/linear_model.py:108):
//   g = (gc - W <W,gc>/||W||^2) / ||W||  when ||W|| > 1, else g = gc
// and apply TF Adam (src/linear_model.py:137): m += (g-m)(1-b1); v += (g^2-v)(1-b2); theta -= alpha_t m/(sqrt(v)+eps).
// One launch: gridDim.y = layer for the weight matrices, the last y-slice covers biases / gamma / beta.
__global__ void adam_clip_kernel(float* __restrict__ theta, float* __restrict__ grad, float* __restrict__ m, float* __restrict__ v,
                                 const LayerTabEntry* __restrict__ tab, int nlay, long long n_w, long long n_train,
                                 const StepScalars* __restrict__ sc, const double* __restrict__ dots, const double* __restrict__ norm2,
                                 int clip) {
  long long beg, end;
  float cs = 1.f, cd = 0.f;
  bool pull = false;
  if (static_cast<int>(blockIdx.y) < nlay) {
    const LayerTabEntry e = tab[blockIdx.y];
    beg = e.off_w; end = e.off_w + static_cast<long long>(e.K) * e.N;
    if (clip) {
      const double n2 = norm2[blockIdx.y];
      if (n2 > 1.0) { cs = static_cast<float>(1.0 / sqrt(n2)); cd = static_cast<float>(dots[blockIdx.y] / n2); pull = true; }
    }
  } else {
    beg = n_w; end = n_train;
  }
  const float alpha = sc->alpha;
  const long long tid = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x, nth = static_cast<long long>(gridDim.x) * blockDim.x;
  if (((beg | (end - beg)) & 3) == 0) {
    for (long long i = beg + tid * 4; i < end; i += nth * 4) {
      float4 g4 = *reinterpret_cast<const float4*>(grad + i);
      float4 t4 = *reinterpret_cast<const float4*>(theta + i);
      float4 m4 = *reinterpret_cast<const float4*>(m + i);
      float4 v4 = *reinterpret_cast<const float4*>(v + i);
      float g[4] = {g4.x, g4.y, g4.z, g4.w}, th[4] = {t4.x, t4.y, t4.z, t4.w}, mm[4] = {m4.x, m4.y, m4.z, m4.w}, vv[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (pull) g[j] = (g[j] - th[j] * cd) * cs;
        mm[j] = mm[j] + (g[j] - mm[j]) * 0.1f;
        vv[j] = vv[j] + (g[j] * g[j] - vv[j]) * 0.001f;
        th[j] -= alpha * mm[j] / (sqrtf(vv[j]) + 1e-8f);
      }
      if (pull) *reinterpret_cast<float4*>(grad + i) = make_float4(g[0], g[1], g[2], g[3]);   // model.gradients exposes the pulled-back gradient
      *reinterpret_cast<float4*>(m + i) = make_float4(mm[0], mm[1], mm[2], mm[3]);
      *reinterpret_cast<float4*>(v + i) = make_float4(vv[0], vv[1], vv[2], vv[3]);
      *reinterpret_cast<float4*>(theta + i) = make_float4(th[0], th[1], th[2], th[3]);
    }
  } else {
    for (long long i = beg + tid; i < end; i += nth) {
      float g = grad[i];
      if (pull) { g = (g - theta[i] * cd) * cs; grad[i] = g; }
      const float mi = m[i] + (g - m[i]) * 0.1f;
      const float vi = v[i] + (g * g - v[i]) * 0.001f;
      m[i] = mi; v[i] = vi;
      theta[i] -= alpha * mi / (sqrtf(vi) + 1e-8f);
    }
  }
}

// ------------------------------------------------------------------ workspace
void free_workspace(p3d_model* m) {
  TrainWorkspace& w = m->tw;
  cudaFree(w.z); cudaFree(w.h); cudaFree(w.dh); cudaFree(w.dz); cudaFree(w.dres); cudaFree(w.dy);
  cudaFree(w.stats); cudaFree(w.mean); cudaFree(w.rstd); cudaFree(w.scal); cudaFree(w.maskbuf);
  cudaFree(w.xb); cudaFree(w.hb); cudaFree(w.dzb); cudaFree(w.dyb); cudaFree(w.wb);
  cudaFree(w.xs); cudaFree(w.hs); cudaFree(w.dzs); cudaFree(w.dys); cudaFree(w.ws);
  cudaFree(w.tab); cudaFree(w.sc); cudaFree(w.gx); cudaFree(w.gt); cudaFree(w.gy); cudaFree(w.gscal);
  for (auto& ge : w.graphs) if (ge.exec) cudaGraphExecDestroy(static_cast<cudaGraphExec_t>(ge.exec));
  if (w.cap_stream) cudaStreamDestroy(w.cap_stream);
  if (w.side_stream) cudaStreamDestroy(w.side_stream);
  for (auto& e : w.ev) if (e) cudaEventDestroy(e);
  w = TrainWorkspace();
  p2p::destroy(m);
  if (m->nccl_comm && nccl()) { nccl()->CommDestroy(static_cast<ncclComm_t>(m->nccl_comm)); m->nccl_comm = nullptr; }
}

constexpr int kOutPad = 48;   // bf16 pitch of dy / W4 rows: 96 B keeps TMA's 16-byte pitch rule for out = 42 too
// bf16 mode runs the step's GEMMs on the tensor cores (tc_gemm.cu); fp32 mode keeps the FFMA GEMMs.  fp16 mode chooses
// inference arithmetic only: it trains on the bf16 route.
static inline bool use_tc(const p3d_model* m) { return (m->cfg.mode == P3D_MODE_BF16 || m->cfg.mode == P3D_MODE_FP16) && (m->L % 8) == 0; }
// P3D_TRAIN_MATMUL_BF16X3 (fp32 / bf16x3 models): the step's GEMMs as three split-bf16 products on the tensor cores;
// widths the tcgen05 GEMM does not tile keep FFMA
static inline bool use_x3(const p3d_model* m) {
  return m->train_matmul == P3D_TRAIN_MATMUL_BF16X3 && m->cfg.mode != P3D_MODE_BF16 && (m->L % 8) == 0;
}
static inline int seg_of(int n) { return (n + 63) / 64 * 64; }   // lo-segment column of a split pair of width n

static void drop_graphs(TrainWorkspace& w) {
  for (auto& ge : w.graphs) if (ge.exec) cudaGraphExecDestroy(static_cast<cudaGraphExec_t>(ge.exec));   // they hold the old pointers
  w.graphs.clear();
}

// the split-pair buffers of the bf16x3 route for cap_B rows, zeroed once (their padding columns are never written)
static int ensure_split_buffers(p3d_model* m) {
  TrainWorkspace& w = m->tw;
  const int nh = static_cast<int>(m->layers.size()) - 1, ld = 2 * seg_of(m->L);
  if (w.x3_B >= w.cap_B) return P3D_OK;
  drop_graphs(w);
  cudaFree(w.xs); cudaFree(w.hs); cudaFree(w.dzs); cudaFree(w.dys);
  w.xs = w.hs = w.dzs = w.dys = nullptr; w.x3_B = 0;
  const size_t B = static_cast<size_t>(w.cap_B);
  const size_t nx = B * 128, nhs = B * ld * nh, ndz = B * ld, ndy = B * 128;
  P3D_CUDA(cudaMalloc(&w.xs, sizeof(__nv_bfloat16) * nx));
  P3D_CUDA(cudaMalloc(&w.hs, sizeof(__nv_bfloat16) * nhs));
  P3D_CUDA(cudaMalloc(&w.dzs, sizeof(__nv_bfloat16) * ndz));
  P3D_CUDA(cudaMalloc(&w.dys, sizeof(__nv_bfloat16) * ndy));
  P3D_CUDA(cudaMemset(w.hs, 0, sizeof(__nv_bfloat16) * nhs));
  P3D_CUDA(cudaMemset(w.dzs, 0, sizeof(__nv_bfloat16) * ndz));
  P3D_CUDA(cudaMemset(w.dys, 0, sizeof(__nv_bfloat16) * ndy));      // (pack_input_split writes every column of xs)
  if (!w.ws) {
    const size_t n = w.ws_off.back() + static_cast<size_t>(m->layers.back().K) * 2 * seg_of(m->out_size);
    P3D_CUDA(cudaMalloc(&w.ws, sizeof(__nv_bfloat16) * n));
    P3D_CUDA(cudaMemset(w.ws, 0, sizeof(__nv_bfloat16) * n));
  }
  w.x3_B = w.cap_B;
  return P3D_OK;
}

static int ensure_workspace(p3d_model* m, int64_t B) {
  TrainWorkspace& w = m->tw;
  const int L = m->L, nh = static_cast<int>(m->layers.size()) - 1, nl = nh + 1;
  if (w.cap_B >= B) return use_x3(m) ? ensure_split_buffers(m) : P3D_OK;
  drop_graphs(w);
  cudaFree(w.xs); cudaFree(w.hs); cudaFree(w.dzs); cudaFree(w.dys);
  w.xs = w.hs = w.dzs = w.dys = nullptr; w.x3_B = 0;
  cudaFree(w.gx); cudaFree(w.gt); cudaFree(w.gy);
  w.gx = w.gt = w.gy = nullptr;
  cudaFree(w.z); cudaFree(w.h); cudaFree(w.dh); cudaFree(w.dz); cudaFree(w.dres); cudaFree(w.dy); cudaFree(w.maskbuf);
  cudaFree(w.xb); cudaFree(w.hb); cudaFree(w.dzb); cudaFree(w.dyb);
  w.z = w.h = w.dh = w.dz = w.dres = w.dy = nullptr; w.maskbuf = nullptr; w.cap_B = 0;
  w.xb = w.hb = w.dzb = w.dyb = nullptr;
  const size_t bl = static_cast<size_t>(B) * L;
  P3D_CUDA(cudaMalloc(&w.z, sizeof(float) * bl * nh));
  P3D_CUDA(cudaMalloc(&w.h, sizeof(float) * bl * nh));
  P3D_CUDA(cudaMalloc(&w.dh, sizeof(float) * bl));
  P3D_CUDA(cudaMalloc(&w.dz, sizeof(float) * bl));
  P3D_CUDA(cudaMalloc(&w.dres, sizeof(float) * bl * 2));              // two more rotating gradient buffers
  P3D_CUDA(cudaMalloc(&w.dy, sizeof(float) * static_cast<size_t>(B) * m->out_size));
  P3D_CUDA(cudaMalloc(&w.maskbuf, bl * nh));                          // uint8 keep-masks [nh][B][L]
  // fixed-address staging of x / t / y for the CUDA-graph replay of the step
  P3D_CUDA(cudaMalloc(&w.gx, sizeof(float) * static_cast<size_t>(B) * kIn));
  P3D_CUDA(cudaMalloc(&w.gt, sizeof(float) * static_cast<size_t>(B) * m->out_size));
  P3D_CUDA(cudaMalloc(&w.gy, sizeof(float) * static_cast<size_t>(B) * m->out_size));
  if (use_tc(m)) {
    // bf16 operands of the tcgen05 GEMMs, all in their natural row-major layouts
    P3D_CUDA(cudaMalloc(&w.xb, sizeof(__nv_bfloat16) * static_cast<size_t>(B) * kIn));
    P3D_CUDA(cudaMalloc(&w.hb, sizeof(__nv_bfloat16) * bl * nh));
    P3D_CUDA(cudaMalloc(&w.dzb, sizeof(__nv_bfloat16) * bl * 2));     // two: the fused backward ping-pongs
    P3D_CUDA(cudaMalloc(&w.dyb, sizeof(__nv_bfloat16) * static_cast<size_t>(B) * kOutPad));
    P3D_CUDA(cudaMemset(w.dyb, 0, sizeof(__nv_bfloat16) * static_cast<size_t>(B) * kOutPad));   // pad columns stay zero
    if (!w.wb) {
      // [all hidden W, same offsets as theta][W4 with its rows padded to kOutPad columns]
      const Layer& lo = m->layers.back();
      const size_t n = lo.off_w + static_cast<size_t>(lo.K) * kOutPad;
      P3D_CUDA(cudaMalloc(&w.wb, sizeof(__nv_bfloat16) * n));
      P3D_CUDA(cudaMemset(w.wb, 0, sizeof(__nv_bfloat16) * n));
    }
  }
  if (!w.stats) {
    // doubles: stats [nh][2][L] | bwd sums [nh][2][L] | dots [nl] | loss [1] | grid-barrier words [2 nh][2] (unsigned)
    P3D_CUDA(cudaMalloc(&w.stats, sizeof(double) * (4ull * nh * L + nl + 1 + 2ull * nh)));
    w.red = w.stats + 2ull * nh * L;
    w.gcount = reinterpret_cast<unsigned*>(w.stats + 4ull * nh * L + nl + 1);
    P3D_CUDA(cudaMalloc(&w.mean, sizeof(float) * static_cast<size_t>(nh) * L));
    P3D_CUDA(cudaMalloc(&w.rstd, sizeof(float) * static_cast<size_t>(nh) * L));
    P3D_CUDA(cudaMalloc(&w.scal, sizeof(float) * (nl + 8)));
    P3D_CUDA(cudaMalloc(&w.gscal, sizeof(float) * 2));
    P3D_CUDA(cudaStreamCreateWithFlags(&w.side_stream, cudaStreamNonBlocking));
    for (auto& e : w.ev) P3D_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    P3D_CUDA(cudaMalloc(&w.sc, sizeof(StepScalars)));
    std::vector<LayerTabEntry> tab(nl);
    w.ws_off.assign(nl, 0);
    size_t off_ws = 0;
    for (int l = 0; l < nl; ++l) {
      const Layer& ly = m->layers[l];
      tab[l].off_w = static_cast<long long>(ly.off_w); tab[l].off_wb = static_cast<long long>(ly.off_w);
      tab[l].K = ly.K; tab[l].N = ly.N; tab[l].ldwb = (l == nl - 1) ? kOutPad : ly.N;
      tab[l].seg = seg_of(ly.N); tab[l].off_ws = static_cast<long long>(off_ws);
      w.ws_off[l] = off_ws;
      off_ws += static_cast<size_t>(ly.K) * 2 * tab[l].seg;
    }
    P3D_CUDA(cudaMalloc(&w.tab, sizeof(LayerTabEntry) * nl));
    P3D_CUDA(cudaMemcpy(w.tab, tab.data(), sizeof(LayerTabEntry) * nl, cudaMemcpyHostToDevice));
  }
  w.cap_B = B;
  return use_x3(m) ? ensure_split_buffers(m) : P3D_OK;
}

// P3D_TRAIN_FUSED=0 forces the unfused path (GEMM + statistics + finalize + activation kernels) at every batch size; read
// at every step so that tests can cover both paths in one process.
static bool fused_enabled() { const char* e = getenv("P3D_TRAIN_FUSED"); return !(e && e[0] == '0'); }
static inline dim3 colgrid(int cols, int64_t B) { return dim3((cols + 31) / 32, static_cast<unsigned>((B + RCH - 1) / RCH)); }
static inline int egrid(long long n) { long long g = (n + 255) / 256; if (g > 148 * 8) g = 148 * 8; return static_cast<int>(g < 1 ? 1 : g); }

// Forward + backward with the BatchNorm / ReLU / dropout math fused into the GEMM epilogues (tc_gemm.cu modes 3 and 4).
// Per hidden layer: 1 forward launch (was GEMM + finalize + activation) and 2 backward launches (weight gradient; data
// gradient fused with the previous layer's activation / BN backward - was 4).  One M tile on one GPU: the column
// statistics are CTA-local.  More tiles (every tile of a layer resident at once, i.e. up to ~4700 poses at width 1024)
// and / or data parallel: the CTAs meet at a grid barrier between the two epilogue passes, and the SyncBN exchange
// over NVLink peer memory happens right there, inside the GEMM (FusedTrain in common.cuh) - no separate reduction
// launches, no NCCL call until the flat gradient all-reduce.
static int fwd_bwd_fused(p3d_model* m, const float* t, int64_t B, bool dropout, const uint8_t* mask_in, int64_t Bg, int64_t row0,
                         float* y, cudaStream_t st) {
  using tcg::GemmArgs;
  TrainWorkspace& w = m->tw;
  const StepScalars* sc = static_cast<const StepScalars*>(w.sc);
  const int L = m->L, nlay = static_cast<int>(m->layers.size()), nh = nlay - 1, out = m->out_size;
  const size_t bl = static_cast<size_t>(B) * L;
  const bool clip = m->cfg.max_norm != 0, residual = m->cfg.residual != 0;
  float* scale = w.scal;
  double* lossacc = w.red + 2ull * nh * L + nlay;
  const float invB = 1.f / static_cast<float>(Bg);
  const int Bi = static_cast<int>(B);
  const bool dp = m->world > 1;
  // grid-synchronised form: per layer and direction [2][L] doubles of column sums (w.stats forward, w.red backward,
  // both zeroed at the top of the step) and an arrival counter + completion flag
  auto grid_operands = [&](tcg::FusedTrain& f, double* sums, int which) {
    f.gsum = sums; f.gcount = w.gcount + 2 * which;
    f.row0 = row0; f.world = m->world; f.rank = m->rank; f.pg_scale = 1.f / static_cast<float>(m->world);
    f.peers = dp ? p2p::device_peers(m) : nullptr;
  };
  // ---------------------------------------------------------------- forward
  for (int li = 0; li < nh; ++li) {
    const Layer& ly = m->layers[li];
    GemmArgs g;
    g.M = Bi; g.N = L; g.K = ly.K;
    g.A = li == 0 ? w.xb : w.hb + (li - 1) * bl; g.lda = li == 0 ? kIn : L;
    g.B = w.wb + ly.off_w; g.ldb = L; g.b_mn = 1;
    g.C = w.z + li * bl; g.ldc = L; g.bias = m->theta + ly.off_b; g.alpha_dev = clip ? scale + li : nullptr;
    g.fused_mode = 3;
    tcg::FusedTrain& f = g.fused;
    f.sc = sc; f.has_bn = ly.has_bn; f.dropout = dropout; f.layer = li; f.invB = invB;
    if (ly.has_bn) {
      f.gamma = m->theta + ly.off_gamma; f.beta = m->theta + ly.off_beta;
      f.mean = w.mean + static_cast<size_t>(li) * L; f.rstd = w.rstd + static_cast<size_t>(li) * L;
      f.mov_mean = m->moving + ly.off_mm; f.mov_var = m->moving + ly.off_mv;
    }
    // the fp32 copy of h is only read back as a residual (by layer li + 2)
    const bool h_needed = residual && (li % 2) == 0 && li + 2 < nh;
    f.h = h_needed ? w.h + li * bl : nullptr; f.hb = w.hb + li * bl; f.mask = w.maskbuf + li * bl; f.mask_in = mask_in ? mask_in + li * bl : nullptr;
    f.hres = (residual && li >= 2 && (li % 2) == 0) ? w.h + (li - 2) * bl : nullptr;
    grid_operands(f, w.stats + 2ull * li * L, li);
    P3D_TRY(tcg::gemm(g, st));
  }
  {
    const Layer& ly = m->layers[nh];
    GemmArgs g;
    g.M = Bi; g.N = out; g.K = L;
    g.A = w.hb + (nh - 1) * bl; g.lda = L;
    g.B = w.wb + ly.off_w; g.ldb = kOutPad; g.b_mn = 1;
    g.C = y; g.ldc = out; g.bias = m->theta + ly.off_b; g.alpha_dev = clip ? scale + nh : nullptr;
    P3D_TRY(tcg::gemm(g, st));
  }
  const size_t ny = static_cast<size_t>(B) * out;
  loss_dy_kernel<<<egrid(static_cast<long long>(ny)), 256, 0, st>>>(y, t, ny, 2.0f * invB / out, w.dy, lossacc, w.dyb, out, kOutPad, 0);
  P3D_LAUNCH_CHECK();
  // ---------------------------------------------------------------- backward
  // (data parallel: the loss sum rides on the first backward exchange, see fused_dgrad)
  __nv_bfloat16* dzb[2] = {w.dzb, w.dzb + bl};
  float* DH[2] = {w.dh, w.dres};
  int db = 0, keep = -1;
  // data gradient of layer `li` (li == nh: the output layer) fused with the activation / BN backward of layer t = li - 1
  auto fused_dgrad = [&](int li, const __nv_bfloat16* A, int lda, int K, int ldb, __nv_bfloat16* dz_out) -> int {
    const int tl = li - 1;
    const Layer& lw = m->layers[li];
    const Layer& lt = m->layers[tl];
    const bool add = residual && li < nh && (li % 2) == 1 && keep >= 0;      // the gradient that bypassed the block
    const bool save = residual && tl >= 2 && (tl % 2) == 0;                   // d(h[tl]) also flows to h[tl-2]
    const int slot = (keep >= 0) ? 1 - keep : 0;
    GemmArgs g;
    g.M = Bi; g.N = L; g.K = K;
    g.A = A; g.lda = lda;
    g.B = w.wb + lw.off_w; g.ldb = ldb;
    g.C = w.dz; g.ldc = L; g.alpha_dev = clip ? scale + li : nullptr;
    if (add) { g.res = DH[keep]; g.ldres = L; }
    g.fused_mode = 4;
    tcg::FusedTrain& f = g.fused;
    f.sc = sc; f.has_bn = lt.has_bn; f.dropout = dropout; f.layer = tl; f.invB = invB;
    f.z = w.z + tl * bl; f.mask = w.maskbuf + tl * bl; f.dzb = dz_out;
    f.dh_out = save ? DH[slot] : nullptr;
    if (lt.has_bn) {
      f.gamma = m->theta + lt.off_gamma; f.beta = m->theta + lt.off_beta;
      f.mean = w.mean + static_cast<size_t>(tl) * L; f.rstd = w.rstd + static_cast<size_t>(tl) * L;
      f.ggamma = m->grad + lt.off_gamma; f.gbeta = m->grad + lt.off_beta;
    } else {
      f.gbias = m->grad + lt.off_b;
    }
    grid_operands(f, w.red + 2ull * tl * L, nh + tl);
    if (dp && li == nh) f.xsum = lossacc;
    P3D_TRY(tcg::gemm(g, st));
    if (add) keep = -1;
    if (save) keep = slot;
    return P3D_OK;
  };
  // The weight gradients only feed the optimizer: they run on a side stream (a parallel branch of the captured graph),
  // off the critical path  loss -> dgrad chain -> Adam.  Events: e_dz[k] = "dz of step k is ready", e_wg[k] = "its
  // weight gradient has read it" (the dz ping-pong buffer may then be overwritten).
  cudaStream_t side = w.side_stream;
  int ne = 0;
  auto fork_wgrad = [&](const GemmArgs& gw, cudaEvent_t* done) -> int {
    cudaEvent_t ready = w.ev[ne++ % 16];
    P3D_CUDA(cudaEventRecord(ready, st));
    P3D_CUDA(cudaStreamWaitEvent(side, ready, 0));
    P3D_TRY(tcg::gemm(gw, side));
    *done = w.ev[ne++ % 16];
    P3D_CUDA(cudaEventRecord(*done, side));
    return P3D_OK;
  };
  cudaEvent_t wg_done[2] = {nullptr, nullptr};   // per dz ping-pong buffer: the weight gradient that last read it
  {
    const Layer& ly = m->layers[nh];
    GemmArgs gw;   // dW4 = h^T dy
    gw.M = L; gw.N = out; gw.K = Bi;
    gw.A = w.hb + (nh - 1) * bl; gw.lda = L; gw.a_mn = 1;
    gw.B = w.dyb; gw.ldb = kOutPad; gw.b_mn = 1;
    gw.C = m->grad + ly.off_w; gw.ldc = out; gw.split_k = 1;
    cudaEvent_t e4;
    P3D_TRY(fork_wgrad(gw, &e4));
    colsum_kernel<<<colgrid(out, B), dim3(32, 8), 0, st>>>(w.dy, B, out, m->grad + ly.off_b);
    P3D_LAUNCH_CHECK();
    P3D_TRY(fused_dgrad(nh, w.dyb, kOutPad, out, kOutPad, dzb[db]));
  }
  for (int li = nh - 1; li >= 0; --li) {
    const Layer& ly = m->layers[li];
    GemmArgs gw;   // dW = in^T dz
    gw.M = ly.K; gw.N = L; gw.K = Bi;
    gw.A = li == 0 ? w.xb : w.hb + (li - 1) * bl; gw.lda = li == 0 ? kIn : L; gw.a_mn = 1;
    gw.B = dzb[db]; gw.ldb = L; gw.b_mn = 1;
    gw.C = m->grad + ly.off_w; gw.ldc = L; gw.split_k = 1;
    P3D_TRY(fork_wgrad(gw, &wg_done[db]));
    if (li > 0) {
      if (wg_done[1 - db]) P3D_CUDA(cudaStreamWaitEvent(st, wg_done[1 - db], 0));   // the buffer about to be overwritten is free
      P3D_TRY(fused_dgrad(li, dzb[db], L, L, L, dzb[1 - db]));
      db ^= 1;
    }
  }
  {   // join: the optimizer needs every weight gradient
    cudaEvent_t joined = w.ev[ne++ % 16];
    P3D_CUDA(cudaEventRecord(joined, side));
    P3D_CUDA(cudaStreamWaitEvent(st, joined, 0));
  }
  return P3D_OK;
}

// The step proper: every launch below depends only on (model, B, Bg, row0, dropout on/off, pointers) - all per-step
// values come from the device StepScalars - so the sequence can be captured once and replayed as a CUDA graph.
static int train_body(p3d_model* m, const float* x, const float* t, int64_t B, bool dropout, const uint8_t* mask_in,
                      int64_t Bg, int64_t row0, float* loss, float* lr_used, float* y, cudaStream_t st) {
  using simt::Epilogue;
  using simt::sgemm;
  TrainWorkspace& w = m->tw;
  const StepScalars* sc = static_cast<const StepScalars*>(w.sc);
  const LayerTabEntry* tab = static_cast<const LayerTabEntry*>(w.tab);
  const int L = m->L, nlay = static_cast<int>(m->layers.size()), nh = nlay - 1, out = m->out_size;
  const size_t bl = static_cast<size_t>(B) * L;
  const bool clip = m->cfg.max_norm != 0;
  const bool residual = m->cfg.residual != 0;
  const bool tc = use_tc(m);
  const bool x3 = use_x3(m);        // bf16x3 split products on tcgen05 (unfused route, FFMA's elementwise kernels)
  const bool lowp = tc || x3;       // the GEMMs read the bf16 operand buffers, not the fp32 activations
  const int seg = seg_of(L), ld = 2 * seg;
  const size_t bls = static_cast<size_t>(B) * ld;   // one layer of split activations
  using tcg::GemmArgs;
  double* dots = w.red + 2ull * nh * L;
  double* lossacc = dots + nlay;
  uint8_t* maskbuf = w.maskbuf;
  float* scale = w.scal;   // [nlay] clip scales
  const double invBg = 1.0 / static_cast<double>(Bg);

  m->dp_y = y; m->dp_rows = B; m->dp_row0 = row0; m->dp_Bg = Bg;
  P3D_CUDA(cudaMemsetAsync(w.stats, 0, sizeof(double) * (4ull * nh * L + nlay + 1 + 2ull * nh), st));
  P3D_CUDA(cudaMemsetAsync(m->grad, 0, sizeof(float) * m->n_train, st));
  if (clip) P3D_CUDA(cudaMemsetAsync(m->norm2, 0, sizeof(double) * nlay, st));
  if (clip || lowp) {
    // one launch over all layers: ||W||_F^2 (clip_by_norm) and, on the tensor-core paths, this step's bf16 copy (or
    // split pair) of the UNCLIPPED W in its natural [K][N] layout (W4 rows padded); the clip scale is the GEMMs' alpha
    wprep_kernel<<<dim3(148, nlay), 256, 0, st>>>(m->theta, tab, tc ? w.wb : nullptr, clip ? m->norm2 : nullptr, x3 ? w.ws : nullptr);
    P3D_LAUNCH_CHECK();
  }
  if (clip) {
    clip_scale_kernel<<<1, 64, 0, st>>>(m->norm2, scale, nlay);
    P3D_LAUNCH_CHECK();
  }
  if (tc) {
    to_bf16_kernel<<<egrid(static_cast<long long>(B) * kIn / 4 + 1), 256, 0, st>>>(x, w.xb, B, kIn, kIn);
    P3D_LAUNCH_CHECK();
  }
  if (x3) P3D_TRY(prep::pack_input_split(x, w.xs, B, st));      // [B][128]: hi columns 0..31, lo 64..95
  // fused epilogues: every tile of a hidden layer must be resident at once; data parallel they need the peer-memory
  // exchange (otherwise the unfused path reduces through NCCL).  Every rank decides alike: B is the same everywhere up
  // to one row and the host layer attaches peer memory on all ranks or on none.
  const bool fused = tc && fused_enabled() && tcg::fused_fits(static_cast<int>(B + (m->world > 1 ? 1 : 0)), L, L, m->num_sms) &&
                     (m->world == 1 || (p2p::ready(m) && 2 * L + 1 <= p2p::MAXN));
  if (fused) {
    P3D_TRY(fwd_bwd_fused(m, t, B, dropout, mask_in, Bg, row0, y, st));
  } else {
  // ---------------------------------------------------------------- forward
  for (int li = 0; li < nh; ++li) {
    const Layer& ly = m->layers[li];
    const float* in = li == 0 ? x : w.h + (li - 1) * bl;
    const int lda = li == 0 ? kIn : L;
    float* z = w.z + li * bl;
    double* stats = w.stats + 2ull * li * L;
    if (tc) {
      GemmArgs g;   // z = (x|h) W * clip + b ; BN column sums in the epilogue
      g.M = static_cast<int>(B); g.N = L; g.K = ly.K;
      g.A = li == 0 ? w.xb : w.hb + (li - 1) * bl; g.lda = lda;
      g.B = w.wb + ly.off_w; g.ldb = L; g.b_mn = 1;
      g.C = z; g.ldc = L; g.bias = m->theta + ly.off_b; g.alpha_dev = clip ? scale + li : nullptr;
      g.colsum = ly.has_bn ? stats : nullptr;
      P3D_TRY(tcg::gemm(g, st));
    } else if (x3) {
      GemmArgs g;   // z = (x|h) W * clip + b: A K-major, W MN-major, both split pairs
      g.M = static_cast<int>(B); g.N = L; g.K = ly.K;
      g.A = li == 0 ? w.xs : w.hs + (li - 1) * bls; g.lda = li == 0 ? 128 : ld; g.seg_a = li == 0 ? 64 : seg;
      g.B = w.ws + w.ws_off[li]; g.ldb = ld; g.b_mn = 1; g.seg_b = seg;
      g.C = z; g.ldc = L; g.bias = m->theta + ly.off_b; g.alpha_dev = clip ? scale + li : nullptr;
      P3D_TRY(tcg::gemm(g, st));
    } else {
      Epilogue e; e.bias = m->theta + ly.off_b; e.alpha_dev = clip ? scale + li : nullptr;
      P3D_TRY(sgemm(false, false, B, L, ly.K, in, lda, m->theta + ly.off_w, L, z, L, e, st));
    }
    float* mean = w.mean + static_cast<size_t>(li) * L;
    float* rstd = w.rstd + static_cast<size_t>(li) * L;
    if (ly.has_bn) {
      if (!tc) {
        colstats_kernel<<<colgrid(L, B), dim3(32, 8), 0, st>>>(z, B, L, stats);
        P3D_LAUNCH_CHECK();
      }
      if (m->world > 1 && 2ull * L <= 8192 && p2p::ready(m)) {
        // peer-memory reduction with the BatchNorm finalisation as its tail: one launch
        p2p::BnFinalize fin;
        fin.invB = invBg; fin.mean = mean; fin.rstd = rstd; fin.mm = m->moving + ly.off_mm; fin.mv = m->moving + ly.off_mv;
        P3D_TRY(p2p::allreduce_small(m, stats, 2ull * L, st, &fin));
      } else {
        P3D_TRY(allreduce(m, stats, 2ull * L, ncclDouble, st));
        bn_finalize_kernel<<<(L + 255) / 256, 256, 0, st>>>(stats, invBg, L, mean, rstd, m->moving + ly.off_mm, m->moving + ly.off_mv);
        P3D_LAUNCH_CHECK();
      }
    }
    ActArgs a;
    a.z = z; a.mean = mean; a.rstd = rstd;
    a.gamma = ly.has_bn ? m->theta + ly.off_gamma : nullptr; a.beta = ly.has_bn ? m->theta + ly.off_beta : nullptr;
    a.res = (residual && li >= 2 && (li % 2) == 0) ? w.h + (li - 2) * bl : nullptr;
    // on the tensor-core paths the fp32 copy of h is only read back as a residual (by layer li + 2)
    const bool h_needed = !lowp || (residual && (li % 2) == 0 && li + 2 < nh);
    a.h = h_needed ? w.h + li * bl : nullptr; a.hb = tc ? w.hb + li * bl : nullptr; a.mask = maskbuf + li * bl; a.mask_in = mask_in ? mask_in + li * bl : nullptr;
    a.hs = x3 ? w.hs + li * bls : nullptr; a.seg = seg;
    a.sc = sc; a.layer = li;
    a.row0 = row0; a.B = B; a.L = L; a.has_bn = ly.has_bn; a.dropout = dropout;
    fwd_act_kernel<<<egrid(static_cast<long long>(bl / 4)), 256, 0, st>>>(a);
    P3D_LAUNCH_CHECK();
  }
  {
    const Layer& ly = m->layers[nh];
    if (tc) {
      GemmArgs g;
      g.M = static_cast<int>(B); g.N = out; g.K = L;
      g.A = w.hb + (nh - 1) * bl; g.lda = L;
      g.B = w.wb + ly.off_w; g.ldb = kOutPad; g.b_mn = 1;
      g.C = y; g.ldc = out; g.bias = m->theta + ly.off_b; g.alpha_dev = clip ? scale + nh : nullptr;
      P3D_TRY(tcg::gemm(g, st));
    } else if (x3) {
      GemmArgs g;   // y = h W4 * clip + b4 (W4 split pair: [L][128], segment 64)
      g.M = static_cast<int>(B); g.N = out; g.K = L;
      g.A = w.hs + (nh - 1) * bls; g.lda = ld; g.seg_a = seg;
      g.B = w.ws + w.ws_off[nh]; g.ldb = 128; g.b_mn = 1; g.seg_b = 64;
      g.C = y; g.ldc = out; g.bias = m->theta + ly.off_b; g.alpha_dev = clip ? scale + nh : nullptr;
      P3D_TRY(tcg::gemm(g, st));
    } else {
      Epilogue e; e.bias = m->theta + ly.off_b; e.alpha_dev = clip ? scale + nh : nullptr;
      P3D_TRY(sgemm(false, false, B, out, L, w.h + (nh - 1) * bl, L, m->theta + ly.off_w, out, y, out, e, st));
    }
  }
  const size_t ny = static_cast<size_t>(B) * out;
  loss_dy_kernel<<<egrid(static_cast<long long>(ny)), 256, 0, st>>>(y, t, ny, static_cast<float>(2.0 * invBg / out), w.dy, lossacc,
                                                                          tc ? w.dyb : (x3 ? w.dys : nullptr), out, tc ? kOutPad : 128,
                                                                          x3 ? 64 : 0);
  P3D_LAUNCH_CHECK();
  P3D_TRY(allreduce(m, lossacc, 1, ncclDouble, st));
  // ---------------------------------------------------------------- backward
  float* G[3] = {w.dh, w.dres, w.dres + bl};
  int cur = 0, keepi = -1;
  {
    const Layer& ly = m->layers[nh];
    if (tc) {
      GemmArgs gw;   // dW4 = h^T dy  (reduction over the batch: both operands MN-major, split-K)
      gw.M = L; gw.N = out; gw.K = static_cast<int>(B);
      gw.A = w.hb + (nh - 1) * bl; gw.lda = L; gw.a_mn = 1;
      gw.B = w.dyb; gw.ldb = kOutPad; gw.b_mn = 1;
      gw.C = m->grad + ly.off_w; gw.ldc = out; gw.split_k = 1;
      P3D_TRY(tcg::gemm(gw, st));
    } else if (x3) {
      GemmArgs gw;   // dW4 = h^T dy: both split pairs MN-major, K = batch rows, split-K
      gw.M = L; gw.N = out; gw.K = static_cast<int>(B);
      gw.A = w.hs + (nh - 1) * bls; gw.lda = ld; gw.a_mn = 1; gw.seg_a = seg;
      gw.B = w.dys; gw.ldb = 128; gw.b_mn = 1; gw.seg_b = 64;
      gw.C = m->grad + ly.off_w; gw.ldc = out; gw.split_k = 1;
      P3D_TRY(tcg::gemm(gw, st));
    } else {
      Epilogue e0;
      P3D_TRY(sgemm(true, false, L, out, static_cast<int>(B), w.h + (nh - 1) * bl, L, w.dy, out, m->grad + ly.off_w, out, e0, st));
    }
    colsum_kernel<<<colgrid(out, B), dim3(32, 8), 0, st>>>(w.dy, B, out, m->grad + ly.off_b);
    P3D_LAUNCH_CHECK();
    if (tc) {
      GemmArgs gd;   // dh = dy W4^T * clip
      gd.M = static_cast<int>(B); gd.N = L; gd.K = out;
      gd.A = w.dyb; gd.lda = kOutPad;
      gd.B = w.wb + ly.off_w; gd.ldb = kOutPad;
      gd.C = G[cur]; gd.ldc = L; gd.alpha_dev = clip ? scale + nh : nullptr;
      P3D_TRY(tcg::gemm(gd, st));
    } else if (x3) {
      GemmArgs gd;   // dh = dy W4^T * clip: both K-major (W4 rows are the output rows), K = out
      gd.M = static_cast<int>(B); gd.N = L; gd.K = out;
      gd.A = w.dys; gd.lda = 128; gd.seg_a = 64;
      gd.B = w.ws + w.ws_off[nh]; gd.ldb = 128; gd.seg_b = 64;
      gd.C = G[cur]; gd.ldc = L; gd.alpha_dev = clip ? scale + nh : nullptr;
      P3D_TRY(tcg::gemm(gd, st));
    } else {
      Epilogue e1; e1.alpha_dev = clip ? scale + nh : nullptr;
      P3D_TRY(sgemm(false, true, B, L, out, w.dy, out, m->theta + ly.off_w, out, G[cur], L, e1, st));
    }
  }
  for (int li = nh - 1; li >= 0; --li) {
    const Layer& ly = m->layers[li];
    if (residual && li >= 2 && (li % 2) == 0) keepi = cur;   // d(h[li]) also flows to h[li-2]
    BwdArgs a;
    a.dh = G[cur]; a.z = w.z + li * bl; a.mean = w.mean + static_cast<size_t>(li) * L; a.rstd = w.rstd + static_cast<size_t>(li) * L;
    a.gamma = ly.has_bn ? m->theta + ly.off_gamma : nullptr; a.beta = ly.has_bn ? m->theta + ly.off_beta : nullptr;
    a.mask = maskbuf + li * bl; a.dz = (lowp && ly.has_bn) ? nullptr : w.dz;   // tensor-core + BN: pass B recomputes da
    a.dzb = (tc && !ly.has_bn) ? w.dzb : nullptr; a.sums = w.red + 2ull * li * L; a.sc = sc;
    a.dzs = (x3 && !ly.has_bn) ? w.dzs : nullptr; a.seg = seg;
    a.B = B; a.L = L; a.has_bn = ly.has_bn; a.dropout = dropout;
    bwd_act_kernel<<<dim3((L / 4 + 31) / 32, static_cast<unsigned>((B + RCH4 - 1) / RCH4)), dim3(32, 8), 0, st>>>(a);
    P3D_LAUNCH_CHECK();
    if (ly.has_bn) {
      P3D_TRY(allreduce(m, a.sums, 2ull * L, ncclDouble, st));
      // dz (bf16 only on the tensor-core path) + dgamma / dbeta.  The sums are already global after the all-reduce,
      // so every rank holds the full dgamma/dbeta: pre-divide by world so that the flat gradient all-reduce (a sum)
      // restores them exactly once.
      bwd_bn_kernel<<<egrid(static_cast<long long>(bl / 4)), 256, 0, st>>>(w.dz, a.z, a.mean, a.rstd, a.gamma, a.sums, static_cast<float>(invBg), B, L,
                                                                           tc ? w.dzb : nullptr, lowp ? 0 : 1, 1.0 / m->world,
                                                                           m->grad + ly.off_gamma, m->grad + ly.off_beta,
                                                                           lowp ? a.dh : nullptr, dropout ? a.mask : nullptr, a.beta, sc,
                                                                           x3 ? w.dzs : nullptr, seg);
      P3D_LAUNCH_CHECK();
      // the bias feeding a BN layer has an exactly-zero gradient (it is removed by the mean subtraction)
    } else {
      colsum_kernel<<<colgrid(L, B), dim3(32, 8), 0, st>>>(w.dz, B, L, m->grad + ly.off_b);
      P3D_LAUNCH_CHECK();
    }
    const float* in = li == 0 ? x : w.h + (li - 1) * bl;
    const int lda = li == 0 ? kIn : L;
    if (tc) {
      GemmArgs gw;   // dW = in^T dz
      gw.M = ly.K; gw.N = L; gw.K = static_cast<int>(B);
      gw.A = li == 0 ? w.xb : w.hb + (li - 1) * bl; gw.lda = lda; gw.a_mn = 1;
      gw.B = w.dzb; gw.ldb = L; gw.b_mn = 1;
      gw.C = m->grad + ly.off_w; gw.ldc = L; gw.split_k = 1;
      P3D_TRY(tcg::gemm(gw, st));
    } else if (x3) {
      GemmArgs gw;   // dW = in^T dz: both split pairs MN-major, K = batch rows, split-K
      gw.M = ly.K; gw.N = L; gw.K = static_cast<int>(B);
      gw.A = li == 0 ? w.xs : w.hs + (li - 1) * bls; gw.lda = li == 0 ? 128 : ld; gw.a_mn = 1; gw.seg_a = li == 0 ? 64 : seg;
      gw.B = w.dzs; gw.ldb = ld; gw.b_mn = 1; gw.seg_b = seg;
      gw.C = m->grad + ly.off_w; gw.ldc = L; gw.split_k = 1;
      P3D_TRY(tcg::gemm(gw, st));
    } else {
      Epilogue e0;
      P3D_TRY(sgemm(true, false, ly.K, L, static_cast<int>(B), in, lda, w.dz, L, m->grad + ly.off_w, L, e0, st));
    }
    if (li > 0) {
      int nxt = 0;
      while (nxt == cur || nxt == keepi) ++nxt;
      const bool add = residual && (li % 2) == 1 && keepi >= 0;
      if (tc) {
        GemmArgs gd;   // dh_prev = dz W^T * clip (+ the gradient that bypassed the block)
        gd.M = static_cast<int>(B); gd.N = L; gd.K = L;
        gd.A = w.dzb; gd.lda = L;
        gd.B = w.wb + ly.off_w; gd.ldb = L;
        gd.C = G[nxt]; gd.ldc = L; gd.alpha_dev = clip ? scale + li : nullptr;
        if (add) { gd.res = G[keepi]; gd.ldres = L; }
        P3D_TRY(tcg::gemm(gd, st));
      } else if (x3) {
        GemmArgs gd;   // dh_prev = dz W^T * clip (+ the gradient that bypassed the block): both K-major split pairs
        gd.M = static_cast<int>(B); gd.N = L; gd.K = L;
        gd.A = w.dzs; gd.lda = ld; gd.seg_a = seg;
        gd.B = w.ws + w.ws_off[li]; gd.ldb = ld; gd.seg_b = seg;
        gd.C = G[nxt]; gd.ldc = L; gd.alpha_dev = clip ? scale + li : nullptr;
        if (add) { gd.res = G[keepi]; gd.ldres = L; }
        P3D_TRY(tcg::gemm(gd, st));
      } else {
        Epilogue e1; e1.alpha_dev = clip ? scale + li : nullptr;
        if (add) e1.res = G[keepi];
        P3D_TRY(sgemm(false, true, B, L, L, w.dz, L, m->theta + ly.off_w, L, G[nxt], L, e1, st));
      }
      if (add) keepi = -1;
      cur = nxt;
    }
  }
  }   // unfused path
  // ---------------------------------------------------------------- gradient exchange + update
  P3D_TRY(allreduce(m, m->grad, m->n_train, ncclFloat, st));
  if (clip) {
    clipdot_kernel<<<dim3(148, nlay), 256, 0, st>>>(m->theta, m->grad, tab, dots);
    P3D_LAUNCH_CHECK();
  }
  finish_step_scalars_kernel<<<1, 1, 0, st>>>(lossacc, static_cast<double>(Bg) * out, sc, loss, lr_used);
  P3D_LAUNCH_CHECK();
  const long long n_w = static_cast<long long>(m->layers[nh].off_w) + static_cast<long long>(m->layers[nh].K) * m->layers[nh].N;
  adam_clip_kernel<<<dim3(296, nlay + 1), 256, 0, st>>>(m->theta, m->grad, m->adam_m, m->adam_v, tab, nlay, n_w,
                                                      static_cast<long long>(m->n_train), sc, dots, m->norm2, clip ? 1 : 0);
  P3D_LAUNCH_CHECK();
  return P3D_OK;
}

// One step on inputs that already sit in the staging buffers (w.gx, w.gt): per-step scalars -> device, then the
// body as a CUDA graph captured on a private stream and replayed on the caller's stream (first call of a shape runs
// directly, second captures).  Results land in w.gy / w.gscal.  Single GPU, generated dropout masks.
static int train_step_staged(p3d_model* m, int64_t B, float keep, uint64_t seed, cudaStream_t st, int64_t Bg = 0, int64_t row0 = 0) {
  if (Bg <= 0) Bg = B;
  TrainWorkspace& w = m->tw;
  const bool dropout = keep < 1.f;
  TrainWorkspace::GraphEntry* ge = nullptr;
  for (auto& g : w.graphs) if (g.B == B && g.dropout == (dropout ? 1 : 0) && g.Bg == Bg && g.row0 == row0) ge = &g;
  if (!ge) { w.graphs.push_back(TrainWorkspace::GraphEntry{B, dropout ? 1 : 0, 0, nullptr, Bg, row0}); ge = &w.graphs.back(); }
  if (ge->exec) {
    P3D_CUDA(cudaGraphLaunch(static_cast<cudaGraphExec_t>(ge->exec), st));
    count_launch(ge->launches > 0 ? ge->launches : 0);
    return P3D_OK;
  }
  if (ge->launches == 0) {
    // first step of this shape: run directly (also performs every one-time cudaFuncSetAttribute)
    const long long before = launch_count_now();
    const int rc = train_body(m, w.gx, w.gt, B, dropout, nullptr, Bg, row0, w.gscal, w.gscal + 1, w.gy, st);
    ge->launches = static_cast<int>(launch_count_now() - before);
    if (ge->launches == 0) ge->launches = -1;
    return rc;
  }
  if (!w.cap_stream) P3D_CUDA(cudaStreamCreateWithFlags(&w.cap_stream, cudaStreamNonBlocking));
  cudaGraph_t graph = nullptr;
  P3D_CUDA(cudaStreamBeginCapture(w.cap_stream, cudaStreamCaptureModeThreadLocal));
  int rc = train_body(m, w.gx, w.gt, B, dropout, nullptr, Bg, row0, w.gscal, w.gscal + 1, w.gy, w.cap_stream);
  const cudaError_t ce = cudaStreamEndCapture(w.cap_stream, &graph);
  count_launch(-(ge->launches > 0 ? ge->launches : 0));       // the captured launches did not run
  if (rc != P3D_OK || ce != cudaSuccess || !graph) {
    if (graph) cudaGraphDestroy(graph);
    if (rc == P3D_OK) { set_error("stream capture of the training step failed: %s", cudaGetErrorString(ce)); rc = P3D_ERR_CUDA; }
    return rc;
  }
  cudaGraphExec_t exec = nullptr;
  const cudaError_t ie = cudaGraphInstantiate(&exec, graph, 0);
  cudaGraphDestroy(graph);
  if (ie != cudaSuccess) { set_error("cudaGraphInstantiate failed: %s", cudaGetErrorString(ie)); return P3D_ERR_CUDA; }
  ge->exec = exec;
  P3D_CUDA(cudaGraphLaunch(exec, st));
  count_launch(ge->launches > 0 ? ge->launches : 0);
  return P3D_OK;
}

static int push_scalars(p3d_model* m, float keep, uint64_t seed, cudaStream_t st) {
  // learning-rate schedule (src/linear_model.py:86-90) and TF's bias-corrected step size
  const double tstep = static_cast<double>(m->global_step);
  StepScalars h;
  h.lr_t = m->cfg.learning_rate * powf(0.96f, static_cast<float>(tstep / 100000.0));
  const double tt = tstep + 1.0;
  h.alpha = static_cast<float>(static_cast<double>(h.lr_t) * std::sqrt(1.0 - std::pow(0.999, tt)) / (1.0 - std::pow(0.9, tt)));
  h.keep = keep; h.inv_keep = 1.f / keep;
  h.step = static_cast<unsigned>(m->global_step); h.pad = 0; h.seed = seed;
  set_scalars_kernel<<<1, 1, 0, st>>>(static_cast<StepScalars*>(m->tw.sc), h);
  P3D_LAUNCH_CHECK();
  return P3D_OK;
}

static bool graphs_enabled() {
  static const bool on = [] { const char* e = getenv("P3D_TRAIN_GRAPH"); return !(e && e[0] == '0'); }();
  return on;
}

// model.step(isTraining=True)
int train_step(p3d_model* m, const float* x, const float* t, int64_t B, float keep, uint64_t seed, const uint8_t* mask_in,
               int64_t Bg, int64_t row0, float* loss, float* lr_used, float* y, cudaStream_t st) {
  P3D_TRY(ensure_workspace(m, B));
  TrainWorkspace& w = m->tw;
  P3D_TRY(l2persist_release(m->cfg.device));     // the fused inference kernel's L2 set-aside goes back to normal traffic
  P3D_TRY(push_scalars(m, keep, seed, st));
  // data parallel: the NCCL all-reduces (SyncBN sums, gradient) are captured into the graph with everything else
  static const bool dp_graph = [] { const char* e = getenv("P3D_TRAIN_GRAPH_DP"); return !(e && e[0] == '0'); }();
  if (graphs_enabled() && (m->world == 1 || dp_graph) && mask_in == nullptr) {
    const size_t out = static_cast<size_t>(m->out_size);
    P3D_CUDA(cudaMemcpyAsync(w.gx, x, sizeof(float) * B * kIn, cudaMemcpyDeviceToDevice, st));
    P3D_CUDA(cudaMemcpyAsync(w.gt, t, sizeof(float) * B * out, cudaMemcpyDeviceToDevice, st));
    P3D_TRY(train_step_staged(m, B, keep, seed, st, Bg, row0));
    P3D_CUDA(cudaMemcpyAsync(y, w.gy, sizeof(float) * B * out, cudaMemcpyDeviceToDevice, st));
    if (loss) P3D_CUDA(cudaMemcpyAsync(loss, w.gscal, sizeof(float), cudaMemcpyDeviceToDevice, st));
    if (lr_used) P3D_CUDA(cudaMemcpyAsync(lr_used, w.gscal + 1, sizeof(float), cudaMemcpyDeviceToDevice, st));
  } else {
    const bool dropout = keep < 1.f || mask_in != nullptr;
    P3D_TRY(train_body(m, x, t, B, dropout, mask_in, Bg, row0, loss, lr_used, y, st));
  }
  m->global_step += 1;
  m->pack_valid = false;
  // (set on every call: a replayed graph does not pass through the host code that decides it at capture time)
  m->dp_Bg = Bg;
  m->dp_y_gathered = m->world > 1 && p2p::grad_ready(m) && Bg * m->out_size <= p2p::YMAX;
  return mark_model_work(m, st);
}

// rows perm[start + i] (or start + i) of X / T -> the staging buffers; publishes the previous step's loss
__global__ void gather_batch_kernel(const float* __restrict__ X, const float* __restrict__ T, const long long* __restrict__ perm,
                                    long long start, int B, int out, float* __restrict__ gx, float* __restrict__ gt) {
  const int per_row = kIn + out;
  const long long total = static_cast<long long>(B) * per_row;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total; i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int r = static_cast<int>(i / per_row), c = static_cast<int>(i - static_cast<long long>(r) * per_row);
    const long long src = perm ? perm[start + r] : start + r;
    if (c < kIn) gx[r * kIn + c] = X[src * kIn + c];
    else gt[r * out + (c - kIn)] = T[src * out + (c - kIn)];
  }
}
__global__ void store_loss_kernel(const float* gscal, float* losses, long long idx, float* lr_last) {
  losses[idx] = gscal[0];
  if (lr_last) *lr_last = gscal[1];
}

// The batch loop of predict_3dpose.train() (src/predict_3dpose.py:231-259) over a device-resident training set.
int train_epoch(p3d_model* m, const float* X, const float* T, int64_t n, const long long* perm, int64_t B, float keep, uint64_t seed,
                float* losses, float* lr_last, cudaStream_t st) {
  P3D_REQUIRE(m->world == 1, "train_epoch: data-parallel models step through p3d_model_train_step");
  P3D_TRY(ensure_workspace(m, B));
  P3D_TRY(l2persist_release(m->cfg.device));
  TrainWorkspace& w = m->tw;
  const int64_t nb = n / B;                                   // the n % B tail is dropped (linear_model.py:311-313)
  int g = static_cast<int>((B * (kIn + m->out_size) + 255) / 256);
  if (g > 148 * 4) g = 148 * 4;
  for (int64_t b = 0; b < nb; ++b) {
    P3D_TRY(push_scalars(m, keep, seed, st));
    gather_batch_kernel<<<g, 256, 0, st>>>(X, T, perm, b * B, static_cast<int>(B), m->out_size, w.gx, w.gt);
    P3D_LAUNCH_CHECK();
    if (graphs_enabled()) P3D_TRY(train_step_staged(m, B, keep, seed, st));
    else P3D_TRY(train_body(m, w.gx, w.gt, B, keep < 1.f, nullptr, B, 0, w.gscal, w.gscal + 1, w.gy, st));
    store_loss_kernel<<<1, 1, 0, st>>>(w.gscal, losses, b, lr_last);
    P3D_LAUNCH_CHECK();
    m->global_step += 1;
  }
  m->pack_valid = false;
  return mark_model_work(m, st);
}

}  // namespace train
}  // namespace p3d

using namespace p3d;

extern "C" {

int p3d_model_train_step(p3d_model* m, const float* x, const float* t, int64_t B, float keep_prob, uint64_t seed,
                         const uint8_t* mask_or_null, int64_t global_B, int64_t row0, float* loss, float* lr_used, float* y,
                         void* stream) {
  P3D_REQUIRE(m && x && t && y, "train_step: null argument");
  P3D_REQUIRE(B >= 1, "train_step: empty batch");
  P3D_REQUIRE(keep_prob > 0.f && keep_prob <= 1.f, "train_step: dropout_keep_prob must be in (0,1]");
  if (global_B <= 0) global_B = B;
  P3D_REQUIRE(m->world > 1 || global_B == B, "train_step: global_B != B without a communicator");
  P3D_CUDA(cudaSetDevice(m->cfg.device));
  if (capturing(static_cast<cudaStream_t>(stream))) {      // the step captures and replays CUDA graphs of its own
    set_error("train_step cannot be captured into a CUDA graph (only inference calls can)");
    return P3D_ERR_STATE;
  }
  return train::train_step(m, x, t, B, keep_prob, seed, mask_or_null, global_B, row0, loss, lr_used, y, static_cast<cudaStream_t>(stream));
}

int p3d_model_train_epoch(p3d_model* m, const float* X, const float* T, int64_t n, const int64_t* perm_or_null, int64_t batch_size,
                          float keep_prob, uint64_t seed, float* losses, float* lr_last_or_null, void* stream) {
  P3D_REQUIRE(m && X && T && losses, "train_epoch: null argument");
  P3D_REQUIRE(batch_size >= 1 && n >= 0, "train_epoch: bad sizes");
  P3D_REQUIRE(keep_prob > 0.f && keep_prob <= 1.f, "train_epoch: dropout_keep_prob must be in (0,1]");
  P3D_CUDA(cudaSetDevice(m->cfg.device));
  if (capturing(static_cast<cudaStream_t>(stream))) {
    set_error("train_epoch cannot be captured into a CUDA graph (only inference calls can)");
    return P3D_ERR_STATE;
  }
  return train::train_epoch(m, X, T, n, reinterpret_cast<const long long*>(perm_or_null), batch_size, keep_prob, seed, losses,
                            lr_last_or_null, static_cast<cudaStream_t>(stream));
}

int p3d_model_set_train_matmul(p3d_model* m, int kind) {
  P3D_REQUIRE(m, "set_train_matmul: null model");
  P3D_REQUIRE(kind == P3D_TRAIN_MATMUL_DEFAULT || kind == P3D_TRAIN_MATMUL_BF16X3, "set_train_matmul: unknown kind %d", kind);
  P3D_REQUIRE(m->cfg.mode != P3D_MODE_BF16 && m->cfg.mode != P3D_MODE_FP16,
              "set_train_matmul: bf16- and fp16-mode models train on their own tcgen05 bf16 route");
  if (kind == m->train_matmul) return P3D_OK;
  P3D_CUDA(cudaSetDevice(m->cfg.device));
  train::drop_graphs(m->tw);        // captured with the other route's launches; the next step captures again
  m->train_matmul = kind;
  return P3D_OK;
}

int p3d_model_gathered_outputs(p3d_model* m, float* y_global, int64_t global_B, void* stream) {
  P3D_REQUIRE(m && y_global && global_B >= 1, "gathered_outputs: bad argument");
  if (m->world <= 1 || !m->dp_y_gathered || global_B != m->dp_Bg) return 1;       // not available: the caller gathers
  const float* src = p2p::gathered_outputs(m);
  if (!src) return 1;
  P3D_CUDA(cudaSetDevice(m->cfg.device));
  P3D_CUDA(cudaMemcpyAsync(y_global, src, sizeof(float) * static_cast<size_t>(global_B) * m->out_size, cudaMemcpyDeviceToDevice,
                           static_cast<cudaStream_t>(stream)));
  return P3D_OK;
}

int p3d_debug_dp_part(p3d_model* m, int what, void* stream) {
  P3D_REQUIRE(m && m->world > 1 && m->tw.stats, "debug_dp_part: needs an attached data-parallel model that has stepped once");
  P3D_CUDA(cudaSetDevice(m->cfg.device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  m->dp_y = nullptr;
  if (what == 0) return train::allreduce(m, m->grad, m->n_train, ncclFloat, st);          // the flat gradient exchange
  return train::allreduce(m, m->tw.stats, 2ull * m->L, ncclDouble, st);                   // one SyncBN-sized exchange
}

int p3d_nccl_unique_id(uint8_t* id_host) {
  P3D_REQUIRE(id_host, "nccl_unique_id: null argument");
  train::NcclApi* api = train::nccl();
  if (!api) return P3D_ERR_NCCL;
  ncclUniqueId id;
  P3D_NCCL(api->GetUniqueId(&id));
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
  memcpy(id_host, &id, 128);
  return P3D_OK;
}

int p3d_model_attach_nccl(p3d_model* m, const uint8_t* id_host, int rank, int world) {
  P3D_REQUIRE(m && id_host && world >= 1 && rank >= 0 && rank < world, "attach_nccl: bad argument");
  train::NcclApi* api = train::nccl();
  if (!api) return P3D_ERR_NCCL;
  P3D_CUDA(cudaSetDevice(m->cfg.device));
  ncclUniqueId id;
  memcpy(&id, id_host, 128);
  ncclComm_t comm;
  P3D_NCCL(api->CommInitRank(&comm, world, id, rank));
  m->nccl_comm = comm; m->rank = rank; m->world = world;
  return P3D_OK;
}

}  // extern "C"
