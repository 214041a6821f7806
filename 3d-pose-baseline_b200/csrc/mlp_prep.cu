// Weight preparation for inference (K0) and input packing.
//
// Folds, per layer, what the reference graph applies at run time:
//   tf.clip_by_norm(w, 1)                   src/linear_model.py:108,123,178,189  (whole-matrix Frobenius clip)
//   tf.layers.batch_normalization(training=False)   :112,181,193 (moving statistics, eps 1e-3)
// into  W' = W * clip_scale * s,  b' = (b - moving_mean) * s + beta,  s = gamma / sqrt(moving_var + eps)
// and writes them (a) fp32 [K,N] for the FFMA path and (b) bf16 transposed [N,Kpad] (K contiguous) for
// the tcgen05 path, all layers stacked along rows (fp16 instead of bf16 for P3D_MODE_FP16 models); bf16x3 models also
// get (c) the split pair of (b), bf16(W') and bf16(W' - bf16(W')), side by side in each row.
#include <cstring>

#include "common.cuh"

namespace p3d {
namespace prep {

__global__ void sumsq_kernel(const float* __restrict__ w, size_t n, double* __restrict__ out) {
  double acc = 0.0;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const double v = w[i];
    acc += v * v;
  }
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  __shared__ double part[32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) part[warp] = acc;
  __syncthreads();
  if (warp == 0) {
    acc = lane < (blockDim.x >> 5) ? part[lane] : 0.0;
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) atomicAdd(out, acc);
  }
}

struct FoldArgs {
  const float* W;      // [K,N]
  const float* b;      // [N]
  const float* gamma;  // [N] or null
  const float* beta;
  const float* mm;
  const float* mv;
  const double* norm2; // ||W||_F^2 (device) or null when max_norm is off
  float* wfold;        // [K,N]
  __nv_bfloat16* wt;   // [N rows starting at row_off][kpad]
  __nv_bfloat16* wt3;  // bf16x3 models: [N rows starting at row_off][2 seg3], hi = bf16(W'), lo = bf16(W' - hi); else null
  float* bias_fold;    // [N] starting at row_off
  int K, N, kpad, seg3;
};

template <bool F16>
__global__ void fold_pack_kernel(const FoldArgs a) {
  __shared__ float tile[32][33];
  const int n0 = blockIdx.x * 32, k0 = blockIdx.y * 32;
  float clip = 1.f;
  if (a.norm2) {
    const float nrm = static_cast<float>(sqrt(*a.norm2));
    clip = 1.f / fmaxf(nrm, 1.f);
  }
  // read [k][n] coalesced along n
  for (int kk = threadIdx.y; kk < 32; kk += blockDim.y) {
    const int k = k0 + kk, n = n0 + threadIdx.x;
    float v = 0.f;
    if (k < a.K && n < a.N) {
      float s = 1.f;
      if (a.gamma) s = a.gamma[n] / sqrtf(a.mv[n] + kBnEps);
      v = a.W[static_cast<size_t>(k) * a.N + n] * clip * s;
      a.wfold[static_cast<size_t>(k) * a.N + n] = v;
    }
    tile[kk][threadIdx.x] = v;
  }
  __syncthreads();
  // write [n][k] coalesced along k
  for (int nn = threadIdx.y; nn < 32; nn += blockDim.y) {
    const int n = n0 + nn, k = k0 + threadIdx.x;
    if (n < a.N && k < a.K) {
      const float v = tile[threadIdx.x][nn];
      if constexpr (F16) {
        reinterpret_cast<__half*>(a.wt)[static_cast<size_t>(n) * a.kpad + k] = __float2half_rn(v);
        continue;
      }
      const __nv_bfloat16 hi = __float2bfloat16_rn(v);
      a.wt[static_cast<size_t>(n) * a.kpad + k] = hi;
      if (a.wt3) {
        __nv_bfloat16* row = a.wt3 + static_cast<size_t>(n) * 2 * a.seg3;
        row[k] = hi;
        row[a.seg3 + k] = __float2bfloat16_rn(v - __bfloat162float(hi));
      }
    }
  }
  if (blockIdx.y == 0 && threadIdx.y == 0) {
    const int n = n0 + threadIdx.x;
    if (n < a.N) {
      float bb = a.b[n];
      if (a.gamma) {
        const float s = a.gamma[n] / sqrtf(a.mv[n] + kBnEps);
        bb = (bb - a.mm[n]) * s + a.beta[n];
      }
      a.bias_fold[n] = bb;
    }
  }
}

// x fp32 [B,32] -> bf16 (fp16: F16) [B,64], columns 32..63 zero (layer 0 runs as one K=64 swizzle atom)
template <bool F16>
__global__ void pack_input_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ xb, long long B) {
  using O = Op16<F16>;
  const long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;   // one 8-element group
  if (idx >= B * 8) return;
  const long long row = idx >> 3;
  const int g = static_cast<int>(idx & 7);
  uint4 o = make_uint4(0, 0, 0, 0);
  if (g < 4) {
    const float4* xp = reinterpret_cast<const float4*>(x + row * kIn + g * 8);
    const float4 a = __ldg(xp), b = __ldg(xp + 1);
    typename O::T2 p0 = O::pack(a.x, a.y), p1 = O::pack(a.z, a.w);
    typename O::T2 p2 = O::pack(b.x, b.y), p3 = O::pack(b.z, b.w);
    o.x = *reinterpret_cast<uint32_t*>(&p0); o.y = *reinterpret_cast<uint32_t*>(&p1);
    o.z = *reinterpret_cast<uint32_t*>(&p2); o.w = *reinterpret_cast<uint32_t*>(&p3);
  }
  reinterpret_cast<uint4*>(xb)[idx] = o;
}

// bf16x3: x fp32 [B,32] -> split pair [B,128]: hi = bf16(x) in columns 0..31, lo = bf16(x - hi) in 64..95, zeros
// elsewhere (each half is one K=64 segment of the layer-0 GEMM)
__global__ void pack_input_split_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ xs, long long B) {
  const long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;   // one 8-element group
  if (idx >= B * 16) return;
  const long long row = idx >> 4;
  const int g = static_cast<int>(idx & 15);
  uint4 o = make_uint4(0, 0, 0, 0);
  if ((g & 7) < 4) {
    const float4* xp = reinterpret_cast<const float4*>(x + row * kIn + (g & 7) * 8);
    const float4 a = __ldg(xp), b = __ldg(xp + 1);
    float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    __nv_bfloat16 h[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      h[j] = __float2bfloat16_rn(v[j]);
      if (g >= 8) h[j] = __float2bfloat16_rn(v[j] - __bfloat162float(h[j]));
    }
    memcpy(&o, h, 16);
  }
  reinterpret_cast<uint4*>(xs)[idx] = o;
}

int prepare(p3d_model* m, cudaStream_t st) {
  const int nl = static_cast<int>(m->layers.size());
  P3D_CUDA(cudaMemsetAsync(m->wt_bf16, 0, sizeof(__nv_bfloat16) * static_cast<size_t>(m->rows_total) * m->kpad, st));
  if (m->cfg.max_norm) {
    P3D_CUDA(cudaMemsetAsync(m->norm2, 0, sizeof(double) * nl, st));
    for (int l = 0; l < nl; ++l) {
      const Layer& ly = m->layers[l];
      const size_t n = static_cast<size_t>(ly.K) * ly.N;
      int blocks = static_cast<int>((n + 256 * 8 - 1) / (256 * 8));
      if (blocks > 1024) blocks = 1024;
      sumsq_kernel<<<blocks, 256, 0, st>>>(m->theta + ly.off_w, n, m->norm2 + l);
      P3D_LAUNCH_CHECK();
    }
  }
  for (int l = 0; l < nl; ++l) {
    const Layer& ly = m->layers[l];
    FoldArgs a;
    a.W = m->theta + ly.off_w; a.b = m->theta + ly.off_b;
    if (ly.has_bn) {
      a.gamma = m->theta + ly.off_gamma; a.beta = m->theta + ly.off_beta;
      a.mm = m->moving + ly.off_mm; a.mv = m->moving + ly.off_mv;
    } else {
      a.gamma = a.beta = a.mm = a.mv = nullptr;
    }
    a.norm2 = m->cfg.max_norm ? m->norm2 + l : nullptr;
    a.wfold = m->wfold + ly.off_wfold;
    a.wt = m->wt_bf16 + static_cast<size_t>(ly.row_off) * m->kpad;
    // the split pair is rewritten in place like wt_bf16; its padding columns were zeroed at model creation
    a.wt3 = m->wt_x3 ? m->wt_x3 + static_cast<size_t>(ly.row_off) * 2 * m->x3_seg : nullptr;
    a.bias_fold = m->bias_fold + ly.row_off;
    a.K = ly.K; a.N = ly.N; a.kpad = m->kpad; a.seg3 = m->x3_seg;
    dim3 grid((ly.N + 31) / 32, (ly.K + 31) / 32), block(32, 8);
    if (m->cfg.mode == P3D_MODE_FP16) fold_pack_kernel<true><<<grid, block, 0, st>>>(a);
    else fold_pack_kernel<false><<<grid, block, 0, st>>>(a);
    P3D_LAUNCH_CHECK();
  }
  m->pack_valid = true;
  return P3D_OK;
}

int pack_input(const float* x, __nv_bfloat16* xb, int64_t B, bool f16, cudaStream_t st) {
  const long long groups = B * 8;
  const unsigned blocks = static_cast<unsigned>((groups + 255) / 256);
  if (f16) pack_input_kernel<true><<<blocks, 256, 0, st>>>(x, xb, B);
  else pack_input_kernel<false><<<blocks, 256, 0, st>>>(x, xb, B);
  P3D_LAUNCH_CHECK();
  return P3D_OK;
}

int pack_input_split(const float* x, __nv_bfloat16* xs, int64_t B, cudaStream_t st) {
  const long long groups = B * 16;
  pack_input_split_kernel<<<static_cast<unsigned>((groups + 255) / 256), 256, 0, st>>>(x, xs, B);
  P3D_LAUNCH_CHECK();
  return P3D_OK;
}

}  // namespace prep
}  // namespace p3d
