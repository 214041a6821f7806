// Evaluation kernels (K5): un-normalise -> per-pose Procrustes alignment -> per-joint error (MPJPE).
//   predict_3dpose.evaluate_batches arithmetic   src/predict_3dpose.py:399-442
//   procrustes.compute_similarity_transform      src/procrustes.py:2-63
//
// Two implementations of the same entry point:
//  * mpjpe_f32_kernel (default, p3d_procrustes_mpjpe): HBM-bound design.  Every lane owns ONE pose (the
//    serial 3x3 solve keeps 32 lanes busy instead of one lane per warp).  Each WARP streams its own
//    32-pose tiles with cp.async into a private shared-memory slab (row pitch padded so that the per-lane
//    LDS.128 row reads are conflict free), pulls its row into registers, immediately re-issues the
//    cp.async of its next tile, and does all arithmetic in fp32 registers (one-sided Jacobi, math_hd.h)
//    while that copy is in flight - no block barrier anywhere.  Per-joint sums: fp32 per lane, flushed
//    through warp shuffles into fp64 atomics.  Measured against the fp64 oracle: MPJPE 2e-7 mm,
//    per-joint means 3e-6 mm, worst single per-pose distance 8e-4 mm (tolerance 1e-3 mm).
//  * procrustes_mpjpe_kernel (p3d_procrustes_mpjpe_f64): the all-fp64 form (fp64-pipe bound, ~3x slower),
//    kept for callers that want per-pose distances to 1e-6 mm.
#include "common.cuh"
#include "math_hd.h"

namespace p3d {
namespace evalk {

constexpr int PB = 128;        // poses per block iteration
constexpr int MAXJ = 17;

struct EvalArgs {
  double mean[48], stdv[48];   // gathered to the used dims (hip excluded)
  double hip[3];               // un-normalised hip = mean3d[0:3] (ignored dims come back as the mean)
  int width;                   // 48 or 42
  int J;                       // joints in the error: 17 (hip + 16) or 14
  int with_hip;                // 1 unless predict_14
  int use_procrustes;
};

__device__ __forceinline__ double warp_sum(double v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---- segmented evaluation (p3d_mpjpe_segments): KINDS = 0 is the unsegmented kernel; otherwise the bitmask of
// distances summed per segment (1 plain, 2 Procrustes-aligned), always with the squared error of the normalised rows.
// Per segment s the sums are [2J+1] doubles: J plain joint sums, J aligned joint sums, the squared-error sum.
constexpr int MAX_SEG = 1024;
struct SegTable {              // segment s holds the global rows [off[s], off[s+1]); row i of the call is global row0 + i
  long long off[MAX_SEG + 1];
  long long row0;
  int S;
};
template <class A> struct SegArgs : A { SegTable t; };
template <class A, int KINDS> using ArgsOf = typename std::conditional<KINDS == 0, A, SegArgs<A>>::type;

// The segment of global row g (the last s with off[s] <= g).  Called with a warp-uniform g: every read of the
// parameter bank is a broadcast.
__device__ __forceinline__ int seg_find(const SegTable& t, long long g, int hint) {
  if (hint >= 0 && t.off[hint] <= g && g < t.off[hint + 1]) return hint;
  int lo = 0, hi = t.S - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (t.off[mid] <= g) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// A tile that straddles segments: one warp sum per distinct segment of the live lanes (lane segment ls),
// dst[ls * stride + i] += v[i] for i < n.
template <int NV, typename F>
__device__ __forceinline__ void seg_scatter(const F* v, int n, bool live, int ls, double* dst, int stride) {
  const int lane = threadIdx.x & 31;
  unsigned pending = __ballot_sync(0xffffffffu, live);
  while (pending) {
    const int u = __shfl_sync(0xffffffffu, ls, __ffs(pending) - 1);
    const bool mine = live && ls == u;
    pending &= ~__ballot_sync(0xffffffffu, mine);
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      if (i < n) {
        const double s = warp_sum(mine ? static_cast<double>(v[i]) : 0.0);
        if (lane == 0) atomicAdd(dst + static_cast<long long>(u) * stride + i, s);
      }
    }
  }
}

// Per-warp segment state of a 32-pose tile whose first pose is global row g0 and which holds nlive poses: the segment
// of the tile's first pose, whether the whole tile lies in it, and this lane's own segment.
struct TileSeg {
  int s, ls;
  bool whole;
};
__device__ __forceinline__ TileSeg tile_segment(const SegTable& t, long long g0, int nlive, int lane, int hint) {
  TileSeg r;
  r.s = seg_find(t, g0, hint);
  r.whole = g0 + nlive - 1 < t.off[r.s + 1];
  r.ls = r.s;
  if (!r.whole && lane < nlive)
    while (t.off[r.ls + 1] <= g0 + lane) ++r.ls;
  return r;
}

// KINDS != 0 (segmented): each warp keeps the sums of its current segment per lane (fp64) and flushes them whenever
// its segment changes; joint_sum is then the [S][2J+1] table.  Two kinds hold two more per-lane arrays: 2 blocks/SM.
template <int KINDS = 0>
__global__ void __launch_bounds__(PB, KINDS == 0 ? 4 : (KINDS == 3 ? 2 : 3))
    procrustes_mpjpe_kernel(const float* __restrict__ pred, const float* __restrict__ gt,
                            const __grid_constant__ ArgsOf<EvalArgs, KINDS> a, float* __restrict__ dists,
                            double* __restrict__ joint_sum, long long N) {
  extern __shared__ float sm[];
  const int W = a.width, WP = a.width + 1;      // padded row pitch: conflict-free per-lane rows
  float* sp = sm;
  float* sg = sm + PB * WP;
  __shared__ double sacc[PB / 32][MAXJ];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  double jacc[MAXJ];
#pragma unroll
  for (int j = 0; j < MAXJ; ++j) jacc[j] = 0.0;
  // segmented: jacc sums the first requested kind, kacc the plain distance when both are, qacc the squared error
  constexpr int NK = KINDS == 3 ? MAXJ : 1;
  double kacc[NK], qacc = 0.0;
#pragma unroll
  for (int j = 0; j < NK; ++j) kacc[j] = 0.0;
  int cur = -1, since_flush = 0;
  auto flush = [&](int s) {
    const int J = a.J, st = 2 * J + 1;
    double* dst = joint_sum + static_cast<long long>(s) * st;
#pragma unroll
    for (int j = 0; j < MAXJ; ++j) {
      if (j < J) {
        const double u = warp_sum(jacc[j]);
        if (lane == 0) atomicAdd(dst + (KINDS == 1 ? 0 : J) + j, u);
        if constexpr (KINDS == 3) {
          const double v = warp_sum(kacc[j]);
          if (lane == 0) atomicAdd(dst + j, v);
        }
      }
      jacc[j] = 0.0;
      if (j < NK) kacc[j] = 0.0;
    }
    const double q = warp_sum(qacc);
    if (lane == 0) atomicAdd(dst + 2 * J, q);
    qacc = 0.0;
  };
  const long long ntiles = (N + PB - 1) / PB;
  const long long per = (ntiles + gridDim.x - 1) / gridDim.x;      // segmented: contiguous tiles per block (see fp32)
  const long long tend = KINDS == 0 ? ntiles : (blockIdx.x * per + per < ntiles ? blockIdx.x * per + per : ntiles);
  for (long long tile = KINDS == 0 ? blockIdx.x : blockIdx.x * per; tile < tend; tile += KINDS == 0 ? gridDim.x : 1) {
    const long long p0 = tile * PB;
    const int np = static_cast<int>((N - p0 < PB) ? (N - p0) : PB);
    const int tot = np * W;
    const float* gp = pred + p0 * W;
    const float* gg = gt + p0 * W;
    if ((W & 3) == 0) {
      for (int i = tid; i < tot / 4; i += PB) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(gp) + i);
        const float4 u = __ldg(reinterpret_cast<const float4*>(gg) + i);
        const int e = i * 4, r = e / W, c = e - r * W;
        float* d = sp + r * WP + c; d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
        float* f = sg + r * WP + c; f[0] = u.x; f[1] = u.y; f[2] = u.z; f[3] = u.w;
      }
    } else {   // width 42: rows are only 8-byte aligned
      for (int i = tid; i < tot / 2; i += PB) {
        const float2 v = __ldg(reinterpret_cast<const float2*>(gp) + i);
        const float2 u = __ldg(reinterpret_cast<const float2*>(gg) + i);
        const int e = i * 2, r = e / W, c = e - r * W;
        sp[r * WP + c] = v.x; sp[r * WP + c + 1] = v.y;
        sg[r * WP + c] = u.x; sg[r * WP + c + 1] = u.y;
      }
    }
    __syncthreads();
    const bool live = tid < np;
    const float* mp = sp + tid * WP;
    const float* mg = sg + tid * WP;
    const int J = a.J, J0 = a.with_hip;          // joints J0..J-1 come from the arrays, joint 0 is the hip
    double dj[MAXJ], dk[NK], sq = 0.0;
#pragma unroll
    for (int j = 0; j < MAXJ; ++j) dj[j] = 0.0;
#pragma unroll
    for (int j = 0; j < NK; ++j) dk[j] = 0.0;
    constexpr int ALIGN_KIND = KINDS & 2;
    if (live) {
      double T[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
      double b = 1.0, c0 = 0.0, c1 = 0.0, c2 = 0.0;
      if constexpr (KINDS != 0) {
        for (int k = 0; k < W; ++k) {
          const double e = static_cast<double>(mp[k]) - static_cast<double>(mg[k]);
          sq += e * e;
        }
      }
      if (KINDS == 0 ? a.use_procrustes : ALIGN_KIND) {
        // means (X = ground truth, Y = prediction)
        double mx[3] = {0, 0, 0}, my[3] = {0, 0, 0};
        if (J0) { for (int d = 0; d < 3; ++d) { mx[d] = a.hip[d]; my[d] = a.hip[d]; } }
        for (int k = 0; k < W; k += 3) {
#pragma unroll
          for (int d = 0; d < 3; ++d) {
            mx[d] += static_cast<double>(mg[k + d]) * a.stdv[k + d] + a.mean[k + d];
            my[d] += static_cast<double>(mp[k + d]) * a.stdv[k + d] + a.mean[k + d];
          }
        }
        const double invJ = 1.0 / J;
        for (int d = 0; d < 3; ++d) { mx[d] *= invJ; my[d] *= invJ; }
        double ssx = 0, ssy = 0, A[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
        for (int j = 0; j < J; ++j) {
          double x[3], y[3];
          if (J0 && j == 0) {
            for (int d = 0; d < 3; ++d) { x[d] = a.hip[d] - mx[d]; y[d] = a.hip[d] - my[d]; }
          } else {
            const int k = (j - J0) * 3;
            for (int d = 0; d < 3; ++d) {
              x[d] = static_cast<double>(mg[k + d]) * a.stdv[k + d] + a.mean[k + d] - mx[d];
              y[d] = static_cast<double>(mp[k + d]) * a.stdv[k + d] + a.mean[k + d] - my[d];
            }
          }
          for (int d = 0; d < 3; ++d) { ssx += x[d] * x[d]; ssy += y[d] * y[d]; }
          for (int r = 0; r < 3; ++r)
            for (int s = 0; s < 3; ++s) A[r * 3 + s] += x[r] * y[s];
        }
        const double normX = sqrt(ssx), normY = sqrt(ssy);
        const double inv = 1.0 / (normX * normY);
        for (int i = 0; i < 9; ++i) A[i] *= inv;          // A = X0^T Y0 of the unit-norm point sets
        double tr;
        kabsch_rotation(A, T, tr);
        b = tr * normX / normY;                            // compute_optimal_scale=True (procrustes.py:52-55)
        c0 = mx[0] - b * (my[0] * T[0] + my[1] * T[3] + my[2] * T[6]);
        c1 = mx[1] - b * (my[0] * T[1] + my[1] * T[4] + my[2] * T[7]);
        c2 = mx[2] - b * (my[0] * T[2] + my[1] * T[5] + my[2] * T[8]);
      }
#pragma unroll
      for (int j = 0; j < MAXJ; ++j) {
        if (j < J) {
          double x[3], y[3];
          if (J0 && j == 0) {
            for (int d = 0; d < 3; ++d) { x[d] = a.hip[d]; y[d] = a.hip[d]; }
          } else {
            const int k = (j - J0) * 3;
            for (int d = 0; d < 3; ++d) {
              x[d] = static_cast<double>(mg[k + d]) * a.stdv[k + d] + a.mean[k + d];
              y[d] = static_cast<double>(mp[k + d]) * a.stdv[k + d] + a.mean[k + d];
            }
          }
          double o0 = y[0], o1 = y[1], o2 = y[2];
          if constexpr (KINDS == 3) {
            const double e0 = y[0] - x[0], e1 = y[1] - x[1], e2 = y[2] - x[2];
            dk[j] = static_cast<double>(sqrtf(static_cast<float>(e0 * e0 + e1 * e1 + e2 * e2)));
          }
          if (KINDS == 0 ? a.use_procrustes : ALIGN_KIND) {     // out = b * out.dot(T) + c  (predict_3dpose.py:419)
            o0 = b * (y[0] * T[0] + y[1] * T[3] + y[2] * T[6]) + c0;
            o1 = b * (y[0] * T[1] + y[1] * T[4] + y[2] * T[7]) + c1;
            o2 = b * (y[0] * T[2] + y[1] * T[5] + y[2] * T[8]) + c2;
          }
          const double e0 = o0 - x[0], e1 = o1 - x[1], e2 = o2 - x[2];
          // the squared error is fp64; its root in fp32 (rel. 6e-8, i.e. < 1e-5 mm) avoids 17 software fp64 sqrt per pose
          dj[j] = static_cast<double>(sqrtf(static_cast<float>(e0 * e0 + e1 * e1 + e2 * e2)));
        } else {
          dj[j] = 0.0;
        }
      }
      if (dists) {
        float* dp = dists + (p0 + tid) * J;
#pragma unroll
        for (int j = 0; j < MAXJ; ++j) if (j < J) dp[j] = static_cast<float>(dj[j]);
      }
    }
    if constexpr (KINDS == 0) {
#pragma unroll
      for (int j = 0; j < MAXJ; ++j) {
        const double v = (live && j < J) ? dj[j] : 0.0;
        jacc[j] += v;
      }
    } else if (warp * 32 < np) {
      const int nlive = np - warp * 32 < 32 ? np - warp * 32 : 32;
      const TileSeg ts = tile_segment(a.t, a.t.row0 + p0 + warp * 32, nlive, lane, cur);
      if (cur >= 0 && (!ts.whole || ts.s != cur)) { flush(cur); since_flush = 0; }
      cur = ts.whole ? ts.s : -1;
      if (ts.whole) {
#pragma unroll
        for (int j = 0; j < MAXJ; ++j) {
          jacc[j] += dj[j];
          if (j < NK) kacc[j] += dk[j];
        }
        qacc += sq;
        if (++since_flush == 64) { flush(cur); since_flush = 0; }
      } else {
        const int st = 2 * J + 1;
        seg_scatter<MAXJ>(dj, J, live, ts.ls, joint_sum + (KINDS == 1 ? 0 : J), st);
        if (KINDS == 3) seg_scatter<NK>(dk, J, live, ts.ls, joint_sum, st);
        seg_scatter<1>(&sq, 1, live, ts.ls, joint_sum + 2 * J, st);
      }
    }
    __syncthreads();
  }
  if constexpr (KINDS != 0) {
    if (cur >= 0) flush(cur);
  } else {
    // block reduction: shuffles within the warp, shared memory across warps, one atomic per joint
#pragma unroll
    for (int j = 0; j < MAXJ; ++j) {
      const double s = warp_sum(jacc[j]);
      if (lane == 0) sacc[warp][j] = s;
    }
    __syncthreads();
    if (tid < a.J) {
      double s = 0;
      for (int w = 0; w < PB / 32; ++w) s += sacc[w][tid];
      atomicAdd(joint_sum + tid, s);
    }
  }
}

// ------------------------------------------------------------------ fp32, warp-autonomous, cp.async fed
template <int W> struct EvalLayout;
template <> struct EvalLayout<48> { static constexpr int PITCH = 52, CB = 16, CPR = 12; };   // padded rows, 16 B chunks
template <> struct EvalLayout<42> { static constexpr int PITCH = 42, CB = 8, CPR = 21; };    // dense rows, 8 B chunks

struct EvalArgsF {
  float sd[48], mc[48], hipc[3];
  int use_procrustes;
};

template <int CB>
__device__ __forceinline__ void cp_async_zfill(uint32_t dst, const void* src, int src_bytes) {
  if (CB == 16) asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
  else asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}

constexpr int EV_WARPS = 4;
#ifndef EV_BLOCKS
#define EV_BLOCKS 3   // 4 blocks (128 registers) spills and is 40% slower; 3 blocks = 168 registers, no hot spills
#endif

// KINDS != 0 (segmented): the fp32 per-lane sums belong to the warp's current segment and are flushed whenever it
// changes; a tile that straddles segments goes straight to the atomics, one warp sum per distinct segment.  joint_sum
// is then the [S][2J+1] table.  Both kinds hold J more accumulators: 2 blocks/SM (DESIGN 3.4).
template <int W, int J0, int KINDS = 0>
__global__ void __launch_bounds__(EV_WARPS * 32, KINDS == 3 ? 2 : EV_BLOCKS)
    mpjpe_f32_kernel(const float* __restrict__ pred, const float* __restrict__ gt, const __grid_constant__ ArgsOf<EvalArgsF, KINDS> a,
                     float* __restrict__ dists, double* __restrict__ joint_sum, long long N) {
  using LY = EvalLayout<W>;
  constexpr int J = W / 3 + J0;
  constexpr int ROW_BYTES = LY::PITCH * 4;
  constexpr int ARR_BYTES = 32 * ROW_BYTES;
  constexpr int CB = LY::CB, CPR = LY::CPR;
  extern __shared__ __align__(16) uint8_t ev_smem[];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  uint8_t* buf = ev_smem + wib * 2 * ARR_BYTES;          // [gt | pred] slab of this warp
  const uint32_t sbuf = static_cast<uint32_t>(__cvta_generic_to_shared(buf));
  const long long ntiles = (N + 31) / 32;
  const long long nwarps = static_cast<long long>(gridDim.x) * EV_WARPS;
  // segmented: each warp walks a contiguous range of tiles, so its segment changes about once per boundary it meets
  // instead of at nearly every tile of a strided walk
  const long long gwarp = static_cast<long long>(blockIdx.x) * EV_WARPS + wib;
  const long long per = (ntiles + nwarps - 1) / nwarps;
  const long long tend = KINDS == 0 ? ntiles : (gwarp * per + per < ntiles ? gwarp * per + per : ntiles);
  const long long tstep = KINDS == 0 ? nwarps : 1;
  const uint8_t* gbytes = reinterpret_cast<const uint8_t*>(gt);
  const uint8_t* pbytes = reinterpret_cast<const uint8_t*>(pred);

  auto issue = [&](long long tile) {
    if (tile < tend) {
      const long long base = tile * 32 * W * 4;
      const long long rem = N * W * 4 - base;             // valid bytes of this tile (rows are multiples of CB)
#pragma unroll
      for (int n = 0; n < CPR; ++n) {
        const int i = lane + 32 * n;                       // chunk index inside the tile
        const int soff = (i / CPR) * ROW_BYTES + (i % CPR) * CB;
        const long long gb = static_cast<long long>(i) * CB;
        const bool ok = gb < rem;
        cp_async_zfill<CB>(sbuf + soff, gbytes + (ok ? base + gb : 0), ok ? CB : 0);
        cp_async_zfill<CB>(sbuf + ARR_BYTES + soff, pbytes + (ok ? base + gb : 0), ok ? CB : 0);
      }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };

  // per-lane sums: J joint sums; segmented, J per requested kind and the squared error last
  constexpr int NA = KINDS == 0 ? J : ((KINDS & 1) + (KINDS >> 1)) * J + 1;
  constexpr int STRIDE = 2 * J + 1;
  float acc[NA];
#pragma unroll
  for (int j = 0; j < NA; ++j) acc[j] = 0.f;
  auto flush = [&](double* dst) {
#pragma unroll
    for (int j = 0; j < NA; ++j) {
      const double s = warp_sum(static_cast<double>(acc[j]));
      const int slot = KINDS == 0 ? j : (j == NA - 1 ? 2 * J : (KINDS == 2 ? J + j : j));
      if (lane == 0) atomicAdd(dst + slot, s);
      acc[j] = 0.f;
    }
  };

  long long tile = KINDS == 0 ? gwarp : gwarp * per;
  issue(tile);
  int since_flush = 0, cur = -1;
  for (; tile < tend; tile += tstep) {
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncwarp();
    float g[W], p[W];
    const uint8_t* row = buf + lane * ROW_BYTES;
    if (CB == 16) {
#pragma unroll
      for (int c = 0; c < W / 4; ++c) {
        const float4 u = *reinterpret_cast<const float4*>(row + c * 16);
        const float4 v = *reinterpret_cast<const float4*>(row + ARR_BYTES + c * 16);
        g[4 * c] = u.x; g[4 * c + 1] = u.y; g[4 * c + 2] = u.z; g[4 * c + 3] = u.w;
        p[4 * c] = v.x; p[4 * c + 1] = v.y; p[4 * c + 2] = v.z; p[4 * c + 3] = v.w;
      }
    } else {
#pragma unroll
      for (int c = 0; c < W / 2; ++c) {
        const float2 u = *reinterpret_cast<const float2*>(row + c * 8);
        const float2 v = *reinterpret_cast<const float2*>(row + ARR_BYTES + c * 8);
        g[2 * c] = u.x; g[2 * c + 1] = u.y;
        p[2 * c] = v.x; p[2 * c + 1] = v.y;
      }
    }
    __syncwarp();                       // every lane holds its row: the slab can take the next tile
    issue(tile + tstep);
    const long long pose = tile * 32 + lane;
    const bool live = pose < N;
    if constexpr (KINDS == 0) {
      float dj[J];
      pose_errors_f32<W, J0>(g, p, a.sd, a.mc, a.hipc, a.use_procrustes, dj);
      if (dists && live) {
        float* dp = dists + pose * J;
#pragma unroll
        for (int j = 0; j < J; ++j) dp[j] = dj[j];
      }
#pragma unroll
      for (int j = 0; j < J; ++j) acc[j] += live ? dj[j] : 0.f;
      if (++since_flush == 64) { flush(joint_sum); since_flush = 0; }   // bounds the fp32 partial sums (<= 64 terms per lane)
    } else {
      const int nlive = N - tile * 32 < 32 ? static_cast<int>(N - tile * 32) : 32;
      const TileSeg ts = tile_segment(a.t, a.t.row0 + tile * 32, nlive, lane, cur);
      if (cur >= 0 && (!ts.whole || ts.s != cur)) { flush(joint_sum + static_cast<long long>(cur) * STRIDE); since_flush = 0; }
      cur = ts.whole ? ts.s : -1;
      // whole tile: into the lane sums; straddling tile: straight to the segments' atomics
      auto take = [&](const float* v, int at, int n, int slot) {
        if (ts.whole) {
#pragma unroll
          for (int i = 0; i < J; ++i)
            if (i < n) acc[at + i] += live ? v[i] : 0.f;
        } else {
          seg_scatter<J>(v, n, live, ts.ls, joint_sum + slot, STRIDE);
        }
      };
      float sq = 0.f;
#pragma unroll
      for (int k = 0; k < W; ++k) { const float e = p[k] - g[k]; sq = fmaf(e, e, sq); }
      float dj[J];
      if constexpr ((KINDS & 1) != 0) {
        pose_errors_f32<W, J0>(g, p, a.sd, a.mc, a.hipc, 0, dj);
        take(dj, 0, J, 0);
      }
      if constexpr ((KINDS & 2) != 0) {     // last: the aligned form overwrites g and p
        pose_errors_f32<W, J0>(g, p, a.sd, a.mc, a.hipc, 1, dj);
        take(dj, (KINDS & 1) ? J : 0, J, J);
      }
      take(&sq, NA - 1, 1, 2 * J);
      if (ts.whole && ++since_flush == 64) { flush(joint_sum + static_cast<long long>(cur) * STRIDE); since_flush = 0; }
    }
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  if constexpr (KINDS == 0) flush(joint_sum);
  else if (cur >= 0) flush(joint_sum + static_cast<long long>(cur) * STRIDE);
}

// Batched procrustes.compute_similarity_transform on raw fp64 poses; one thread per pose.
__global__ void similarity_transform_kernel(const double* __restrict__ X, const double* __restrict__ Y, int J, int scale,
                                            long long N, double* d_out, double* Z, double* T_out, double* b_out, double* c_out) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < N;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const double* x = X + i * J * 3;
    const double* y = Y + i * J * 3;
    double mx[3] = {0, 0, 0}, my[3] = {0, 0, 0};
    for (int j = 0; j < J; ++j)
      for (int d = 0; d < 3; ++d) { mx[d] += x[j * 3 + d]; my[d] += y[j * 3 + d]; }
    for (int d = 0; d < 3; ++d) { mx[d] /= J; my[d] /= J; }
    double ssx = 0, ssy = 0, A[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int j = 0; j < J; ++j) {
      double a[3], b[3];
      for (int d = 0; d < 3; ++d) { a[d] = x[j * 3 + d] - mx[d]; b[d] = y[j * 3 + d] - my[d]; ssx += a[d] * a[d]; ssy += b[d] * b[d]; }
      for (int r = 0; r < 3; ++r)
        for (int s = 0; s < 3; ++s) A[r * 3 + s] += a[r] * b[s];
    }
    const double normX = sqrt(ssx), normY = sqrt(ssy);
    const double inv = 1.0 / (normX * normY);
    for (int k = 0; k < 9; ++k) A[k] *= inv;
    double T[9], tr;
    kabsch_rotation(A, T, tr);
    double b, dd, zs;
    if (scale) { b = tr * normX / normY; dd = 1.0 - tr * tr; zs = normX * tr; }
    else { b = 1.0; dd = 1.0 + ssy / ssx - 2.0 * tr * normY / normX; zs = normY; }
    if (d_out) d_out[i] = dd;
    if (b_out) b_out[i] = b;
    if (T_out) for (int k = 0; k < 9; ++k) T_out[i * 9 + k] = T[k];
    if (c_out)
      for (int s = 0; s < 3; ++s) c_out[i * 3 + s] = mx[s] - b * (my[0] * T[s] + my[1] * T[3 + s] + my[2] * T[6 + s]);
    if (Z)
      for (int j = 0; j < J; ++j) {
        const double y0 = (y[j * 3] - my[0]) / normY, y1 = (y[j * 3 + 1] - my[1]) / normY, y2 = (y[j * 3 + 2] - my[2]) / normY;
        for (int s = 0; s < 3; ++s) Z[(i * J + j) * 3 + s] = zs * (y0 * T[s] + y1 * T[3 + s] + y2 * T[6 + s]) + mx[s];
      }
  }
}

}  // namespace evalk
}  // namespace p3d

using namespace p3d;
using namespace p3d::evalk;

namespace {

const int kJ16[16] = {1, 2, 3, 6, 7, 8, 12, 13, 14, 15, 17, 18, 19, 25, 26, 27};
const int kJ14[14] = {1, 2, 3, 6, 7, 8, 13, 15, 17, 18, 19, 25, 26, 27};

void fill_args_f64(EvalArgs& a, const double* mean3d, const double* std3d, int predict_14, int use_procrustes) {
  memset(&a, 0, sizeof(a));
  const int nj = predict_14 ? 14 : 16;
  const int* jt = predict_14 ? kJ14 : kJ16;
  for (int j = 0; j < nj; ++j)
    for (int d = 0; d < 3; ++d) { a.mean[j * 3 + d] = mean3d[jt[j] * 3 + d]; a.stdv[j * 3 + d] = std3d[jt[j] * 3 + d]; }
  for (int d = 0; d < 3; ++d) a.hip[d] = mean3d[d];
  a.width = nj * 3;
  a.with_hip = predict_14 ? 0 : 1;      // dtu3d = [0,1,2] U dim_to_use_3d unless predict_14 (predict_3dpose.py:405)
  a.J = nj + a.with_hip;
  a.use_procrustes = use_procrustes ? 1 : 0;
}

void fill_args_f32(EvalArgsF& a, const double* mean3d, const double* std3d, int predict_14, int use_procrustes) {
  const int nj = predict_14 ? 14 : 16;
  const int* jt = predict_14 ? kJ14 : kJ16;
  const int J = nj + (predict_14 ? 0 : 1);
  // mean over the J joints of the un-normalised MEAN pose (the hip, data_mean_3d[0:3], is joint 0 unless predict_14)
  double mbar[3] = {0, 0, 0};
  for (int d = 0; d < 3; ++d) {
    for (int j = 0; j < nj; ++j) mbar[d] += mean3d[jt[j] * 3 + d];
    if (!predict_14) mbar[d] += mean3d[d];
    mbar[d] /= J;
  }
  memset(&a, 0, sizeof(a));
  for (int j = 0; j < nj; ++j)
    for (int d = 0; d < 3; ++d) {
      a.sd[j * 3 + d] = static_cast<float>(std3d[jt[j] * 3 + d]);
      a.mc[j * 3 + d] = static_cast<float>(mean3d[jt[j] * 3 + d] - mbar[d]);
    }
  for (int d = 0; d < 3; ++d) a.hipc[d] = static_cast<float>(mean3d[d] - mbar[d]);
  a.use_procrustes = use_procrustes ? 1 : 0;
}

template <int KINDS>
void launch_f64(const float* pred_n, const float* gt_n, const ArgsOf<EvalArgs, KINDS>& a, float* dists, double* sums,
                int64_t N, cudaStream_t st) {
  const size_t smem = sizeof(float) * 2 * PB * (a.width + 1);
  const long long ntiles = (N + PB - 1) / PB;
  const int grid = ntiles < 148 * 4 ? (int)ntiles : 148 * 4;
  procrustes_mpjpe_kernel<KINDS><<<grid, PB, smem, st>>>(pred_n, gt_n, a, dists, sums, N);
}

template <int W, int J0, int KINDS>
int launch_f32(const float* pred_n, const float* gt_n, const ArgsOf<EvalArgsF, KINDS>& a, float* dists, double* sums,
               int64_t N, cudaStream_t st) {
  constexpr int smem = EV_WARPS * 2 * 32 * EvalLayout<W>::PITCH * 4;
  constexpr int blocks = KINDS == 3 ? 2 : EV_BLOCKS;     // the kernel's __launch_bounds__
  static PerDeviceOnce attr;
  if (attr.needed()) {
    P3D_CUDA(cudaFuncSetAttribute(mpjpe_f32_kernel<W, J0, KINDS>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    attr.mark();
  }
  const long long ntiles = (N + 31) / 32;
  const long long nblocks = (ntiles + EV_WARPS - 1) / EV_WARPS;
  const int grid = nblocks < 148 * blocks ? (int)nblocks : 148 * blocks;
  mpjpe_f32_kernel<W, J0, KINDS><<<grid, EV_WARPS * 32, smem, st>>>(pred_n, gt_n, a, dists, sums, N);
  return P3D_OK;
}

// Argument checks of p3d_mpjpe_segments[_f64]; fills the segment table of the launch.
int segment_table(const float* pred_n, const float* gt_n, const double* mean3d, const double* std3d, int kinds, int64_t N,
                  int64_t row0, const int64_t* offsets, int S, const double* sums, const char* fn, SegTable& t) {
  P3D_REQUIRE(pred_n && gt_n && mean3d && std3d && offsets && sums && N >= 0, "%s: null argument or N < 0", fn);
  P3D_REQUIRE(S >= 1 && S <= MAX_SEG, "%s: S = %d segments, must be 1..%d", fn, S, MAX_SEG);
  P3D_REQUIRE(kinds >= 1 && kinds <= 3, "%s: kinds = %d, must be 1 (plain), 2 (aligned) or 3 (both)", fn, kinds);
  P3D_REQUIRE(((reinterpret_cast<uintptr_t>(pred_n) | reinterpret_cast<uintptr_t>(gt_n)) & 15) == 0,
              "%s: pred/gt must be 16-byte aligned", fn);
  for (int s = 0; s < S; ++s)
    P3D_REQUIRE(offsets[s] <= offsets[s + 1], "%s: offsets descend at segment %d (%lld > %lld)", fn, s,
                (long long)offsets[s], (long long)offsets[s + 1]);
  P3D_REQUIRE(row0 >= offsets[0] && row0 + N <= offsets[S], "%s: rows [%lld, %lld) lie outside the segments [%lld, %lld)", fn,
              (long long)row0, (long long)(row0 + N), (long long)offsets[0], (long long)offsets[S]);
  for (int s = 0; s <= S; ++s) t.off[s] = offsets[s];
  t.row0 = row0;
  t.S = S;
  return P3D_OK;
}

}  // namespace

extern "C" {

int p3d_procrustes_mpjpe_f64(const float* pred_n, const float* gt_n, const double* mean3d, const double* std3d, int predict_14,
                         int use_procrustes, int64_t N, float* dists, double* joint_sum, void* stream) {
  P3D_REQUIRE(pred_n && gt_n && mean3d && std3d && joint_sum && N >= 0, "procrustes_mpjpe: null argument");
  if (N == 0) return P3D_OK;
  EvalArgs a;
  fill_args_f64(a, mean3d, std3d, predict_14, use_procrustes);
  static PerDeviceOnce attr;
  if (attr.needed()) {
    P3D_CUDA(cudaFuncSetAttribute(procrustes_mpjpe_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
    attr.mark();
  }
  launch_f64<0>(pred_n, gt_n, a, dists, joint_sum, N, (cudaStream_t)stream);
  P3D_LAUNCH_CHECK();
  return P3D_OK;
}

int p3d_procrustes_mpjpe(const float* pred_n, const float* gt_n, const double* mean3d, const double* std3d, int predict_14,
                         int use_procrustes, int64_t N, float* dists, double* joint_sum, void* stream) {
  P3D_REQUIRE(pred_n && gt_n && mean3d && std3d && joint_sum && N >= 0, "procrustes_mpjpe: null argument");
  if (N == 0) return P3D_OK;
  P3D_REQUIRE(((reinterpret_cast<uintptr_t>(pred_n) | reinterpret_cast<uintptr_t>(gt_n)) & 15) == 0,
              "procrustes_mpjpe: pred/gt must be 16-byte aligned");
  EvalArgsF a;
  fill_args_f32(a, mean3d, std3d, predict_14, use_procrustes);
  cudaStream_t st = (cudaStream_t)stream;
  const int rc = predict_14 ? launch_f32<42, 0, 0>(pred_n, gt_n, a, dists, joint_sum, N, st)
                            : launch_f32<48, 1, 0>(pred_n, gt_n, a, dists, joint_sum, N, st);
  if (rc != P3D_OK) return rc;
  P3D_LAUNCH_CHECK();
  return P3D_OK;
}

int p3d_mpjpe_segments(const float* pred_n, const float* gt_n, const double* mean3d, const double* std3d, int predict_14,
                       int kinds, int64_t N, int64_t row0, const int64_t* offsets, int S, double* sums, void* stream) {
  SegArgs<EvalArgsF> a;
  const int rc = segment_table(pred_n, gt_n, mean3d, std3d, kinds, N, row0, offsets, S, sums, "mpjpe_segments", a.t);
  if (rc != P3D_OK) return rc;
  if (N == 0) return P3D_OK;
  fill_args_f32(a, mean3d, std3d, predict_14, 0);
  cudaStream_t st = (cudaStream_t)stream;
  int r;
  if (!predict_14) {
    r = kinds == 1 ? launch_f32<48, 1, 1>(pred_n, gt_n, a, nullptr, sums, N, st)
      : kinds == 2 ? launch_f32<48, 1, 2>(pred_n, gt_n, a, nullptr, sums, N, st)
                   : launch_f32<48, 1, 3>(pred_n, gt_n, a, nullptr, sums, N, st);
  } else {
    r = kinds == 1 ? launch_f32<42, 0, 1>(pred_n, gt_n, a, nullptr, sums, N, st)
      : kinds == 2 ? launch_f32<42, 0, 2>(pred_n, gt_n, a, nullptr, sums, N, st)
                   : launch_f32<42, 0, 3>(pred_n, gt_n, a, nullptr, sums, N, st);
  }
  if (r != P3D_OK) return r;
  P3D_LAUNCH_CHECK();
  return P3D_OK;
}

int p3d_mpjpe_segments_f64(const float* pred_n, const float* gt_n, const double* mean3d, const double* std3d, int predict_14,
                           int kinds, int64_t N, int64_t row0, const int64_t* offsets, int S, double* sums, void* stream) {
  SegArgs<EvalArgs> a;
  const int rc = segment_table(pred_n, gt_n, mean3d, std3d, kinds, N, row0, offsets, S, sums, "mpjpe_segments_f64", a.t);
  if (rc != P3D_OK) return rc;
  if (N == 0) return P3D_OK;
  fill_args_f64(a, mean3d, std3d, predict_14, 0);
  static PerDeviceOnce attr;
  if (attr.needed()) {
    P3D_CUDA(cudaFuncSetAttribute(procrustes_mpjpe_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
    P3D_CUDA(cudaFuncSetAttribute(procrustes_mpjpe_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
    P3D_CUDA(cudaFuncSetAttribute(procrustes_mpjpe_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
    attr.mark();
  }
  cudaStream_t st = (cudaStream_t)stream;
  if (kinds == 1) launch_f64<1>(pred_n, gt_n, a, nullptr, sums, N, st);
  else if (kinds == 2) launch_f64<2>(pred_n, gt_n, a, nullptr, sums, N, st);
  else launch_f64<3>(pred_n, gt_n, a, nullptr, sums, N, st);
  P3D_LAUNCH_CHECK();
  return P3D_OK;
}

int p3d_similarity_transform_f64(const double* X, const double* Y, int J, int compute_optimal_scale, int64_t N, double* d,
                                 double* Z, double* T, double* b, double* c, void* stream) {
  P3D_REQUIRE(X && Y && J >= 1 && N >= 0, "similarity_transform: bad argument");
  if (N == 0) return P3D_OK;
  long long g = (N + 127) / 128;
  if (g > 148 * 8) g = 148 * 8;
  similarity_transform_kernel<<<(int)g, 128, 0, (cudaStream_t)stream>>>(X, Y, J, compute_optimal_scale, N, d, Z, T, b, c);
  P3D_LAUNCH_CHECK();
  return P3D_OK;
}

}  // extern "C"
