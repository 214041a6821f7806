// Fused LinearModel inference on the sm_100a tensor cores (tcgen05 + TMEM + TMA).
//
// Replaces the op-by-op TensorFlow graph of src/linear_model.py:102-125,154-201 at inference
// (isTraining=False): x[B,32] -> Linear+BN+ReLU -> num_layers x (two_linear + residual) -> Linear.
// clip_by_norm and the moving-statistics BatchNorm are folded into W',b' by mlp_prep.cu, so every
// stage is  h' = relu(h W' + b') (+ residual)  and the last one  y = h W' + b'.
//
// One persistent CTA per SM walks 128-pose row tiles through ALL layers:
//   warp 0   TMA producer A: A tile [128 x 64] bf16 of the current activations (gated by the slab barriers of the
//                           previous layer) into the smem ring (128B swizzle)
//   warp 2   TMEM allocator, then TMA producer B: the matching W' tile; weights depend on nothing, so this warp
//                           runs ahead of the layer chain by up to a full ring (+10 % at 16 K poses, where the
//                           layer transitions are a larger share)
//   warp 1   MMA issuer   : tcgen05.mma 128x256x16 (one elected lane, warp-uniform operands), fp32
//                           accumulators in TMEM, 2 x 256 columns double buffered against the epilogue
//   warps 4-7 epilogue    : tcgen05.ld -> +bias -> ReLU -> bf16 -> swizzled smem tile -> TMA store
//                           (cp.reduce.async.bulk .add when the block's residual is added: the L2
//                           performs  P += tile  so the residual is never re-read by the SM), or fp32 y
// Layers are chained through per-256-column "chunk done" mbarriers: the producer may load the K
// slices of layer l+1 that depend only on finished chunks of layer l, so the tensor pipe does not
// drain while the last chunk's epilogue runs.
// The activation tile of a CTA (2 x [128 x L] bf16) lives in a per-CTA global scratch that stays in
// L2; only x (128 B/pose) and y (192 B/pose) are compulsory HBM traffic.
#include <cstdlib>

#include "common.cuh"
#include "ptx.cuh"

namespace p3d {

// Persisting-L2 set-aside of the fused inference kernel: a per-device, process-wide resource (cudaLimitPersistingL2CacheSize).
// While it is set, that part of the L2 is withheld from normal traffic - also from every OTHER kernel of the process
// (measured: a training step ran 30 % slower after an inference pass had left 77 MB set aside).  So it is acquired by
// the fused forward and handed back by whoever needs the whole L2 next (the training step, p3d::l2persist_release).
static std::atomic<unsigned long long> g_l2_set_aside[64];
int l2persist_acquire(int dev, size_t bytes) {
  if (dev < 0 || dev >= 64) return P3D_OK;
  if (g_l2_set_aside[dev].load(std::memory_order_acquire) >= bytes) return P3D_OK;
  P3D_CUDA(cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, bytes));
  g_l2_set_aside[dev].store(bytes, std::memory_order_release);
  return P3D_OK;
}
bool l2persist_held(int dev, size_t bytes) {
  return dev >= 0 && dev < 64 && g_l2_set_aside[dev].load(std::memory_order_acquire) >= bytes;
}
int l2persist_release(int dev) {
  if (dev < 0 || dev >= 64 || g_l2_set_aside[dev].load(std::memory_order_acquire) == 0) return P3D_OK;
  cudaCtxResetPersistingL2Cache();
  P3D_CUDA(cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, 0));
  g_l2_set_aside[dev].store(0, std::memory_order_release);
  return P3D_OK;
}

namespace tc {

using namespace ptx;

constexpr int BM = 128;
constexpr int BN = 256;
constexpr int BK = 64;
constexpr int A_BYTES = BM * BK * 2;   // 16 KB
constexpr int OUT_BYTES = BM * 64 * 2; // 16 KB staging tile [128 rows x 64 cols] bf16
constexpr int NTHREADS = 256;
constexpr int TMEM_COLS = 512;
constexpr int MAX_SLABS = 64;          // 64-column slabs per layer: linear_size <= 4096

// CG = 1: one CTA per 128-pose tile, W' tile [256 x 64] per stage (48 KB/stage, 4 stages).
// CG = 2: a CTA PAIR (cta_group::2) per 256-pose tile; each CTA stages its own A [128 x 64] and HALF
//         of the W' tile [128 x 64] (32 KB/stage, 6 stages) - the pair's tensor cores share the halves,
//         which cuts the L2->SM operand traffic per FLOP by a third (the measured limiter at CG = 1).
template <int CG> struct Tile {
  static constexpr int STAGES = CG == 1 ? 4 : 6;
  static constexpr int BAR_BYTES = 1024;       // mbarriers + tmem slot
  static constexpr int B_ROWS = BN / CG;
  static constexpr int B_BYTES = B_ROWS * BK * 2;
  static constexpr int SMEM_BYTES = 1024 /*align slack*/ + STAGES * (A_BYTES + B_BYTES) + OUT_BYTES + 2 * BN * 4 + BAR_BYTES;
  static_assert(SMEM_BYTES <= 232448, "exceeds the 227 KB of shared memory per CTA");
};

struct Params {
  int L;           // linear_size (multiple of 256)
  int nlayers;     // 2*num_layers + 2
  int out_n;       // output width padded to a multiple of 16 (48)
  int out_valid;   // 48 or 42
  int residual;
  int ntiles;      // 128-row tiles
  long long B;
  long long act_half_rows;   // gridDim.x * 128 : row offset of buffer Q inside the scratch
  const float* bias;         // folded bias, indexed by packed weight row
  float* y;                  // [B][out_valid]
};

__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}

// descriptor for (1024B-aligned tile base + byte offset inside the first 128B row)
__device__ __forceinline__ uint64_t desc_at(uint32_t smem_addr) {
  constexpr uint32_t hi = (1024u >> 4) | (1u << 14) | (2u << 29);   // SBO | version=1 | SWIZZLE_128B
  const uint32_t lo = ((smem_addr >> 4) & 0x3FFFu) | (1u << 16);    // start address | LBO (unused) = 1
  return (static_cast<uint64_t>(hi) << 32) | lo;
}

template <int CG>
__global__ void __launch_bounds__(NTHREADS, 1)
mlp_forward_tc_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_act,
                      const __grid_constant__ CUtensorMap tm_w, const __grid_constant__ CUtensorMap tm_wout,
                      const Params p) {
  using T = Tile<CG>;
  constexpr int STAGES = T::STAGES;
  constexpr int B_BYTES = T::B_BYTES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = smem;
  uint8_t* sB = smem + STAGES * A_BYTES;
  uint8_t* sOut = sB + STAGES * B_BYTES;                       // 1024-aligned (all sizes are multiples of 1 KB)
  float* sBiasAll = reinterpret_cast<float*>(sOut + OUT_BYTES);   // [2][256], double buffered per chunk
  uint64_t* bars = reinterpret_cast<uint64_t*>(sBiasAll + 2 * BN);
  uint64_t* full = bars;                 // [STAGES]   (CG = 2: only the leader CTA's are used)
  uint64_t* empty = bars + STAGES;       // [STAGES]
  uint64_t* tfull = bars + 2 * STAGES;   // [2]
  uint64_t* tempty = tfull + 2;          // [2]        (CG = 2: only the leader CTA's are used)
  uint64_t* stg_full = tempty + 2;       // [1] staging tile written by the 4 epilogue warps
  uint64_t* stg_free = stg_full + 1;     // [1] staging tile read out by the TMA store
  uint64_t* slab_done = stg_free + 1;    // [MAX_SLABS] 64-column slab of the current layer is complete in global memory
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(slab_done + MAX_SLABS);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = (CG == 2) ? cluster_ctarank() : 0u;
  const bool leader = (rank == 0);
  const int group_id = blockIdx.x / CG, ngroups = gridDim.x / CG;
  const int ngtiles = (p.ntiles + CG - 1) / CG;     // tiles of 128*CG rows

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tm_x); tma_prefetch_desc(&tm_act); tma_prefetch_desc(&tm_w); tma_prefetch_desc(&tm_wout);
    // full: one arrival per producer warp (A = activations, B = weights) of the leader's accounting
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 2); mbar_init(&empty[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&tfull[a], 1); mbar_init(&tempty[a], 4 * CG); }
    mbar_init(stg_full, 4); mbar_init(stg_free, 1);
    for (int c = 0; c < MAX_SLABS; ++c) mbar_init(&slab_done[c], 1);
    fence_barrier_init();
  }
  if (warp == 2) {
    if (CG == 2) { tmem_alloc_2sm(tmem_slot, TMEM_COLS); tmem_relinquish_2sm(); }
    else { tmem_alloc(tmem_slot, TMEM_COLS); tmem_relinquish(); }
  }
  tc_fence_before();
  if (CG == 2) cluster_sync(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int L = p.L;
  const int nlayers = p.nlayers;
  const int nk_hidden = L / BK;
  const int nchunks_hidden = L / BN;

  if (warp == 0 || warp == 2) {
    // ------------------------------------------------------------ TMA producers (warp-uniform loops)
    // warp 0 fetches the A tiles (activations: gated by the slab barriers of the previous layer), warp 2 - idle after
    // the TMEM allocation - the W' tiles, which depend on nothing and may run ahead of the layer chain by a full ring.
    // Each arrives on full[stage] with its own byte count.
    const bool prodA = (warp == 0);
    int stage = 0; uint32_t phase = 0; uint32_t dep_layers = 0;
    for (int gt = group_id; gt < ngtiles; gt += ngroups) {
      const int tile = gt * CG + static_cast<int>(rank);
      for (int l = 0; l < nlayers; ++l) {
        const bool first = (l == 0), last = (l == nlayers - 1);
        const int nk = first ? 1 : nk_hidden;
        const int nchunks = last ? 1 : nchunks_hidden;
        const CUtensorMap* tmA = first ? &tm_x : &tm_act;
        const int a_row = first ? tile * BM
                                : static_cast<int>(((l & 1) ? 0 : p.act_half_rows) + static_cast<long long>(blockIdx.x) * BM);
        const int b_rows = last ? p.out_n / CG : T::B_ROWS;
        const uint32_t bytes = prodA ? A_BYTES : b_rows * BK * 2;
        for (int c = 0; c < nchunks; ++c) {
          const int b_row = (last ? 0 : l * L + c * BN) + static_cast<int>(rank) * b_rows;
          for (int ks = 0; ks < nk; ++ks) {
            // K slice ks reads columns [64ks, 64ks+64) = slab ks of the previous layer (this CTA's rows), written
            // by TMA stores (async proxy, completed before the arrive): no proxy fence needed
            if (prodA && !first && c == 0) mbar_wait(&slab_done[ks], dep_layers & 1, 100 + l);
            mbar_wait(&empty[stage], phase ^ 1, 1);
            if (elect_one()) {
              if (CG == 1) {
                mbar_arrive_expect_tx(&full[stage], bytes);
                if (prodA) tma_load_2d_hint(sA + stage * A_BYTES, tmA, &full[stage], ks * BK, a_row, first ? kEvictFirst : kEvictLast);
                else       tma_load_2d_hint(sB + stage * B_BYTES, last ? &tm_wout : &tm_w, &full[stage], ks * BK, b_row, kEvictLast);
              } else {
                // both CTAs' bytes are accounted on the leader's barrier
                if (leader) mbar_arrive_expect_tx(&full[stage], 2 * bytes);
                if (prodA) tma_load_2d_2sm_hint(sA + stage * A_BYTES, tmA, &full[stage], ks * BK, a_row, first ? kEvictFirst : kEvictLast);
                else       tma_load_2d_2sm_hint(sB + stage * B_BYTES, last ? &tm_wout : &tm_w, &full[stage], ks * BK, b_row, kEvictLast);
              }
            }
            __syncwarp();
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
        }
        if (!first) ++dep_layers;
      }
    }
  } else if (warp == 1 && leader) {
    // ------------------------------------------------------------ MMA issuer (warp-uniform loop, one elected lane issues)
    int stage = 0; uint32_t phase = 0; uint32_t q = 0;
    const uint32_t idesc_hidden = umma_idesc_bf16_f32(BM * CG, BN);
    const uint32_t idesc_out = umma_idesc_bf16_f32(BM * CG, p.out_n);
    const uint32_t a_base = smem_u32(sA), b_base = smem_u32(sB);
    for (int gt = group_id; gt < ngtiles; gt += ngroups) {
      for (int l = 0; l < nlayers; ++l) {
        const bool first = (l == 0), last = (l == nlayers - 1);
        const int nk = first ? 1 : nk_hidden;
        const int nchunks = last ? 1 : nchunks_hidden;
        const uint32_t idesc = last ? idesc_out : idesc_hidden;
        for (int c = 0; c < nchunks; ++c, ++q) {
          const uint32_t acc = q & 1, aphase = (q >> 1) & 1;
          mbar_wait(&tempty[acc], aphase ^ 1, 2);
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + acc * BN;
          for (int ks = 0; ks < nk; ++ks) {
            mbar_wait(&full[stage], phase, 3);
            tc_fence_after();
            if (elect_one()) {
              const uint64_t ad = desc_at(a_base + stage * A_BYTES);
              const uint64_t bd = desc_at(b_base + stage * B_BYTES);
#pragma unroll
              for (int k = 0; k < BK / 16; ++k) {    // +32 B per K=16 slice -> +2 in the (addr >> 4) field
                if (CG == 1) umma_bf16_ss(d_tmem, ad + 2 * k, bd + 2 * k, idesc, (ks | k) != 0 ? 1u : 0u);
                else         umma_bf16_ss_2sm(d_tmem, ad + 2 * k, bd + 2 * k, idesc, (ks | k) != 0 ? 1u : 0u);
              }
              if (CG == 1) {
                umma_commit(&empty[stage]);                   // frees the smem slot once these MMAs have read it
                if (ks == nk - 1) umma_commit(&tfull[acc]);   // accumulator complete -> epilogue
              } else {
                umma_commit_2sm(&empty[stage], 0x3);          // ... in both CTAs of the pair
                if (ks == nk - 1) umma_commit_2sm(&tfull[acc], 0x3);
              }
            }
            __syncwarp();
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 3) {
    // ------------------------------------------------------------ TMA store warp: staging tile -> this CTA's activation rows
    // One lane owns the bulk async-groups: it frees the staging tile as soon as the store has READ it and
    // publishes "slab done" (to the producer of the next layer) when the store has fully completed.
    if (lane == 0) {
      uint32_t n = 0;
      for (int gt = group_id; gt < ngtiles; gt += ngroups) {
        for (int l = 0; l < nlayers - 1; ++l) {
          const bool to_p = (l == 0) || ((l & 1) == 0);
          const bool add_res = p.residual && l >= 2 && ((l & 1) == 0);
          const int drow = static_cast<int>((to_p ? 0 : p.act_half_rows) + static_cast<long long>(blockIdx.x) * BM);
          const int nsl = L / 64;
          for (int sl = 0; sl < nsl; ++sl, ++n) {
            mbar_wait(stg_full, n & 1, 6);
            if (add_res) tma_reduce_add_2d_hint(&tm_act, sOut, sl * 64, drow, kEvictLast);   // P += relu(.)  (residual, added in the L2)
            else         tma_store_2d_hint(&tm_act, sOut, sl * 64, drow, kEvictLast);
            tma_store_commit();
            tma_store_wait_read<0>();
            mbar_arrive(stg_free);
            if (sl > 0) { tma_store_wait<1>(); mbar_arrive(&slab_done[sl - 1]); }
          }
          tma_store_wait<0>();
          mbar_arrive(&slab_done[nsl - 1]);
        }
      }
    }
  } else if (warp >= 4) {
    // ------------------------------------------------------------ epilogue (128 threads = this CTA's 128 rows)
    const int ew = warp - 4;                 // == warp % 4 : the TMEM lane quadrant this warp may read
    const int row = ew * 32 + lane;
    uint8_t* my_out = sOut + row * 128;
    uint32_t q = 0, nslab = 0;
    for (int gt = group_id; gt < ngtiles; gt += ngroups) {
      const int tile = gt * CG + static_cast<int>(rank);
      for (int l = 0; l < nlayers; ++l) {
        const bool last = (l == nlayers - 1);
        const int nchunks = last ? 1 : nchunks_hidden;
        for (int c = 0; c < nchunks; ++c, ++q) {
          const uint32_t acc = q & 1, aphase = (q >> 1) & 1;
          const int wrow0 = last ? (nlayers - 1) * L : l * L + c * BN;
          // bias of this chunk -> smem.  Double buffered: a fast warp may stage chunk q+1 while a slow one still
          // reads chunk q; the named barrier below keeps everybody within one chunk of each other.  The output layer
          // has only out_n packed rows (bias_fold ends 16 floats after them): its other rows stay unstaged, unread.
          float* sBias = sBiasAll + (q & 1) * BN;
          if (!last || row < p.out_n) sBias[row] = __ldg(p.bias + wrow0 + row);
          if (!last) sBias[row + 128] = __ldg(p.bias + wrow0 + row + 128);
          named_bar_sync(1, 128);
          mbar_wait(&tfull[acc], aphase, 4);
          tc_fence_after();
          const uint32_t taddr = tmem_base + (static_cast<uint32_t>(ew * 32) << 16) + acc * BN;
          if (!last) {
#pragma unroll 1
            for (int s = 0; s < BN / 64; ++s) {
              uint32_t v0[32], v1[32];
              tmem_ld_32x32b_x32(taddr + s * 64, v0);
              tmem_ld_32x32b_x32(taddr + s * 64 + 32, v1);
              tmem_ld_wait();
              if (s == BN / 64 - 1) {          // accumulator drained: hand it back to the MMA warp (of the leader CTA)
                tc_fence_before();
                __syncwarp();
                if (lane == 0) { if (CG == 1) mbar_arrive(&tempty[acc]); else mbar_arrive_cluster(&tempty[acc], 0); }
              }
              uint32_t o[32];
              const float* bs = sBias + s * 64;
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                o[j] = pack_bf16x2(fmaxf(__uint_as_float(v0[2 * j]) + bs[2 * j], 0.f),
                                   fmaxf(__uint_as_float(v0[2 * j + 1]) + bs[2 * j + 1], 0.f));
                o[16 + j] = pack_bf16x2(fmaxf(__uint_as_float(v1[2 * j]) + bs[32 + 2 * j], 0.f),
                                        fmaxf(__uint_as_float(v1[2 * j + 1]) + bs[32 + 2 * j + 1], 0.f));
              }
              mbar_wait(stg_free, (nslab & 1) ^ 1, 5);    // the store warp has read the previous slab out of the staging tile
              // row `row` = 128 B = 8 x 16 B chunks at chunk index (j ^ (row & 7)): the SWIZZLE_128B layout
#pragma unroll
              for (int j = 0; j < 8; ++j)
                *reinterpret_cast<uint4*>(my_out + ((j ^ (row & 7)) << 4)) = make_uint4(o[4 * j], o[4 * j + 1], o[4 * j + 2], o[4 * j + 3]);
              fence_proxy_async_smem();
              __syncwarp();
              if (lane == 0) mbar_arrive(stg_full);
              ++nslab;
            }
          } else {
            const long long grow = static_cast<long long>(tile) * BM + row;
            for (int g = 0; g < p.out_n / 16; ++g) {
              uint32_t v[16];
              tmem_ld_32x32b_x16(taddr + g * 16, v);
              tmem_ld_wait();
              if (grow < p.B) {
                float* yp = p.y + grow * p.out_valid + g * 16;
#pragma unroll
                for (int j = 0; j < 16; j += 2) {
                  const int col = g * 16 + j;
                  if (col + 1 < p.out_valid) {
                    float2 o2 = make_float2(__uint_as_float(v[j]) + sBias[col], __uint_as_float(v[j + 1]) + sBias[col + 1]);
                    __stcs(reinterpret_cast<float2*>(yp + j), o2);
                  } else if (col < p.out_valid) {
                    __stcs(yp + j, __uint_as_float(v[j]) + sBias[col]);
                  }
                }
              }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) { if (CG == 1) mbar_arrive(&tempty[acc]); else mbar_arrive_cluster(&tempty[acc], 0); }
          }
        }
      }
    }
  }

  tc_fence_before();
  if (CG == 2) cluster_sync(); else __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    if (CG == 2) tmem_dealloc_2sm(tmem_base, TMEM_COLS); else tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// ----------------------------------------------------------------------------- debug GEMM
// C[128,N] = A[128,K] W[N,K]^T with one CTA, one smem stage, fully serialised: exercises the TMA
// tensor maps, the UMMA smem/instruction descriptors and the TMEM load layout in isolation.
constexpr int B_BYTES = BN * BK * 2;   // 32 KB (debug kernel: full W tile in one CTA)
__global__ void __launch_bounds__(128, 1)
umma_gemm_debug_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_w,
                       float* C, int N, int K) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = smem;
  uint8_t* sB = smem + A_BYTES;
  uint64_t* bar_full = reinterpret_cast<uint64_t*>(sB + B_BYTES);
  uint64_t* bar_mma = bar_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar_mma + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) { mbar_init(bar_full, 1); mbar_init(bar_mma, 1); fence_barrier_init(); }
  if (warp == 0) { tmem_alloc(tmem_slot, 256); tmem_relinquish(); }
  tc_fence_before(); __syncthreads(); tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (threadIdx.x == 0) {
    const uint32_t idesc = umma_idesc_bf16_f32(128, N);
    for (int ks = 0; ks < K / BK; ++ks) {
      mbar_arrive_expect_tx(bar_full, A_BYTES + N * BK * 2);
      tma_load_2d(sA, &tm_a, bar_full, ks * BK, 0);
      tma_load_2d(sB, &tm_w, bar_full, ks * BK, 0);
      mbar_wait(bar_full, ks & 1, 10);
      tc_fence_after();
      for (int k = 0; k < BK / 16; ++k)
        umma_bf16_ss(tmem_base, umma_desc_k_sw128(smem_u32(sA) + k * 32), umma_desc_k_sw128(smem_u32(sB) + k * 32),
                     idesc, (ks | k) != 0 ? 1u : 0u);
      umma_commit(bar_mma);
      mbar_wait(bar_mma, ks & 1, 11);
    }
  }
  tc_fence_before(); __syncthreads(); tc_fence_after();
  const int row = warp * 32 + lane;
  for (int g = 0; g < N / 16; ++g) {
    uint32_t v[16];
    tmem_ld_32x32b_x16(tmem_base + (static_cast<uint32_t>(warp * 32) << 16) + g * 16, v);
    tmem_ld_wait();
    for (int j = 0; j < 16; ++j) C[row * N + g * 16 + j] = __uint_as_float(v[j]);
  }
  tc_fence_before(); __syncthreads();
  if (warp == 0) { tc_fence_after(); tmem_dealloc(tmem_base, 256); }
}

// ----------------------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess)
      return nullptr;
    fn = reinterpret_cast<EncodeTiledFn>(ptr);
  }
  return fn;
}

// bf16 row-major [rows][pitch_elems] tensor, box = [box_rows][64 cols], 128B swizzle
static int make_tmap(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t pitch_elems,
                     uint32_t box_rows) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) { set_error("cuTensorMapEncodeTiled entry point not available"); return P3D_ERR_CUDA; }
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstride[1] = {pitch_elems * 2};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(BK), box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstride, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed with CUresult %d", (int)r); return P3D_ERR_CUDA; }
  return P3D_OK;
}

template <int CG>
static int launch_forward(p3d_model* m, const __nv_bfloat16* xb, float* y, int64_t B, cudaStream_t st) {
  using T = Tile<CG>;
  const int L = m->L;
  const int ntiles = static_cast<int>((B + BM - 1) / BM);
  const int ngtiles = (ntiles + CG - 1) / CG;
  const int max_groups = m->num_sms / CG;
  const int grid = CG * (ngtiles < max_groups ? ngtiles : max_groups);
  const int nlayers = static_cast<int>(m->layers.size());
  const int out_n = (m->out_size + 15) / 16 * 16;
  CUtensorMap tm_x, tm_act, tm_w, tm_wout;
  P3D_TRY(make_tmap(&tm_x, xb, static_cast<uint64_t>(B), 64, 64, BM));
  P3D_TRY(make_tmap(&tm_act, m->act_scratch, 2ull * grid * BM, L, L, BM));
  P3D_TRY(make_tmap(&tm_w, m->wt_bf16, static_cast<uint64_t>(nlayers - 1) * L, m->kpad, m->kpad, T::B_ROWS));
  P3D_TRY(make_tmap(&tm_wout, m->wt_bf16 + static_cast<size_t>(nlayers - 1) * L * m->kpad, out_n, m->kpad, m->kpad, out_n / CG));
  Params p;
  p.L = L; p.nlayers = nlayers; p.out_n = out_n; p.out_valid = m->out_size; p.residual = m->cfg.residual;
  p.ntiles = ntiles; p.B = B; p.act_half_rows = static_cast<long long>(grid) * BM;
  p.bias = m->bias_fold; p.y = y;
  static PerDeviceOnce attr_set;
  if (attr_set.needed()) {
    P3D_CUDA(cudaFuncSetAttribute(mlp_forward_tc_kernel<CG>, cudaFuncAttributeMaxDynamicSharedMemorySize, T::SMEM_BYTES));
    attr_set.mark();
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(NTHREADS); cfg.dynamicSmemBytes = T::SMEM_BYTES; cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CG; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  // The per-CTA activation scratch (2 x 128 x L bf16 per CTA, 77.6 MB for 148 CTAs at L = 1024) is written and re-read
  // five times per tile and never needed after the launch, yet without help the streaming x / y lines push dirty scratch
  // lines out of the L2 (the evict_last hints on the TMA operations do not prevent it): ncu measured 4.86 GB of DRAM
  // traffic per 2^20-pose launch against 0.34 GB of compulsory x / y bytes.  An access-policy window on the scratch with
  // a persisting-L2 set-aside keeps those lines resident: 2.42 GB, and 156.6 -> 159.7 M poses/s on the same box
  // (round 2, profiles/r2_l2persist.md).  P3D_L2_PERSIST=0 switches it off.
  // Under graph capture nothing host-side may change: the window goes into the graph only while the set-aside is held.
  // A replay after a training step has handed the set-aside back is slower (the scratch competes for the L2), not wrong.
  static const bool l2_persist = [] { const char* e = getenv("P3D_L2_PERSIST"); return !(e && e[0] == '0'); }();
  const bool cap = capturing(st);
  if (l2_persist) {
    int dev = 0, max_persist = 0, max_window = 0;
    P3D_CUDA(cudaGetDevice(&dev));
    P3D_CUDA(cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, dev));
    P3D_CUDA(cudaDeviceGetAttribute(&max_window, cudaDevAttrMaxAccessPolicyWindowSize, dev));
    const size_t scratch = sizeof(__nv_bfloat16) * 2ull * grid * BM * L;
    // only when the whole scratch fits the set-aside (width 1024: 77.6 MB); a partial window over the 310 MB of the
    // width-4096 model bought nothing and cost the weights their L2 share (0.73 -> 0.65 of peak)
    if (scratch <= static_cast<size_t>(max_persist) && scratch <= static_cast<size_t>(max_window) &&
        (!cap || l2persist_held(dev, scratch))) {
      if (!cap) P3D_TRY(l2persist_acquire(dev, scratch));
      attr[1].id = cudaLaunchAttributeAccessPolicyWindow;
      attr[1].val.accessPolicyWindow.base_ptr = m->act_scratch;
      attr[1].val.accessPolicyWindow.num_bytes = scratch;
      attr[1].val.accessPolicyWindow.hitRatio = 1.0f;
      attr[1].val.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
      attr[1].val.accessPolicyWindow.missProp = cudaAccessPropertyNormal;
      cfg.numAttrs = 2;
    }
  }
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  if (prof::enabled() && !cap) prof::begin(st, &e0, &e1);     // timing events are read on the host: eager launches only
  P3D_CUDA(cudaLaunchKernelEx(&cfg, mlp_forward_tc_kernel<CG>, tm_x, tm_act, tm_w, tm_wout, p));
  P3D_LAUNCH_CHECK();
  if (e0) prof::end(st, e0, e1);
  return P3D_OK;
}

int forward_bf16(p3d_model* m, const __nv_bfloat16* xb, float* y, int64_t B, cudaStream_t st) {
  const int L = m->L;
  P3D_REQUIRE(L % BN == 0 && L / 64 <= MAX_SLABS, "bf16 tensor-core path needs linear_size %% 256 == 0 and <= 4096 (got %d)", L);
  // per-CTA activation scratch, sized for a full grid once
  if (m->act_grid < m->num_sms) {
    P3D_TRY(refuse_in_capture(st, "forward: allocating the fused kernel's activation scratch"));
    if (m->act_scratch) cudaFree(m->act_scratch);
    P3D_CUDA(cudaMalloc(&m->act_scratch, sizeof(__nv_bfloat16) * 2ull * m->num_sms * BM * L));
    m->act_grid = m->num_sms;
  }
  static int cg = -1;
  if (cg < 0) {
    const char* e = getenv("P3D_TC_CG");       // 1 = single-CTA tiles, 2 = CTA pairs (default)
    cg = (e && e[0] == '1') ? 1 : 2;
  }
  return cg == 1 ? launch_forward<1>(m, xb, y, B, st) : launch_forward<2>(m, xb, y, B, st);
}

int debug_umma_gemm(const void* A, const void* W, float* C, int N, int K, cudaStream_t st) {
  P3D_REQUIRE(N % 16 == 0 && N >= 16 && N <= 256 && K % 64 == 0 && K >= 64, "debug gemm: bad N=%d K=%d", N, K);
  CUtensorMap tm_a, tm_w;
  P3D_TRY(make_tmap(&tm_a, A, 128, K, K, 128));
  P3D_TRY(make_tmap(&tm_w, W, N, K, K, N));
  const int smem = 1024 + A_BYTES + B_BYTES + 64;
  P3D_CUDA(cudaFuncSetAttribute(umma_gemm_debug_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  umma_gemm_debug_kernel<<<1, 128, smem, st>>>(tm_a, tm_w, C, N, K);
  P3D_LAUNCH_CHECK();
  return P3D_OK;
}

}  // namespace tc
}  // namespace p3d
