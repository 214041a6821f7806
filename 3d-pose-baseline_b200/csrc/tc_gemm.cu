// Generic tcgen05 GEMM for the training step (src/linear_model.py:129-145: the MatMuls of the forward
// graph, of tf.gradients and of the weight gradients), bf16 operands, fp32 accumulation in TMEM.
//
//   C[M,N] (+)= alpha * sum_k A(m,k) B(n,k)  (+ bias[n]) (+ res[m,n])
//
// Each operand is described by how it lies in memory:
//   K-major  : [rows = M or N][K contiguous]   (activations for Z = H W;  dZ and W for dH = dZ W^T)
//   MN-major : [K rows][M or N contiguous]     (W for Z = H W;  H and dZ for dW = H^T dZ)
// so the three GEMMs of a layer read H, dZ and W in their NATURAL row-major layouts - no transposed
// copies exist anywhere.  MN-major tiles are fetched as 64-column TMA boxes (128B swizzle) and consumed
// through the MN-major canonical UMMA layout ((8,n),(8,k)):((1,LBO),(8,SBO)) [16-byte units].
//
// One CTA per 128 x BN output tile (BN = 32/64/128/256 chosen per problem so the grid covers the SMs),
// optional split-K over gridDim.z (fp32 atomics into a zeroed C - the weight-gradient GEMMs have only
// (L/128)*(L/BN) tiles but K = batch).  Warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer,
// warps 2-9 = epilogue (TMEM -> registers -> alpha/bias/residual -> global).  Out-of-range rows/cols
// and the K tail are zero-filled by TMA, so M, N, K need no padding (K=32 input layer, N=48 output).
//
// Fused training epilogues (OUT = 3 / 4): the BatchNorm / ReLU / dropout arithmetic of a hidden layer, forward and
// backward, runs on the accumulator while it sits in TMEM; the per-column batch statistics they need are CTA-local
// for one M tile and otherwise meet at a grid barrier - with the data-parallel SyncBN exchange over NVLink peer
// memory in the same place (see FusedTrain in common.cuh).
//
// Variants measured on B200 and removed again (numbers in DESIGN.md 3.5): CTA pairs (cta_group::2), two CTAs per SM,
// A-tile multicast across a cluster, BatchNorm-backward sums in the dh epilogue of one-tile CTAs, TMA-store epilogue,
// and the general (descriptor-rebuilding) MMA issue loop that the lean one below replaced.
#include <cstring>

#include "common.cuh"
#include "ptx.cuh"
#include "train_common.cuh"

namespace p3d {
namespace tcg {

using namespace ptx;

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int MAX_STAGES = 16;
constexpr int A_BYTES = BM * BK * 2;        // 16 KB
constexpr int BOX_BYTES = 64 * BK * 2;      // one [64 rows x 64 cols] bf16 box = 8 KB
constexpr int NTHREADS = 320;             // warp 0 TMA, warp 1 MMA, warps 2-9 epilogue (two per TMEM lane quadrant)
constexpr int EPI_THREADS = 256;
// Epilogue warps of the fused training kernels (a multiple of 4: warps per TMEM lane quadrant).  Measured on B200 at 4096
// poses: 12 warps (448 threads, 128 registers, small spills) 408.5 us per step against 408.4 us with 8 - the fused
// epilogues are bound by their instruction COUNT (~67 K warp instructions per 128 x 256 tile, half of them Philox), not
// by the number of warps that share it.
#ifndef P3D_FUSED_EPI_WARPS
#define P3D_FUSED_EPI_WARPS 8
#endif
constexpr int FUSED_EPI_THREADS = 32 * P3D_FUSED_EPI_WARPS;
constexpr int FUSED_NTHREADS = 64 + FUSED_EPI_THREADS;
constexpr int RING_BYTES = 4 * (A_BYTES + 256 * BK * 2);   // 192 KB: 4 stages at BN=256, 6 at 128, 8 at 64
constexpr int BAR_BYTES = 512;               // full[16] | empty[16] | accf | tmem slot | grid-sync scratch
// align slack | operand ring | barriers | bias[256] | column sums [4 quadrants][2][256] | per-column finals [2][256] f32 | totals [2][256] f64
// | per-column constants of the fused epilogues [4][256] f32 (gamma, beta, mean, rstd)
constexpr int TAIL_BYTES = 1024 + 8192 + 2048 + 4096 + 4096;
constexpr int SMEM_BYTES = 1024 + RING_BYTES + BAR_BYTES + TAIL_BYTES;
// the narrower the tile, the deeper the ring: small problems are latency bound on the L2 -> SM round trip

struct Params {
  int M, N, K;
  int bn;            // 32 / 64 / 128 / 256
  int k_per_split;   // multiple of BK
  int a_mn, b_mn;
  float* C; int ldc;
  const float* bias;        // [N] or null (added by split 0 only)
  const float* res; int ldres;   // [M,N] or null (added by split 0 only)
  const float* alpha_dev;   // optional device scalar
  float alpha;
  int atomic;               // accumulate into C with fp32 atomics (split-K)
  double* colsum;           // optional [2][N]: column sums of the stored values and of their squares
  // bf16 output (inference layers): out = bf16(relu?(alpha*acc + bias)); with res_b: out = bf16(out + res_b)
  __nv_bfloat16* out_b; int ldob;
  const __nv_bfloat16* res_b; int ldrb;
  int relu;
  int stages;               // ring depth: what fits into 192 KB at this tile size, 16 at most
  int a_bytes;              // bytes of A actually fetched per stage (K-major A of a short problem: only round_up(M, 8) rows)
  int b_independent;        // B does not depend on preceding kernels of the stream (weights): prefetch it before the PDL wait
  unsigned long long* dbg;  // optional [ctas][32] globaltimer stamps (diagnostics)
  FusedTrain ft;            // OUT = 3 / 4 only
  long long wait_limit_ns;  // > 0: a wait for peers / the grid longer than this traps (diagnostics; 0 = wait like NCCL does)
  int seg_a, seg_b;         // SEG: column of the lo segment of A / B (see GemmArgs::seg_a)
  int ob_lo;                // OUT = 5: column of the lo halves in out_b
};
__device__ __forceinline__ unsigned long long gtime() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
#define P3D_STAMP(i) do { if (p.dbg && lane == 0) p.dbg[(static_cast<size_t>(blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x) * 32 + (i)] = gtime(); } while (0)

__device__ __forceinline__ void grid_dependency_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void grid_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// K-major operand, 128B swizzle: rows 128 B apart, 8-row groups 1024 B apart
__device__ __forceinline__ uint64_t desc_k(uint32_t smem_addr) {
  constexpr uint32_t hi = (1024u >> 4) | (1u << 14) | (2u << 29);
  const uint32_t lo = ((smem_addr >> 4) & 0x3FFFu) | (1u << 16);
  return (static_cast<uint64_t>(hi) << 32) | lo;
}
// MN-major operand, 128B swizzle: 64 MN-elements (128 B) contiguous, k rows 128 B apart, 8-k groups SBO = 1024 B
// apart, the next 64 MN-elements LBO = one box (8 KB) further
__device__ __forceinline__ uint64_t desc_mn(uint32_t smem_addr) {
  constexpr uint32_t hi = (1024u >> 4) | (1u << 14) | (2u << 29);
  const uint32_t lo = ((smem_addr >> 4) & 0x3FFFu) | (static_cast<uint32_t>(BOX_BYTES >> 4) << 16);
  return (static_cast<uint64_t>(hi) << 32) | lo;
}

// shared-space accessors: the tile pointer is derived from the aligned dynamic-smem base by integer arithmetic, which
// makes the compiler fall back to GENERIC ld/st (long-scoreboard latency) - say the address space explicitly
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
  return v;
}

// ------------------------------------------------------------------ grid / peer synchronisation of the fused epilogues
__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu(unsigned* p, unsigned v) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned ld_acquire_gpu(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_volatile_u4(uint4* p, uint4 v) {
  asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ uint4 ld_volatile_u4(const uint4* p) {
  uint4 v;
  asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ double ld_cg_f64(const double* p) {
  double v;
  asm volatile("ld.global.cg.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
  return v;
}

// Column sums of the whole (global) batch for the columns n0 .. n0 + bn of this CTA (totals_arrive + totals_wait: whatever
// does not need the sums runs between the two, in the shadow of the barrier), called by the 256 epilogue threads
// after pass 1 has left this CTA's per-quadrant partial sums in scol ([4][2][256] floats).  Result: tot[j], tot[256 + j]
// (doubles, shared memory) for column n0 + j.
//   one M tile, one GPU : the four quadrant partials are the batch.
//   otherwise           : partials -> gsum (fp64 atomics) -> arrival counter; the CTA that arrives last owns the complete
//                         sums of this GPU.  One GPU: everybody spins on the counter reaching the grid size.  Data parallel: it
//                         stores the vector into slot [seq % NSLOTS][rank] of EVERY rank's exchange buffer as self-validating
//                         16-byte words {lo, tag, hi, tag} (tag = sequence number; 8-byte halves arrive whole over NVLink), and
//                         every thread of every CTA of every rank polls exactly the words it consumes and adds the `world`
//                         values in rank order - bit-identical sums everywhere, one NVLink write latency per exchange (the
//                         first version published the vector with a system-scope release fence and a flag per peer: two more
//                         hops, 17 us per exchange on 8 GPUs).  Slot reuse is safe: nobody can be more than one exchange ahead
//                         of the slowest rank (it needs that rank's words).  No timeout by default: like an NCCL collective
//                         this waits for its peers (Params::wait_limit_ns is the diagnostics switch).
template <int EPI_THREADS>
__device__ __forceinline__ void totals_arrive(const Params& p, int n0, int et, const float* scol, double* tot, uint32_t* sflag,
                                              unsigned long long seq) {
  const FusedTrain& ft = p.ft;
  const int N = p.N;
  if (ft.gsum == nullptr) {
    for (int j = et; j < p.bn; j += EPI_THREADS) {
      tot[j] = static_cast<double>((scol[j] + scol[512 + j]) + (scol[1024 + j] + scol[1536 + j]));
      tot[256 + j] = static_cast<double>((scol[256 + j] + scol[768 + j]) + (scol[1280 + j] + scol[1792 + j]));
    }
    return;
  }
  for (int j = et; j < p.bn; j += EPI_THREADS) {
    if (n0 + j < N) {
      atomicAdd(ft.gsum + n0 + j, static_cast<double>((scol[j] + scol[512 + j]) + (scol[1024 + j] + scol[1536 + j])));
      atomicAdd(ft.gsum + N + n0 + j, static_cast<double>((scol[256 + j] + scol[768 + j]) + (scol[1280 + j] + scol[1792 + j])));
    }
  }
  // arrive: the block barrier orders the CTA's atomics before thread 0, whose fence (cumulative) publishes them before the
  // counter moves - one membar per CTA instead of 256 (ncu: ERRBAR among the top stall sites of the first version)
  named_bar_sync(1, EPI_THREADS);
  const unsigned nctas = gridDim.x * gridDim.y;
  if (et == 0) {
    __threadfence();
    const unsigned prev = atomicAdd(ft.gcount, 1u);
    *sflag = (prev == nctas - 1u) ? 1u : 0u;
  }
  if (ft.world == 1) return;                            // one GPU: everybody spins on the counter itself (totals_wait)
  named_bar_sync(1, EPI_THREADS);
  if (*sflag != 0u) {                                   // the last CTA of this GPU: its sums are complete
    const p2p::Peers* peers = static_cast<const p2p::Peers*>(ft.peers);
    const int slot = static_cast<int>(seq % p2p::NSLOTS);
    const uint32_t tag = static_cast<uint32_t>(seq);
    if (et == 0) __threadfence();
    named_bar_sync(1, EPI_THREADS);
    // every value to every rank (this one included) as self-validating 16-byte stores {lo, tag, hi, tag}; one more scalar
    // rides along at index 2 N (the step's loss sum on the first backward exchange)
    const int nv = 2 * N + (ft.xsum ? 1 : 0);
    for (int i = et; i < nv; i += EPI_THREADS) {
      const double d = ld_cg_f64(i < 2 * N ? ft.gsum + i : ft.xsum);
      const unsigned long long u = static_cast<unsigned long long>(__double_as_longlong(d));
      const uint4 w = make_uint4(static_cast<uint32_t>(u), tag, static_cast<uint32_t>(u >> 32), tag);
      for (int r = 0; r < ft.world; ++r) st_volatile_u4(&peers->p[r]->ll[slot][ft.rank][i], w);
    }
    if (et == 0) peers->p[ft.rank]->seq = seq;
  }
}

template <int EPI_THREADS>
__device__ __forceinline__ void totals_wait(const Params& p, int n0, int et, double* tot, unsigned long long seq) {
  const FusedTrain& ft = p.ft;
  const int N = p.N;
  if (ft.gsum == nullptr) { named_bar_sync(1, EPI_THREADS); return; }
  const unsigned long long t0 = p.wait_limit_ns > 0 ? gtime() : 0ull;
  if (ft.world == 1) {
    // one GPU: wait for the other CTAs (the counter reaches the grid size), then read the sums
    if (et == 0) {
      const unsigned nctas = gridDim.x * gridDim.y;
      while (ld_acquire_gpu(ft.gcount) < nctas) {
        if (p.wait_limit_ns > 0 && gtime() - t0 > static_cast<unsigned long long>(p.wait_limit_ns)) { printf("p3d: grid barrier timed out\n"); __trap(); }
      }
    }
    named_bar_sync(1, EPI_THREADS);
    for (int j = et; j < p.bn; j += EPI_THREADS) {
      double s1 = 0.0, s2 = 0.0;
      if (n0 + j < N) { s1 = ld_cg_f64(ft.gsum + n0 + j); s2 = ld_cg_f64(ft.gsum + N + n0 + j); }
      tot[j] = s1; tot[256 + j] = s2;
    }
  } else {
    // data parallel: every thread polls the words it consumes (column n0 + j of every rank) until they carry this
    // exchange's tag, and adds them in rank order - bit-identical sums on every rank
    const p2p::Layout* me = static_cast<const p2p::Peers*>(ft.peers)->p[ft.rank];
    const int slot = static_cast<int>(seq % p2p::NSLOTS);
    const uint32_t tag = static_cast<uint32_t>(seq);
    auto valid = [&](const uint4& w) { return w.y == tag && w.w == tag; };
    auto value = [&](const uint4& w) { return __longlong_as_double(static_cast<long long>((static_cast<unsigned long long>(w.z) << 32) | w.x)); };
    auto fetch = [&](int r, int i) {
      uint4 w = ld_volatile_u4(&me->ll[slot][r][i]);
      while (!valid(w)) {
        if (p.wait_limit_ns > 0 && gtime() - t0 > static_cast<unsigned long long>(p.wait_limit_ns)) {
          printf("p3d: SyncBN exchange timed out (rank %d waits for rank %d, seq %llu)\n", ft.rank, r, seq); __trap();
        }
        w = ld_volatile_u4(&me->ll[slot][r][i]);
      }
      return value(w);
    };
    for (int j = et; j < p.bn; j += EPI_THREADS) {
      double s1 = 0.0, s2 = 0.0;
      if (n0 + j < N) {
        // four ranks at a time: their eight words are requested together and the whole batch is re-polled until every
        // word carries the tag - one L2 round trip per poll (the first version polled word by word: eight to sixteen
        // round trips in a row, 15 us per exchange on 8 GPUs)
        for (int r0 = 0; r0 < ft.world; r0 += 4) {
          uint4 a[4], b[4];
          for (;;) {
            bool ok = true;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const int r = (r0 + q < ft.world) ? r0 + q : r0;
              a[q] = ld_volatile_u4(&me->ll[slot][r][n0 + j]);
              b[q] = ld_volatile_u4(&me->ll[slot][r][N + n0 + j]);
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) ok = ok && valid(a[q]) && valid(b[q]);
            if (ok) break;
            if (p.wait_limit_ns > 0 && gtime() - t0 > static_cast<unsigned long long>(p.wait_limit_ns)) {
              printf("p3d: SyncBN exchange timed out (rank %d waits for ranks %d.., seq %llu)\n", ft.rank, r0, seq); __trap();
            }
          }
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            if (r0 + q < ft.world) { s1 += value(a[q]); s2 += value(b[q]); }
          }
        }
      }
      tot[j] = s1; tot[256 + j] = s2;
    }
    if (ft.xsum && et == 0 && blockIdx.x == 0 && blockIdx.y == 0) {
      double sx = 0.0;
      for (int r = 0; r < ft.world; ++r) sx += fetch(r, 2 * N);
      *ft.xsum = sx;
    }
  }
  named_bar_sync(1, EPI_THREADS);
}

// OUT: 0 = fp32 store, 1 = fp32 reduction (split-K / accumulate), 2 = bf16 (relu, residual in bf16), 3 / 4 = fused
// training epilogues (forward / backward), 5 = split pair (relu, fp32 residual; the fp32 value to C when given, its
// bf16 hi / lo halves to out_b).  RES: a residual operand is added.  CS: column sums of the result and its
// square are accumulated (BatchNorm statistics of a forward layer on the unfused path).  SEG: segment schedule of the
// split-precision (bf16x3) GEMMs, inference and training - the K loop runs three passes, reading the (A, B) segments
// (hi, hi), (lo, hi), (hi, lo) into one accumulator; either operand K-major or MN-major, K split or not.  F16: fp16
// operands (P3D_MODE_FP16 inference: the fp32 store and the 16-bit activation store, OUT 0 / 2), where OUT = 2 stores
// and reads fp16 activations.
template <int OUT, bool RES, int CS, bool SEG = false, bool F16 = false>
__global__ void __launch_bounds__((OUT == 3 || OUT == 4) ? FUSED_NTHREADS : NTHREADS, 1)
tc_gemm_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b, const Params p) {
  static_assert(CS == 0 || OUT < 2, "column sums are taken of the fp32 stores only");
  static_assert(!F16 || ((OUT == 0 || OUT == 2) && !SEG && CS == 0), "fp16 operands: the inference epilogues only");
  using O16 = Op16<F16>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int STAGES = p.stages;
  const int B_BYTES = p.bn * BK * 2;
  const int A_SLOT = p.a_bytes;                  // slots are as large as what is fetched (multiple of 1024 B)
  uint8_t* sA = smem;
  uint8_t* sB = smem + STAGES * A_SLOT;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + RING_BYTES);
  uint64_t* empty = full + MAX_STAGES;
  uint64_t* accf = empty + MAX_STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accf + 1);
  uint32_t* sflag = tmem_slot + 1;
  float* sbias = reinterpret_cast<float*>(smem + RING_BYTES + BAR_BYTES);
  float* scol = sbias + 256;
  float* sfin = scol + 2048;                     // [2][256] per-column finals of the fused epilogues
  double* stot = reinterpret_cast<double*>(sfin + 512);   // [2][256] column totals of the global batch
  float* scst = reinterpret_cast<float*>(stot + 512);     // [4][256] gamma | beta | mean | rstd of this CTA's columns

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0) P3D_STAMP(0);
  const int n0 = blockIdx.x * p.bn, m0 = blockIdx.y * BM;
  const int kbeg = blockIdx.z * p.k_per_split;
  const int kend = (kbeg + p.k_per_split < p.K) ? kbeg + p.k_per_split : p.K;
  const int nkp = (kend - kbeg + BK - 1) / BK;   // k-blocks of one pass
  const int nk = SEG ? 3 * nkp : nkp;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tm_a); tma_prefetch_desc(&tm_b);
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(accf, 1);
    fence_barrier_init();
  }
  constexpr uint32_t TMEM_MULT = (OUT == 4) ? 2u : 1u;      // the fused backward epilogue keeps xhat in a second half
  if (warp == 1) { tmem_alloc(tmem_slot, TMEM_MULT * static_cast<uint32_t>(p.bn)); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  grid_launch_dependents();     // the next kernel of a programmatic-dependent chain may start its prologue now
  if (warp == 0) P3D_STAMP(1);

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    // Every TMA operation of a stage belongs to its own lane and all of them leave in ONE instruction: issuing them
    // one after the other from a single thread costs ~0.12 us each, which is what bounded short-M GEMMs (16 serial
    // k-blocks x 2 operations = 4.3 us of a 7.6 us kernel).  Lanes [0, na) fetch A boxes, lanes [na, na + nb) B boxes.
    // Everything that does not change from k-block to k-block - which box this lane fetches, through which map, into
    // which offset of a slot, its fixed coordinate - is settled before the loop; a k-block is barrier wait, expect_tx,
    // one TMA instruction per box-owning lane.
    const uint32_t bytes = p.a_bytes + B_BYTES;
    const int na = p.a_mn ? 2 : 1, nb = p.b_mn ? p.bn / 64 : 1;
    const bool is_a = lane < na, is_b = lane >= na && lane < na + nb;
    const CUtensorMap* my_map = is_a ? &tm_a : &tm_b;
    const bool my_mn = is_a ? (p.a_mn != 0) : (p.b_mn != 0);
    const int my_box = is_a ? lane : lane - na;
    const int my_row0 = is_a ? m0 : n0;
    const uint32_t dst0 = smem_u32(is_a ? sA : sB) + static_cast<uint32_t>(my_box) * BOX_BYTES;
    const uint32_t slot = is_a ? static_cast<uint32_t>(A_SLOT) : static_cast<uint32_t>(B_BYTES);
    const int fix = my_mn ? my_row0 + 64 * my_box : my_row0;             // MN-major: the row coordinate of this lane's box
    const uint32_t full_s = smem_u32(full);
    auto load = [&](int stg, int k0) {
      tma_load_2d_s(dst0 + static_cast<uint32_t>(stg) * slot, my_map, full_s + static_cast<uint32_t>(stg) * 8u, my_mn ? fix : k0, my_mn ? k0 : fix);
    };
    // K coordinate of k-block kb for this lane's operand.
    auto kcoord = [&](int kb) { return kbeg + kb * BK; };
    // SEG: pass 1 reads A's lo segment, pass 2 B's.  The lo segment lies `seg` columns along the operand's CONTIGUOUS
    // dimension: the K coordinate of a K-major operand, the MN coordinate (fix) of an MN-major one.  Each pass walks
    // this split's own K range [kbeg, kend).
    auto load_seg = [&](int stg, int kb) {
      const int pass = kb / nkp;
      const int lo = is_a ? (pass == 1 ? p.seg_a : 0) : (pass == 2 ? p.seg_b : 0);
      const int k0 = kbeg + (kb - pass * nkp) * BK;
      tma_load_2d_s(dst0 + static_cast<uint32_t>(stg) * slot, my_map, full_s + static_cast<uint32_t>(stg) * 8u,
                    my_mn ? fix + lo : k0 + lo, my_mn ? k0 : fix);
    };
    auto fetch = [&](int stg, int kb) {
      if constexpr (SEG) load_seg(stg, kb);
      else load(stg, kcoord(kb));
    };
    // Programmatic dependent launch: when B is marked independent of the preceding kernels (weights), its tiles for
    // the first ring pass are requested BEFORE griddepcontrol.wait, i.e. while the previous layer is still running.
    const int npre = p.b_independent ? (nk < STAGES ? nk : STAGES) : 0;
    for (int kb = 0; kb < npre; ++kb) {            // ring slots are free on the first pass
      if (lane == 0) mbar_arrive_expect_tx(&full[kb], bytes);
      __syncwarp();
      if (is_b) fetch(kb, kb);
    }
    __syncwarp();
    grid_dependency_wait();
    int stage = 0; uint32_t phase = 0;
    for (int kb = 0; kb < nk; ++kb) {
      mbar_wait(&empty[stage], phase ^ 1, 1);
      if (kb >= npre && lane == 0) mbar_arrive_expect_tx(&full[stage], bytes);
      __syncwarp();
      if (is_a || (is_b && kb >= npre)) fetch(stage, kb);
      if (p.dbg) { if (kb == 3) P3D_STAMP(8); if (kb == 7) P3D_STAMP(9); if (kb == 11) P3D_STAMP(10); }
      if (++stage == STAGES) { stage = 0; phase ^= 1; }
    }
    P3D_STAMP(2);
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer
    // A descriptor's start-address field is (address >> 4) in its low 14 bits and every operand address is a multiple
    // of 16 below 256 KB, so the field advances LINEARLY: one descriptor per operand is built before the loop, a
    // k-block adds stage * (slot >> 4), a K = 16 slice adds (step >> 4) - no carry can leave the field.  (Rebuilding
    // eight descriptors per k-block from byte addresses cost ~110 SASS instructions between the barrier and the first
    // tcgen05.mma, against 4 x 56 cycles of tensor work at N <= 64; measured: 16.9 -> 14.7 us for a 4096 x 1024 x 1024
    // GEMM, 48 -> 40 us for the six-layer batch-64 inference chain.)
    const uint32_t idesc = umma_idesc_16_f32<F16>(BM, p.bn) | (p.a_mn ? (1u << 15) : 0u) | (p.b_mn ? (1u << 16) : 0u);
    const uint32_t a_base = smem_u32(sA), b_base = smem_u32(sB);
    const uint32_t a_step = p.a_mn ? 2048u : 32u, b_step = p.b_mn ? 2048u : 32u;   // bytes per K=16 slice
    const uint64_t a0 = p.a_mn ? desc_mn(a_base) : desc_k(a_base), b0 = p.b_mn ? desc_mn(b_base) : desc_k(b_base);
    const uint32_t a_slot16 = static_cast<uint32_t>(A_SLOT) >> 4, b_slot16 = static_cast<uint32_t>(B_BYTES) >> 4;
    const uint32_t a_k16 = a_step >> 4, b_k16 = b_step >> 4;
    int stage = 0; uint32_t phase = 0;
    for (int kb = 0; kb < nk; ++kb) {
      mbar_wait(&full[stage], phase, 2);
      if (p.dbg) { if (kb == 0) P3D_STAMP(3); if (kb == 4) P3D_STAMP(11); if (kb == 8) P3D_STAMP(12); if (kb == 12) P3D_STAMP(13); }
      tc_fence_after();
      if (elect_one()) {
        const uint64_t ad = a0 + static_cast<uint32_t>(stage) * a_slot16, bd = b0 + static_cast<uint32_t>(stage) * b_slot16;
#pragma unroll
        for (int k = 0; k < BK / 16; ++k)
          umma_bf16_ss(tmem_base, ad + static_cast<uint32_t>(k) * a_k16, bd + static_cast<uint32_t>(k) * b_k16, idesc, (kb | k) != 0 ? 1u : 0u);
        umma_commit(&empty[stage]);
        if (kb == nk - 1) umma_commit(accf);
      }
      __syncwarp();
      if (++stage == STAGES) { stage = 0; phase ^= 1; }
    }
    P3D_STAMP(4);
  } else {
    // ------------------------------------------------------------ epilogue: warp w owns TMEM lanes 32*(w%4)..+31
    // tcgen05.ld hands every lane one ROW (32 consecutive columns).  Storing that directly makes each instruction
    // touch 32 different lines, 16 bytes each.  Instead the 32 x 32 chunk is transposed through a padded smem tile
    // (the operand ring is free once the accumulator is complete) so that a lane owns 4 COLUMNS x 8 rows: every
    // global access (C, residual, bf16 output, fp32 reductions) is then 4 full 128-byte lines per instruction, bias
    // is a per-lane constant and the column sums need 2 shuffle steps instead of a 31-shuffle butterfly.
    if constexpr (OUT == 3 || OUT == 4) {
      // ------------------------------------------------------------ fused training epilogues
      // Two passes over the tile with the column statistics of the (global) batch in between (totals_arrive / _wait):
      // GEMM + statistics + finalize + activation kernels -> 1 launch, both directions.  Eight warps cannot hide the
      // latency of an elementwise pass the way a standalone kernel with 64 warps per SM does (first version: 27 of the
      // 34 us of a 4096-pose forward layer were epilogue), so the work is arranged around what they CAN overlap:
      //   phase 0, under the mainloop (these warps would only wait for the accumulator): everything that does not need
      //            it.  Forward: the dropout keep-bits (Philox or the injected mask) - kept as one bit per element in
      //            registers, the mask bytes stored for the backward pass; what is not finished when the accumulator
      //            arrives is done later in the shadow of the grid barrier.  Backward: z and the keep-mask are read,
      //            xhat = (z - mean) rstd goes into the spare half of the TMEM allocation, relu' * keep into bits.
      //   pass 1:  accumulator -> (alpha, bias, residual) -> column partial sums; the values every lane has produced are
      //            written back over the accumulator chunk they came from with tcgen05.st - lane l's 32 registers go to
      //            TMEM lane l, so TMEM serves as 128 bytes per lane and chunk of private scratch, already in the
      //            4-columns-x-8-rows arrangement the global accesses want (no second trip through shared memory).
      //   shadow:  between arriving at the grid barrier and the sums being known (3-4 us): the stores of z (forward).
      //   pass 2:  reads the scratch; per-column constants come from shared memory (staged once; an __ldg per chunk
      //            exposed an L2 round trip each time); no global loads besides the residual operand.
      constexpr int EPI_THREADS = FUSED_EPI_THREADS;           // (shadows the plain epilogues' constant)
      constexpr int PARTS = P3D_FUSED_EPI_WARPS / 4;           // warps per TMEM lane quadrant
      const int ew = warp & 3, part = (warp - 2) >> 2;
      // the tile's 32-column chunks go round robin over the warps of a quadrant: chunk k of this warp = columns
      // 32 (part + PARTS k) ..
      const int cbeg = 32 * part;
      constexpr int CSTEP = 32 * PARTS;
      int nch = 0;                                             // chunks this warp owns (<= 4)
      for (int c0 = cbeg; c0 < p.bn && n0 + c0 < p.N; c0 += CSTEP) ++nch;
      const train::StepScalars* sc = static_cast<const train::StepScalars*>(p.ft.sc);
      const int et = (warp - 2) * 32 + lane;
      // data parallel: the sequence number of this exchange - read before anybody of this grid can have advanced it
      unsigned long long seq = 0;
      if (p.ft.world > 1) seq = static_cast<const p2p::Peers*>(p.ft.peers)->p[p.ft.rank]->seq + 1;
      grid_dependency_wait();
      const float alpha = p.alpha * (p.alpha_dev ? __ldg(p.alpha_dev) : 1.f);
      const bool has_bn = p.ft.has_bn != 0, dropout = p.ft.dropout != 0;
      for (int j = et; j < p.bn; j += EPI_THREADS) {
        const int n = n0 + j;
        const bool okc = n < p.N;
        sbias[j] = (p.bias && okc) ? __ldg(p.bias + n) : 0.f;
        scst[j] = (has_bn && okc) ? __ldg(p.ft.gamma + n) : 1.f;
        scst[256 + j] = (has_bn && okc) ? __ldg(p.ft.beta + n) : 0.f;
        if (OUT == 4) {
          scst[512 + j] = (has_bn && okc) ? __ldg(p.ft.mean + n) : 0.f;
          scst[768 + j] = (has_bn && okc) ? __ldg(p.ft.rstd + n) : 1.f;
        }
      }
      named_bar_sync(1, EPI_THREADS);
      constexpr int TP = 36;
      const uint32_t tile_s = smem_u32(smem) + (warp - 2) * 32 * TP * 4;
      const uint32_t sbias_s = smem_u32(sbias);
      const int rg = lane >> 3, cq = (lane & 7) * 4;
      const int mrow0 = m0 + ew * 32 + rg;
      const float keep = sc->keep, inv_keep = sc->inv_keep;
      const bool writer = (blockIdx.y == 0);                   // of the CTAs that share a column: the one that stores per-column results
      const double invB = static_cast<double>(p.ft.invB);
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(ew * 32) << 16);
      // chunk k of this warp: bit (4 i + j) = row mrow0 + 4 i, column cq + j.  Four scalars picked by selects: an array
      // indexed by the chunk counter would live in local memory.
      uint32_t g0 = 0xffffffffu, g1 = 0xffffffffu, g2 = 0xffffffffu, g3 = 0xffffffffu;
      auto set_gate = [&](int k, uint32_t b) { if (k == 0) g0 = b; else if (k == 1) g1 = b; else if (k == 2) g2 = b; else g3 = b; };
      auto get_gate = [&](int k) { return k == 0 ? g0 : (k == 1 ? g1 : (k == 2 ? g2 : g3)); };
      auto cst4 = [&](int which, int c) { return *reinterpret_cast<const float4*>(scst + which * 256 + c); };

      // ---------------------------------------------------------------- phase 0 (under the mainloop), one chunk at a time
      auto pre_chunk = [&](int k) {
        const int c0 = cbeg + CSTEP * k;
        const int n = n0 + c0 + cq;
        if constexpr (OUT == 3) {
          uint32_t bits = 0;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int m = mrow0 + 4 * i;
            if (m >= p.M) continue;
            const size_t off = static_cast<size_t>(m) * p.N + n;
            uchar4 kb;
            if (p.ft.mask_in) {
              kb = *reinterpret_cast<const uchar4*>(p.ft.mask_in + off);
            } else {
              const uint4 w4 = train::dropout_words(sc->seed, sc->step, static_cast<uint32_t>(p.ft.layer),
                                                    static_cast<uint32_t>(p.ft.row0 + m), static_cast<uint32_t>(n >> 2));
              kb = make_uchar4(train::keep_bit(w4.x, keep), train::keep_bit(w4.y, keep), train::keep_bit(w4.z, keep), train::keep_bit(w4.w, keep));
            }
            *reinterpret_cast<uchar4*>(p.ft.mask + off) = kb;
            bits |= ((kb.x ? 1u : 0u) | (kb.y ? 2u : 0u) | (kb.z ? 4u : 0u) | (kb.w ? 8u : 0u)) << (4 * i);
          }
          set_gate(k, bits);
        } else {
          const float4 g4 = cst4(0, c0 + cq), b4 = cst4(1, c0 + cq), m4 = cst4(2, c0 + cq), r4 = cst4(3, c0 + cq);
          const float mu[4] = {m4.x, m4.y, m4.z, m4.w}, rs[4] = {r4.x, r4.y, r4.z, r4.w};
          const float ga[4] = {g4.x, g4.y, g4.z, g4.w}, be[4] = {b4.x, b4.y, b4.z, b4.w};
          float4 z4[8];
          uchar4 mk[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int m = mrow0 + 4 * i;
            const size_t off = static_cast<size_t>(m < p.M ? m : 0) * p.N + n;
            z4[i] = __ldg(reinterpret_cast<const float4*>(p.ft.z + off));
            mk[i] = dropout ? *reinterpret_cast<const uchar4*>(p.ft.mask + off) : make_uchar4(1, 1, 1, 1);
          }
          uint32_t xh[32], bits = 0;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const bool live = mrow0 + 4 * i < p.M;
            const float zz[4] = {z4[i].x, z4[i].y, z4[i].z, z4[i].w};
            const unsigned char kk[4] = {mk[i].x, mk[i].y, mk[i].z, mk[i].w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float x = has_bn ? (zz[j] - mu[j]) * rs[j] : 0.f;
              const float act = has_bn ? ga[j] * x + be[j] : zz[j];
              xh[4 * i + j] = __float_as_uint(x);
              if (live && act > 0.f && kk[j]) bits |= 1u << (4 * i + j);
            }
          }
          set_gate(k, bits);
          tmem_st_32x32b_x32(taddr + p.bn + c0, xh);          // the spare half of the allocation: columns bn .. 2 bn
        }
      };
      int kdone = 0;
      if constexpr (OUT == 3) {
        if (!dropout) kdone = nch;
        while (kdone < nch && !mbar_try_wait(accf, 0)) pre_chunk(kdone++);     // the rest follows in the barrier's shadow
      } else {
        while (kdone < nch) pre_chunk(kdone++);                                // pass 1 needs all of it
        tmem_st_wait();
      }
      if (warp == 2) P3D_STAMP(14);                            // phase 0 done (forward: as far as the mainloop allowed)
      mbar_wait(accf, 0, 3);
      if (warp == 2) P3D_STAMP(5);
      tc_fence_after();
      // accumulator chunk (already in registers, row per lane) -> this lane's 4 columns x 8 rows (rows mrow0 + 4 i), as
      // alpha * acc + bias.  The registers are free again after the shared-memory stores: the caller re-issues the TMEM
      // load of the next chunk into them before it works on this one.
      auto transpose = [&](int c0, uint32_t (&v)[32], float (&o)[8][4], bool more) {
        tmem_ld_wait();
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 32; j += 4) sts128(tile_s + (lane * TP + j) * 4, v[j], v[j + 1], v[j + 2], v[j + 3]);
        __syncwarp();
        if (more) tmem_ld_32x32b_x32(taddr + c0 + CSTEP, v);
        const float4 b4 = lds128(sbias_s + (c0 + cq) * 4);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 t = lds128(tile_s + ((i * 4 + rg) * TP + cq) * 4);
          o[i][0] = alpha * t.x + b4.x; o[i][1] = alpha * t.y + b4.y; o[i][2] = alpha * t.z + b4.z; o[i][3] = alpha * t.w + b4.w;
        }
      };
      auto stash = [&](uint32_t col, const float (&o)[8][4]) {          // this lane's 32 values -> its private TMEM scratch
        uint32_t v[32];
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) v[4 * i + j] = __float_as_uint(o[i][j]);
        tmem_st_32x32b_x32(taddr + col, v);
      };
      auto unstash = [&](uint32_t col, float (&o)[8][4]) {
        uint32_t v[32];
        tmem_ld_32x32b_x32(taddr + col, v);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) o[i][j] = __uint_as_float(v[4 * i + j]);
      };
      auto publish = [&](int c0, float (&s1)[4], float (&s2)[4]) {     // fold the 4 row groups, quadrant partial -> smem
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          s1[j] += __shfl_xor_sync(0xffffffffu, s1[j], 8);  s2[j] += __shfl_xor_sync(0xffffffffu, s2[j], 8);
          s1[j] += __shfl_xor_sync(0xffffffffu, s1[j], 16); s2[j] += __shfl_xor_sync(0xffffffffu, s2[j], 16);
        }
        if (rg == 0) {
          float* q1 = scol + ew * 512 + c0 + cq;
          *reinterpret_cast<float4*>(q1) = make_float4(s1[0], s1[1], s1[2], s1[3]);
          *reinterpret_cast<float4*>(q1 + 256) = make_float4(s2[0], s2[1], s2[2], s2[3]);
        }
      };
      uint32_t acc[32];
      if (nch > 0) tmem_ld_32x32b_x32(taddr + cbeg, acc);
      if constexpr (OUT == 3) {
        // ---- forward pass 1: z = alpha acc + bias, column sums, z -> scratch
        const bool z_in_shadow = has_bn && p.ft.gsum != nullptr;       // with a grid barrier to wait for, z is stored behind it
        for (int k = 0; k < nch; ++k) {
          const int c0 = cbeg + CSTEP * k;
          float o[8][4], s1[4] = {0.f, 0.f, 0.f, 0.f}, s2[4] = {0.f, 0.f, 0.f, 0.f};
          transpose(c0, acc, o, k + 1 < nch);
          if (!z_in_shadow) {
            const int n = n0 + c0 + cq;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const int m = mrow0 + 4 * i;
              if (m < p.M) *reinterpret_cast<float4*>(p.C + static_cast<size_t>(m) * p.N + n) = make_float4(o[i][0], o[i][1], o[i][2], o[i][3]);
            }
          }
          if (has_bn) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const bool live = mrow0 + 4 * i < p.M;
#pragma unroll
              for (int j = 0; j < 4; ++j) { const float q = live ? o[i][j] : 0.f; s1[j] += q; s2[j] += q * q; }
            }
            publish(c0, s1, s2);
          }
          stash(c0, o);
        }
        tmem_st_wait();
        if (warp == 2) P3D_STAMP(15);                          // pass 1 done
        if (has_bn) {
          named_bar_sync(1, EPI_THREADS);
          totals_arrive<EPI_THREADS>(p, n0, et, scol, stot, sflag, seq);
        }
        // ---- in the shadow of the barrier: what is left of the dropout bits, and z -> global (the backward pass reads it)
        while (kdone < nch) pre_chunk(kdone++);
        for (int k = 0; z_in_shadow && k < nch; ++k) {
          const int c0 = cbeg + CSTEP * k, n = n0 + c0 + cq;
          float o[8][4];
          unstash(c0, o);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int m = mrow0 + 4 * i;
            if (m < p.M) *reinterpret_cast<float4*>(p.C + static_cast<size_t>(m) * p.N + n) = make_float4(o[i][0], o[i][1], o[i][2], o[i][3]);
          }
        }
        if (has_bn) {
          totals_wait<EPI_THREADS>(p, n0, et, stot, seq);
          if (warp == 2) P3D_STAMP(16);                        // column totals of the global batch known
          // mean / biased variance over the global batch in double, as train.cu's bn_finalize_kernel does it;
          // moving averages with momentum .99 (one writer per column)
          for (int j = et; j < p.bn; j += EPI_THREADS) {
            const int n = n0 + j;
            const double mu = stot[j] * invB;
            double var = stot[256 + j] * invB - mu * mu;
            if (var < 0) var = 0;
            const float muf = static_cast<float>(mu), rsf = static_cast<float>(1.0 / sqrt(var + static_cast<double>(kBnEps)));
            sfin[j] = muf; sfin[256 + j] = rsf;
            if (writer && n < p.N) {
              p.ft.mean[n] = muf; p.ft.rstd[n] = rsf;
              p.ft.mov_mean[n] = p.ft.mov_mean[n] * kBnMomentum + muf * (1.f - kBnMomentum);
              p.ft.mov_var[n] = p.ft.mov_var[n] * kBnMomentum + static_cast<float>(var) * (1.f - kBnMomentum);
            }
          }
          named_bar_sync(1, EPI_THREADS);
        }
        // ---- forward pass 2: BN, ReLU, dropout, + residual -> h (fp32, where a later layer adds it), hb (bf16 operand)
        for (int k = 0; k < nch; ++k) {
          const int c0 = cbeg + CSTEP * k, n = n0 + c0 + cq;
          float4 hr[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int m = mrow0 + 4 * i;
            hr[i] = p.ft.hres ? __ldg(reinterpret_cast<const float4*>(p.ft.hres + static_cast<size_t>(m < p.M ? m : 0) * p.N + n)) : make_float4(0.f, 0.f, 0.f, 0.f);
          }
          float o[8][4];
          unstash(c0, o);
          if (has_bn) {
            const float4 g4 = cst4(0, c0 + cq), b4 = cst4(1, c0 + cq);
            const float4 m4 = *reinterpret_cast<const float4*>(sfin + c0 + cq), r4 = *reinterpret_cast<const float4*>(sfin + 256 + c0 + cq);
            const float ga[4] = {g4.x, g4.y, g4.z, g4.w}, be[4] = {b4.x, b4.y, b4.z, b4.w};
            const float mu[4] = {m4.x, m4.y, m4.z, m4.w}, rs[4] = {r4.x, r4.y, r4.z, r4.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
              for (int j = 0; j < 4; ++j) o[i][j] = ga[j] * ((o[i][j] - mu[j]) * rs[j]) + be[j];      // same operation order as the unfused kernels
          }
          const uint32_t bits = get_gate(k);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int m = mrow0 + 4 * i;
            if (m >= p.M) continue;
            const size_t off = static_cast<size_t>(m) * p.N + n;
            float r[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              r[j] = fmaxf(o[i][j], 0.f);
              if (dropout) r[j] = ((bits >> (4 * i + j)) & 1u) ? r[j] * inv_keep : 0.f;
            }
            r[0] += hr[i].x; r[1] += hr[i].y; r[2] += hr[i].z; r[3] += hr[i].w;
            if (p.ft.h) *reinterpret_cast<float4*>(p.ft.h + off) = make_float4(r[0], r[1], r[2], r[3]);
            __nv_bfloat162 lo = __floats2bfloat162_rn(r[0], r[1]), hi = __floats2bfloat162_rn(r[2], r[3]);
            uint2 pk; pk.x = *reinterpret_cast<uint32_t*>(&lo); pk.y = *reinterpret_cast<uint32_t*>(&hi);
            *reinterpret_cast<uint2*>(static_cast<__nv_bfloat16*>(p.ft.hb) + off) = pk;
          }
        }
      } else {
        // ---- backward pass 1: dh = alpha acc (+ res) (-> dh_out); da = dh * keep/relu' gate; column sums of da, da * xhat
        for (int k = 0; k < nch; ++k) {
          const int c0 = cbeg + CSTEP * k, n = n0 + c0 + cq;
          float4 r4[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int m = mrow0 + 4 * i;
            r4[i] = p.res ? __ldg(reinterpret_cast<const float4*>(p.res + static_cast<size_t>(m < p.M ? m : 0) * p.N + n)) : make_float4(0.f, 0.f, 0.f, 0.f);
          }
          float o[8][4], xh[8][4], s1[4] = {0.f, 0.f, 0.f, 0.f}, s2[4] = {0.f, 0.f, 0.f, 0.f};
          transpose(c0, acc, o, k + 1 < nch);
          unstash(p.bn + c0, xh);
          const uint32_t bits = get_gate(k);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int m = mrow0 + 4 * i;
            o[i][0] += r4[i].x; o[i][1] += r4[i].y; o[i][2] += r4[i].z; o[i][3] += r4[i].w;
            if (p.ft.dh_out && m < p.M)
              *reinterpret_cast<float4*>(p.ft.dh_out + static_cast<size_t>(m) * p.N + n) = make_float4(o[i][0], o[i][1], o[i][2], o[i][3]);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              float gr = o[i][j];
              if (dropout) gr *= inv_keep;
              const float da = ((bits >> (4 * i + j)) & 1u) ? gr : 0.f;
              o[i][j] = da;
              s1[j] += da; s2[j] += da * xh[i][j];
            }
          }
          publish(c0, s1, s2);
          stash(c0, o);
        }
        tmem_st_wait();
        if (warp == 2) P3D_STAMP(15);
        named_bar_sync(1, EPI_THREADS);
        totals_arrive<EPI_THREADS>(p, n0, et, scol, stot, sflag, seq);
        totals_wait<EPI_THREADS>(p, n0, et, stot, seq);
        if (warp == 2) P3D_STAMP(16);
        // sum da (= dbeta, or the bias gradient) and sum da * xhat (= dgamma) over the global batch; every rank holds
        // them in full, so they enter the flat gradient pre-divided by the world size
        for (int j = et; j < p.bn; j += EPI_THREADS) {
          const int n = n0 + j;
          const float P = static_cast<float>(stot[j]), Q = static_cast<float>(stot[256 + j]);
          sfin[j] = P; sfin[256 + j] = Q;
          if (writer && n < p.N) {
            if (has_bn) { p.ft.gbeta[n] = P * p.ft.pg_scale; p.ft.ggamma[n] = Q * p.ft.pg_scale; }
            else p.ft.gbias[n] = P * p.ft.pg_scale;
          }
        }
        named_bar_sync(1, EPI_THREADS);
        // ---- backward pass 2: dz = gamma rstd (da - mean(da) - xhat mean(da xhat)) -> bf16 operand of the next GEMMs
        const float invBf = p.ft.invB;
        for (int k = 0; k < nch; ++k) {
          const int c0 = cbeg + CSTEP * k, n = n0 + c0 + cq;
          float o[8][4], xh[8][4];
          unstash(c0, o);
          float gr[4] = {1.f, 1.f, 1.f, 1.f}, P[4] = {0.f, 0.f, 0.f, 0.f}, Q[4] = {0.f, 0.f, 0.f, 0.f};
          if (has_bn) {
            unstash(p.bn + c0, xh);
            const float4 g4 = cst4(0, c0 + cq), r4 = cst4(3, c0 + cq);
            const float4 P4 = *reinterpret_cast<const float4*>(sfin + c0 + cq), Q4 = *reinterpret_cast<const float4*>(sfin + 256 + c0 + cq);
            gr[0] = g4.x * r4.x; gr[1] = g4.y * r4.y; gr[2] = g4.z * r4.z; gr[3] = g4.w * r4.w;
            P[0] = P4.x * invBf; P[1] = P4.y * invBf; P[2] = P4.z * invBf; P[3] = P4.w * invBf;
            Q[0] = Q4.x * invBf; Q[1] = Q4.y * invBf; Q[2] = Q4.z * invBf; Q[3] = Q4.w * invBf;
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int m = mrow0 + 4 * i;
            if (m >= p.M) continue;
            float d[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) d[j] = has_bn ? gr[j] * (o[i][j] - P[j] - xh[i][j] * Q[j]) : o[i][j];
            __nv_bfloat162 lo = __floats2bfloat162_rn(d[0], d[1]), hi = __floats2bfloat162_rn(d[2], d[3]);
            uint2 pk; pk.x = *reinterpret_cast<uint32_t*>(&lo); pk.y = *reinterpret_cast<uint32_t*>(&hi);
            *reinterpret_cast<uint2*>(static_cast<__nv_bfloat16*>(p.ft.dzb) + static_cast<size_t>(m) * p.N + n) = pk;
          }
        }
      }
    } else {
    // The epilogue variant is a template parameter and the bias sits in smem before the accumulator is complete:
    // the first version (runtime flags, generic smem accesses, bias re-loaded per chunk) spent 11 of the 20 us of a
    // 4096 x 1024 x 1024 GEMM here, one warp per scheduler crawling through ~2800 SASS instructions of branches.
    const int ew = warp & 3;                     // TMEM lane quadrant of this warp
    const int half = (warp - 2) >> 2;            // which half of the tile's columns
    const int hw = p.bn >= 64 ? p.bn / 2 : 32;                       // columns per half (BN = 32: the second half idles)
    const int cbeg = half * hw, cend = (cbeg + hw < p.bn) ? cbeg + hw : p.bn;
    const bool first_split = (blockIdx.z == 0);
    grid_dependency_wait();       // residual / alpha / C written by earlier kernels
    const float alpha = p.alpha * (p.alpha_dev ? __ldg(p.alpha_dev) : 1.f);
    const int et = (warp - 2) * 32 + lane;       // 0..255
    for (int j = et; j < p.bn; j += EPI_THREADS) {
      sbias[j] = (first_split && p.bias && n0 + j < p.N) ? __ldg(p.bias + n0 + j) : 0.f;
    }
    named_bar_sync(1, EPI_THREADS);
    const uint32_t sbias_s = smem_u32(sbias);
    {
    constexpr int TP = 36;                                   // tile pitch in floats (144 B): conflict-free both ways
    const uint32_t tile_s = smem_u32(smem) + (warp - 2) * 32 * TP * 4;
    const int rg = lane >> 3, cq = (lane & 7) * 4;           // row group (rows rg, rg+4, ...), first of this lane's 4 columns
    const int mrow0 = m0 + ew * 32 + rg;                     // this lane's rows: mrow0 + 4 i
    const bool use_res = RES && (OUT == 2 || first_split);
    // fast path: the whole tile is inside N and every pointer/pitch allows vector accesses
    bool fast = (n0 + p.bn <= p.N);
    if (OUT == 2) fast = fast && ((p.ldob & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.out_b) & 7) == 0) &&
                         (!RES || (((p.ldrb & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.res_b) & 7) == 0)));
    else if (OUT == 5) fast = fast && ((p.ldob & 3) == 0) && ((p.ob_lo & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.out_b) & 7) == 0) &&
                              (!p.C || (((p.ldc & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.C) & 15) == 0))) &&
                              (!RES || (((p.ldres & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.res) & 15) == 0)));
    else fast = fast && ((p.ldc & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.C) & 15) == 0) &&
                        (!RES || (((p.ldres & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.res) & 15) == 0)));
    mbar_wait(accf, 0, 3);
    if (warp == 2) P3D_STAMP(5);
    tc_fence_after();
    const uint32_t taddr = tmem_base + (static_cast<uint32_t>(ew * 32) << 16);
    uint32_t v[32];
    if (cbeg < cend && n0 + cbeg < p.N) tmem_ld_32x32b_x32(taddr + cbeg, v);
    for (int c0 = cbeg; c0 < cend; c0 += 32) {
      if (n0 + c0 >= p.N) break;     // warp-uniform
      const bool more = (c0 + 32 < cend) && (n0 + c0 + 32 < p.N);
      tmem_ld_wait();
      __syncwarp();                  // the previous chunk's readers are done with the tile
#pragma unroll
      for (int j = 0; j < 32; j += 4) sts128(tile_s + (lane * TP + j) * 4, v[j], v[j + 1], v[j + 2], v[j + 3]);
      __syncwarp();
      if (more) tmem_ld_32x32b_x32(taddr + c0 + 32, v);      // in flight while this chunk is processed
      const int n = n0 + c0 + cq;                            // this lane's columns n .. n+3
      const float4 b4 = lds128(sbias_s + (c0 + cq) * 4);
      float cs1[4] = {0.f, 0.f, 0.f, 0.f}, cs2[4] = {0.f, 0.f, 0.f, 0.f};
      if (fast) {
        float4 t4[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) t4[i] = lds128(tile_s + ((i * 4 + rg) * TP + cq) * 4);
        float4 r4[8];
        uint2 rb[8];
        if (use_res) {
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int m = mrow0 + 4 * i;
            r4[i] = make_float4(0.f, 0.f, 0.f, 0.f); rb[i] = make_uint2(0u, 0u);
            if (m < p.M) {
              if (OUT == 2) rb[i] = *reinterpret_cast<const uint2*>(p.res_b + static_cast<size_t>(m) * p.ldrb + n);
              // in place (res == C): a plain load, not the read-only path, for memory this kernel writes
              else if (OUT == 5) r4[i] = *reinterpret_cast<const float4*>(p.res + static_cast<size_t>(m) * p.ldres + n);
              else r4[i] = __ldg(reinterpret_cast<const float4*>(p.res + static_cast<size_t>(m) * p.ldres + n));
            }
          }
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int m = mrow0 + 4 * i;
          const bool live = m < p.M;
          float o[4] = {alpha * t4[i].x + b4.x, alpha * t4[i].y + b4.y, alpha * t4[i].z + b4.z, alpha * t4[i].w + b4.w};
          if (OUT == 2) {
            // bf16 activations of the layered inference path: same rounding points as the fused persistent kernel
            // (relu(.) rounded to bf16 / fp16, then the residual added and rounded again)
            typename O16::T ob[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) ob[j] = O16::from(p.relu ? fmaxf(o[j], 0.f) : o[j]);
            if (use_res) {
              typename O16::T rv[4];
              memcpy(rv, &rb[i], 8);
#pragma unroll
              for (int j = 0; j < 4; ++j) ob[j] = O16::from(O16::to(ob[j]) + O16::to(rv[j]));
            }
            uint2 q; memcpy(&q, ob, 8);
            if (live) *reinterpret_cast<uint2*>(p.out_b + static_cast<size_t>(m) * p.ldob + n) = q;
          } else if (OUT == 5) {
            // split pair: r = relu(.) (+ fp32 residual) stays fp32; hi = bf16(r), lo = bf16(r - hi) (r - hi is exact)
            __nv_bfloat16 hb[4], lb[4];
            float r[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) r[j] = p.relu ? fmaxf(o[j], 0.f) : o[j];
            if (use_res) { r[0] += r4[i].x; r[1] += r4[i].y; r[2] += r4[i].z; r[3] += r4[i].w; }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              hb[j] = __float2bfloat16_rn(r[j]);
              lb[j] = __float2bfloat16_rn(r[j] - __bfloat162float(hb[j]));
            }
            if (live) {
              if (p.C) *reinterpret_cast<float4*>(p.C + static_cast<size_t>(m) * p.ldc + n) = make_float4(r[0], r[1], r[2], r[3]);
              uint2 qh, ql; memcpy(&qh, hb, 8); memcpy(&ql, lb, 8);
              __nv_bfloat16* ob = p.out_b + static_cast<size_t>(m) * p.ldob + n;
              *reinterpret_cast<uint2*>(ob) = qh;
              *reinterpret_cast<uint2*>(ob + p.ob_lo) = ql;
            }
          } else {
            if (use_res) { o[0] += r4[i].x; o[1] += r4[i].y; o[2] += r4[i].z; o[3] += r4[i].w; }
            if (CS == 1) {            // sums of the stored values: residual included
#pragma unroll
              for (int j = 0; j < 4; ++j) { const float q = live ? o[j] : 0.f; cs1[j] += q; cs2[j] += q * q; }
            }
            float* crow = p.C + static_cast<size_t>(m) * p.ldc + n;
            if (live) {
              if (OUT == 1) asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(crow), "f"(o[0]), "f"(o[1]), "f"(o[2]), "f"(o[3]) : "memory");
              else *reinterpret_cast<float4*>(crow) = make_float4(o[0], o[1], o[2], o[3]);
            }
          }
        }
      } else {
        // ragged / unaligned tile (N = 48 or 42 output layer, odd pitches): element by element; rows not unrolled.
        // The column loop IS unrolled: with a runtime column index, bias / tv and - shared with the fast path above -
        // cs1 / cs2 were demoted to local memory (ncu: STL/LDL of the column sums after every row of the hot loop).
        const float bias[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll 1
        for (int i = 0; i < 8; ++i) {
          const int m = mrow0 + 4 * i;
          if (m >= p.M) continue;
          const float4 t = lds128(tile_s + ((i * 4 + rg) * TP + cq) * 4);
          const float tv[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            if (n + j >= p.N) continue;
            float o = alpha * tv[j] + bias[j];
            if (OUT == 2) {
              using T16 = typename O16::T;
              T16 ob = O16::from(p.relu ? fmaxf(o, 0.f) : o);
              if (use_res) ob = O16::from(O16::to(ob) + O16::to(reinterpret_cast<const T16*>(p.res_b)[static_cast<size_t>(m) * p.ldrb + n + j]));
              reinterpret_cast<T16*>(p.out_b)[static_cast<size_t>(m) * p.ldob + n + j] = ob;
            } else if (OUT == 5) {
              float r = p.relu ? fmaxf(o, 0.f) : o;
              if (use_res) r += p.res[static_cast<size_t>(m) * p.ldres + n + j];
              if (p.C) p.C[static_cast<size_t>(m) * p.ldc + n + j] = r;
              const __nv_bfloat16 hb = __float2bfloat16_rn(r);
              p.out_b[static_cast<size_t>(m) * p.ldob + n + j] = hb;
              p.out_b[static_cast<size_t>(m) * p.ldob + p.ob_lo + n + j] = __float2bfloat16_rn(r - __bfloat162float(hb));
            } else {
              if (use_res) o += __ldg(p.res + static_cast<size_t>(m) * p.ldres + n + j);
              if (CS == 1) { cs1[j] += o; cs2[j] += o * o; }
              float* c = p.C + static_cast<size_t>(m) * p.ldc + n + j;
              if (OUT == 1) atomicAdd(c, o); else *c = o;
            }
          }
        }
      }
      if (CS) {
        // this lane holds 8 of the warp's 32 rows for its 4 columns: fold the 4 row groups, then lanes 0..7 publish
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          cs1[j] += __shfl_xor_sync(0xffffffffu, cs1[j], 8);  cs2[j] += __shfl_xor_sync(0xffffffffu, cs2[j], 8);
          cs1[j] += __shfl_xor_sync(0xffffffffu, cs1[j], 16); cs2[j] += __shfl_xor_sync(0xffffffffu, cs2[j], 16);
        }
        if (rg == 0) {            // this quadrant's partial sums -> smem (plain stores: one writer per slot)
          float* q1 = scol + ew * 512 + c0 + cq;
          *reinterpret_cast<float4*>(q1) = make_float4(cs1[0], cs1[1], cs1[2], cs1[3]);
          *reinterpret_cast<float4*>(q1 + 256) = make_float4(cs2[0], cs2[1], cs2[2], cs2[3]);
        }
      }
    }
    }
    if (CS) {
      named_bar_sync(1, EPI_THREADS);
      for (int j = et; j < p.bn; j += EPI_THREADS) {        // one global fp64 atomic per column per CTA
        if (n0 + j < p.N) {
          const float s1 = (scol[j] + scol[512 + j]) + (scol[1024 + j] + scol[1536 + j]);
          const float s2 = (scol[256 + j] + scol[768 + j]) + (scol[1280 + j] + scol[1792 + j]);
          atomicAdd(p.colsum + n0 + j, static_cast<double>(s1));
          atomicAdd(p.colsum + p.N + n0 + j, static_cast<double>(s2));
        }
      }
    }
    }   // plain epilogues
  }
  if (warp == 2) P3D_STAMP(6);
  tc_fence_before();
  __syncthreads();
  if (warp == 0) P3D_STAMP(7);
  if (warp == 1) { tc_fence_after(); tmem_dealloc(tmem_base, TMEM_MULT * static_cast<uint32_t>(p.bn)); }
}

// ----------------------------------------------------------------------------- MMA issue-rate probe
// One CTA, operands resident in shared memory (zeros), `iters` back-to-back tcgen05.mma 128 x N x 16 into one
// accumulator, timed with clock64 from the first issue to the completion of the commit: cycles per MMA as a function
// of N (what a k-block of four MMAs costs when nothing else is in the way).
__global__ void __launch_bounds__(128, 1) mma_rate_kernel(int N, int iters, long long* out) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + 48 * 1024);
  uint32_t* slot = reinterpret_cast<uint32_t*>(bar + 1);
  for (int i = threadIdx.x; i < 48 * 1024 / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(smem)[i] = 0u;
  if (threadIdx.x == 0) { mbar_init(bar, 1); fence_barrier_init(); }
  fence_proxy_async_smem();
  if (threadIdx.x < 32) { tmem_alloc(slot, 256); tmem_relinquish(); }
  tc_fence_before(); __syncthreads(); tc_fence_after();
  const uint32_t tmem = *slot;
  if (threadIdx.x == 0) {
    const uint32_t idesc = umma_idesc_bf16_f32(128, N);
    const uint64_t ad = desc_k(smem_u32(smem)), bd = desc_k(smem_u32(smem + 16 * 1024));
    const long long t0 = clock64();
    for (int i = 0; i < iters; ++i) umma_bf16_ss(tmem, ad + 2 * (i & 3), bd + 2 * (i & 3), idesc, i ? 1u : 0u);
    umma_commit(bar);
    const long long t1 = clock64();
    mbar_wait(bar, 0, 9);
    const long long t2 = clock64();
    out[0] = t1 - t0; out[1] = t2 - t0;
  }
  tc_fence_before(); __syncthreads();
  if (threadIdx.x < 32) { tc_fence_after(); tmem_dealloc(tmem, 256); }
}

int mma_rate(int N, int iters, long long* out_dev, cudaStream_t st) {
  P3D_REQUIRE(N >= 16 && N <= 256 && N % 16 == 0 && iters >= 1, "mma_rate: bad argument");
  const int smem = 1024 + 48 * 1024 + 64;
  P3D_CUDA(cudaFuncSetAttribute(mma_rate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  mma_rate_kernel<<<1, 128, smem, st>>>(N, iters, out_dev);
  P3D_LAUNCH_CHECK();
  return P3D_OK;
}

// ----------------------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_fn() {
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
// bf16 row-major [outer][inner] (pitch in elements), box [box_outer][64], 128B swizzle, zero fill out of range
static int make_map(CUtensorMap* out, const void* base, uint64_t inner, uint64_t outer, uint64_t pitch, uint32_t box_outer) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) { set_error("cuTensorMapEncodeTiled entry point not available"); return P3D_ERR_CUDA; }
  if ((pitch * 2) % 16 != 0 || (reinterpret_cast<uintptr_t>(base) & 15) != 0) {
    set_error("tc_gemm: operand pitch/base must be 16-byte aligned (pitch %llu elements)", (unsigned long long)pitch);
    return P3D_ERR_ARG;
  }
  cuuint64_t gdim[2] = {inner, outer};
  cuuint64_t gstride[1] = {pitch * 2};
  cuuint32_t box[2] = {64, box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstride, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed with CUresult %d", (int)r); return P3D_ERR_CUDA; }
  return P3D_OK;
}

// A: a_mn ? [K][M] : [M][K];  B: b_mn ? [K][N] : [N][K]  (bf16, pitches lda/ldb in elements)
struct PlanData { CUtensorMap ta, tb; Params p; dim3 grid; int pdl; int fused_mode; int coop; int f16; };
static_assert(sizeof(PlanData) <= sizeof(GemmPlan::blob), "GemmPlan::blob too small");

// tile width: the widest BN that still gives the grid about one CTA per SM; a split-K problem keeps the
// wide tile (better MMA efficiency) and fills the machine through gridDim.z instead
static int pick_bn(int M, int N, int K, bool split_k, bool b_mn) {
  const int mt = (M + BM - 1) / BM;
  const int n64 = (N + 63) / 64 * 64;
  const int kblocks = (K + BK - 1) / BK;
  int bn = 256;
  while (bn > 64 && (bn > n64 || (!split_k && mt * ((N + bn - 1) / bn) < 100))) bn >>= 1;
  // a split-K problem whose K is only a few blocks long (weight gradients of a small batch) is all epilogue:
  // narrow tiles spread it over the machine instead
  if (split_k && kblocks <= 4) { while (bn > 64 && mt * ((N + bn - 1) / bn) < 100) bn >>= 1; }
  // one short M tile (small-batch inference): 32-wide tiles put twice as many SMs on the weight stream
  if (bn == 64 && !b_mn && !split_k && mt == 1 && N >= 256 && (N % 32) == 0) bn = 32;
  return bn;
}

// Can the fused training epilogues (modes 3 / 4) serve an M x N layer?  Every tile must be resident at once (the grid
// meets at a barrier while the accumulators wait in TMEM), i.e. tiles <= SMs.
bool fused_fits(int M, int N, int K, int num_sms) {
  if ((N % 32) != 0) return false;
  const int bn = pick_bn(M, N, K, false, true);
  return ((M + BM - 1) / BM) * ((N + bn - 1) / bn) <= num_sms;
}

int plan(const GemmArgs& g, GemmPlan* out) {
  P3D_REQUIRE(g.M >= 1 && g.N >= 1 && g.K >= 1 && g.A && g.B && (g.C || g.out_bf16), "tc_gemm: bad argument");
  int num_sms = 148;
  { int dev = 0; if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev); }
  const int mt = (g.M + BM - 1) / BM;
  const int kblocks = (g.K + BK - 1) / BK;
  const int bn = pick_bn(g.M, g.N, g.K, g.split_k != 0, g.b_mn != 0);
  const int nt = (g.N + bn - 1) / bn;
  int splits = 1;
  if (g.split_k) {
    splits = num_sms / (mt * nt);
    if (splits < 1) splits = 1;
    if (splits > kblocks) splits = kblocks;
    if (splits > 32) splits = 32;
  }
  const int kps = ((kblocks + splits - 1) / splits) * BK;
  splits = (g.K + kps - 1) / kps;
  PlanData* d = reinterpret_cast<PlanData*>(out->blob);
  // K-major A of a short problem: fetch only the rows that exist (the MMA still reads 128 smem rows; what it makes
  // of the stale ones lands in accumulator rows >= M, which are never stored)
  const int a_rows = (!g.a_mn && g.M < BM) ? ((g.M + 7) / 8 * 8) : BM;
  const bool seg = g.seg_a != 0 || g.seg_b != 0;
  if (seg) {
    P3D_REQUIRE(g.seg_a > 0 && g.seg_b > 0 && !g.accumulate && !g.colsum && !g.fused_mode && !g.res_bf16,
                "tc_gemm: the segment schedule takes split pairs on both sides and the plain, reduction or split-pair epilogues");
    // the lo segment starts past the hi segment's contiguous extent: K (rounded up to a k-block) for a K-major
    // operand, M or N for an MN-major one
    const int need_a = g.a_mn ? g.M : kblocks * BK, need_b = g.b_mn ? g.N : kblocks * BK;
    P3D_REQUIRE(g.seg_a % BK == 0 && g.seg_b % BK == 0 && g.seg_a >= need_a && g.seg_b >= need_b,
                "tc_gemm: lo segments must start at a multiple of %d columns past the hi segment (M %d, N %d, K %d, seg %d / %d)",
                BK, g.M, g.N, g.K, g.seg_a, g.seg_b);
    P3D_REQUIRE(!g.out_bf16 || g.out_lo > 0, "tc_gemm: the segment schedule writes fp32 or split-pair output");
  }
  P3D_REQUIRE(!g.out_lo || (seg && g.out_bf16), "tc_gemm: split-pair output needs the segment schedule and out_bf16");
  // SEG: a map covers both segments of the contiguous dimension; its outer extent is the operand's own, so the K tail
  // of an MN-major operand (batch rows of a weight gradient) is zero-filled by TMA.
  //   K-major: reads past the lo segment's K are zero-filled, the hi segment's K tail is zero padding (must be).
  //   MN-major: a 64-column box past M (N) reads padding, the other segment or zero fill into accumulator rows
  //             (columns) >= M (N), which are never stored - harmless.
  if (!g.a_mn) P3D_TRY(make_map(&d->ta, g.A, g.seg_a + g.K, g.M, g.lda, a_rows));
  else P3D_TRY(make_map(&d->ta, g.A, g.seg_a + g.M, g.K, g.lda, BK));
  if (!g.b_mn) P3D_TRY(make_map(&d->tb, g.B, g.seg_b + g.K, g.N, g.ldb, bn));
  else P3D_TRY(make_map(&d->tb, g.B, g.seg_b + g.N, g.K, g.ldb, BK));
  Params& p = d->p;
  p.M = g.M; p.N = g.N; p.K = g.K; p.bn = bn; p.k_per_split = kps; p.a_mn = g.a_mn; p.b_mn = g.b_mn;
  p.C = g.C; p.ldc = g.ldc; p.bias = g.bias; p.res = g.res; p.ldres = g.ldres; p.alpha_dev = g.alpha_dev; p.alpha = g.alpha;
  p.atomic = (splits > 1 || g.accumulate) ? 1 : 0;
  p.colsum = g.colsum;
  p.out_b = static_cast<__nv_bfloat16*>(g.out_bf16); p.ldob = g.ld_out_bf16;
  p.res_b = static_cast<const __nv_bfloat16*>(g.res_bf16); p.ldrb = g.ld_res_bf16; p.relu = g.relu;
  p.a_bytes = a_rows * BK * 2;
  p.stages = RING_BYTES / (p.a_bytes + bn * BK * 2);
  if (p.stages > MAX_STAGES) p.stages = MAX_STAGES;
  p.b_independent = g.pdl ? 1 : 0;
  p.dbg = static_cast<unsigned long long*>(g.dbg);
  {   // diagnostics (tools/diag_fused_phases.py): stamp the fused kernel of one layer / direction of a training step
    const char* e = getenv("P3D_GEMM_DBG_PTR");
    const char* em = getenv("P3D_GEMM_DBG_MODE");
    const char* el = getenv("P3D_GEMM_DBG_LAYER");
    if (!p.dbg && e && em && g.fused_mode == atoi(em) && (!el || g.fused.layer == atoi(el)))
      p.dbg = reinterpret_cast<unsigned long long*>(strtoull(e, nullptr, 0));
  }
  // diagnostics: P3D_SYNC_TIMEOUT_S=<seconds> makes a grid / peer wait that long trap with a message; by default
  // the fused epilogues wait for their peers like an NCCL collective does (ranks must stay in lockstep)
  static const long long wait_ns = [] { const char* e = getenv("P3D_SYNC_TIMEOUT_S"); return e ? static_cast<long long>(atof(e) * 1e9) : 0LL; }();
  p.wait_limit_ns = wait_ns;
  p.seg_a = g.seg_a; p.seg_b = g.seg_b; p.ob_lo = g.out_lo;
  d->pdl = g.pdl;
  p.ft = g.fused;
  d->fused_mode = g.fused_mode;
  d->coop = 0;
  d->f16 = g.f16;
  P3D_REQUIRE(!g.f16 || (!seg && !g.fused_mode && !g.colsum && !g.split_k && !g.accumulate && !(g.C && g.out_bf16)),
              "tc_gemm: fp16 operands take the inference epilogues only (fp32 store or 16-bit activations)");
  if (g.fused_mode) {
    P3D_REQUIRE(g.fused_mode == 3 || g.fused_mode == 4, "tc_gemm: unknown fused mode %d", g.fused_mode);
    P3D_REQUIRE(splits == 1 && (g.N % 32) == 0 && g.ldc == g.N && !g.out_bf16 && !g.colsum && !g.pdl,
                "tc_gemm: fused training epilogues need N %% 32 == 0, unsplit K, dense C");
    P3D_REQUIRE(!g.res || g.ldres == g.N, "tc_gemm: fused epilogue residual must be dense");
    const bool grid_sync = mt > 1 || g.fused.world > 1;
    if (grid_sync) {
      P3D_REQUIRE(g.fused.gsum && g.fused.gcount, "tc_gemm: grid-synchronised fused epilogue needs gsum / gcount");
      P3D_REQUIRE(mt * nt <= num_sms, "tc_gemm: fused epilogue needs every tile resident (%d tiles, %d SMs)", mt * nt, num_sms);
      P3D_REQUIRE(g.fused.world == 1 || (g.fused.peers && 2 * g.N + 1 <= p2p::MAXN), "tc_gemm: peer exchange not attached / vector too long");
      d->coop = 1;
    } else {
      p.ft.gsum = nullptr;       // one tile: the column sums are CTA-local
    }
  }
  P3D_REQUIRE(!(p.colsum && splits > 1), "tc_gemm: column sums need an unsplit K");
  P3D_REQUIRE(!(p.out_b && splits > 1), "tc_gemm: bf16 output needs an unsplit K");
  d->grid = dim3(nt, mt, splits);
  out->valid = 1;
  return P3D_OK;
}

int launch(const GemmPlan& pl, cudaStream_t st) {
  P3D_REQUIRE(pl.valid, "tc_gemm: launch of an unplanned GEMM");
  const PlanData* d = reinterpret_cast<const PlanData*>(pl.blob);
  using KernelFn = void (*)(const CUtensorMap, const CUtensorMap, const Params);
  const Params& q = d->p;
  const int out = q.ob_lo ? 5 : (q.out_b ? 2 : (q.atomic ? 1 : 0));
  const bool res = (out == 2) ? (q.res_b != nullptr) : (q.res != nullptr);
  const int cs = q.colsum ? 1 : 0;
  const bool seg = q.seg_a != 0;
  KernelFn fn = nullptr;
#define P3D_TCG_PICK(O, R, S) if (!seg && out == O && res == R && cs == S) fn = tc_gemm_kernel<O, R, S>;
  P3D_TCG_PICK(0, false, 0) P3D_TCG_PICK(0, false, 1) P3D_TCG_PICK(0, true, 0) P3D_TCG_PICK(0, true, 1)
  P3D_TCG_PICK(1, false, 0) P3D_TCG_PICK(1, true, 0)
  P3D_TCG_PICK(2, false, 0) P3D_TCG_PICK(2, true, 0)
#undef P3D_TCG_PICK
  if (d->f16) {      // fp16 inference: the output layer (fp32 store) and the hidden layers (16-bit activations)
    fn = nullptr;
    if (!seg && out == 0 && !res && cs == 0) fn = tc_gemm_kernel<0, false, 0, false, true>;
    if (!seg && out == 2 && !res) fn = tc_gemm_kernel<2, false, 0, false, true>;
    if (!seg && out == 2 && res) fn = tc_gemm_kernel<2, true, 0, false, true>;
  }
#define P3D_TCG_PICK_SEG(O, R) if (seg && out == O && res == R && cs == 0) fn = tc_gemm_kernel<O, R, 0, true>;
  P3D_TCG_PICK_SEG(0, false) P3D_TCG_PICK_SEG(5, false) P3D_TCG_PICK_SEG(5, true)
  P3D_TCG_PICK_SEG(0, true) P3D_TCG_PICK_SEG(1, false)       // bf16x3 training: data gradient + residual, split-K weight gradient
#undef P3D_TCG_PICK_SEG
  if (d->fused_mode == 3) fn = tc_gemm_kernel<3, false, 0>;
  if (d->fused_mode == 4) fn = tc_gemm_kernel<4, false, 0>;
  P3D_REQUIRE(fn != nullptr, "tc_gemm: unsupported epilogue combination (out %d res %d colsum %d)", out, (int)res, (int)cs);
  static PerDeviceOnce attr;
  if (attr.needed()) {
    KernelFn all[] = {tc_gemm_kernel<0, false, 0>, tc_gemm_kernel<0, false, 1>, tc_gemm_kernel<0, true, 0>,
                      tc_gemm_kernel<0, true, 1>, tc_gemm_kernel<1, false, 0>, tc_gemm_kernel<1, true, 0>,
                      tc_gemm_kernel<2, false, 0>, tc_gemm_kernel<2, true, 0>,
                      tc_gemm_kernel<3, false, 0>, tc_gemm_kernel<4, false, 0>,
                      tc_gemm_kernel<0, false, 0, true>, tc_gemm_kernel<5, false, 0, true>, tc_gemm_kernel<5, true, 0, true>,
                      tc_gemm_kernel<0, true, 0, true>, tc_gemm_kernel<1, false, 0, true>,
                      tc_gemm_kernel<0, false, 0, false, true>, tc_gemm_kernel<2, false, 0, false, true>, tc_gemm_kernel<2, true, 0, false, true>};
    for (KernelFn f : all) P3D_CUDA(cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    attr.mark();
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = d->grid; cfg.blockDim = dim3(d->fused_mode ? FUSED_NTHREADS : NTHREADS); cfg.dynamicSmemBytes = SMEM_BYTES; cfg.stream = st;
  cudaLaunchAttribute attrs[2];
  if (d->pdl) {
    // programmatic dependent launch: this kernel may start while its predecessor in the stream drains; it orders
    // itself behind the predecessor's memory with griddepcontrol.wait
    attrs[cfg.numAttrs].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attrs[cfg.numAttrs].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attrs; ++cfg.numAttrs;
  }
  if (d->coop) {
    // the grid meets at a barrier inside the kernel: the runtime must place every CTA before any of them waits
    attrs[cfg.numAttrs].id = cudaLaunchAttributeCooperative;
    attrs[cfg.numAttrs].val.cooperative = 1;
    cfg.attrs = attrs; ++cfg.numAttrs;
  }
  P3D_CUDA(cudaLaunchKernelEx(&cfg, fn, d->ta, d->tb, d->p));
  P3D_LAUNCH_CHECK();
  return P3D_OK;
}

int gemm(const GemmArgs& g, cudaStream_t st) {
  GemmPlan pl;
  P3D_TRY(plan(g, &pl));
  return launch(pl, st);
}

}  // namespace tcg
}  // namespace p3d
