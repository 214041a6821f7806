// LinearModel inference for 9 .. 64 poses (BASELINE configs[0]: batch 64) in ONE launch on the whole chip.
//   reference: linear_model.py:96-127 (the forward graph), :237-245 (step, isTraining=False), batch_size flag = 64
//
// The per-layer tcgen05 GEMM chain (mlp_layered.cu) needs ~7 us per layer at these sizes whatever the batch: launch ->
// TMA -> 16 serial k-blocks -> TMEM -> store -> exit, six times (41 us at 64 poses for 2 us of tensor work).  Here, like
// in the batch-1 whole-chip kernel (mlp_simt.cu), every CTA owns a slice of the output features of EVERY layer, keeps
// its whole share of the weights in shared memory (requested by bulk copies in the first instructions) and the layers
// hand over through self-validating words in L2 - no grid barrier, no kernel boundary:
//
//   grid     64 feature groups (16 features of every hidden layer) x G row groups (16 or 32 poses each), G <= 2:
//            64 or 128 CTAs, cooperative launch (all resident: consumers spin on what the others produce)
//   weights  4 hidden layers x 16 rows x 2 KB (+ 8 rows of the output layer) = 145 KB per CTA, rows 16 B apart from a
//            multiple of 128 B so that the MMA fragment loads are bank-conflict free
//   math     mma.sync.m16n8k16 bf16 -> fp32 (legacy tensor-core path: a 32 x 16 x 1024 problem per CTA and layer is far
//            below what tcgen05 needs to pay for its TMEM round trip); the 8 warps split K, partial sums meet in
//            shared memory
//   exchange act[layer][pose][512] words {2 x bf16, launch tag}: a producer stores each word with ONE 8-byte store, the
//            consumers poll the words they need until they carry this launch's tag (no flag, no fence: an 8-byte
//            aligned access is single-copy atomic); the tag comes from the model's epoch word in device memory, which
//            every launch advances on its way out (xchg_tag in common.cuh), so nothing is ever cleared and a launch
//            captured into a CUDA graph gets a fresh tag on every replay
//   rounding the same points as the tcgen05 paths (x, every ReLU output and every residual sum rounded to bf16, fp32
//            accumulation): tests/helpers.py:emulate_bf16_forward
//   fp16     P3D_MODE_FP16 models: F16 = true - fp16 weights, mma.sync .f16 operands, fp16 rounding and {2 x fp16, tag}
//            exchange words, everything else as above
#include "common.cuh"

namespace p3d {
namespace mid {

constexpr int MGT = 256;                  // threads per CTA: 8 warps, each takes 1/8 of K
constexpr int NF = 16;                    // features per CTA and hidden layer (two n8 tiles)
constexpr int NFG = 1024 / NF;            // feature groups
constexpr int PITCH = 2048 + 16;          // bytes per shared-memory row: word index = row * 516 + k / 2 -> bank 4 row + t
constexpr int MAXHID = 4;
constexpr int NOUT = 8;                   // output-layer features per CTA (one n8 tile); CTAs fg < ceil(out / 8) compute them

struct Args {
  const float* x; float* y; const __nv_bfloat16* wt; const float* bias;
  unsigned long long* act;                // [nlayers - 1][64 poses][512] {bf16 pair, tag}
  unsigned* xchg;                         // epoch + arrival counter (p3d_model::xchg)
  int nlayers, out, kpad, residual, rows;
  int sentinel;                           // poll one pose until it arrives before requesting the batch (diagnostics switch)
  unsigned long long* stamps;             // optional [16] %globaltimer stamps of CTA 0 (P3D_LAT_STAMPS=1, tools/bench_latency.py)
};
#define MID_STAMP(i) do { if (a.stamps && threadIdx.x == 0 && blockIdx.x == 0) { unsigned long long t_; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_)); a.stamps[i] = t_; } } while (0)

__device__ __forceinline__ uint32_t smem_addr(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbar_init(uint64_t* b, uint32_t n) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(b)), "r"(n) : "memory"); }
__device__ __forceinline__ void mbar_expect(uint64_t* b, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* b, uint32_t parity) {
  uint32_t ok = 0, spins = 0;
  while (!ok) {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok) : "r"(smem_addr(b)), "r"(parity) : "memory");
    if (!ok && ++spins > (1u << 24)) { printf("p3d: mid-batch kernel: weights never arrived (block %d)\n", (int)blockIdx.x); __trap(); }
  }
}
__device__ __forceinline__ void bulk_row(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_addr(dst)), "l"(src), "r"(bytes), "r"(smem_addr(bar)) : "memory");
}
__device__ __forceinline__ void st_word(unsigned long long* p, uint32_t data, uint32_t tag) {
  const unsigned long long v = static_cast<unsigned long long>(data) | (static_cast<unsigned long long>(tag) << 32);
  asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void ld_words(const unsigned long long* p, unsigned long long& a, unsigned long long& b) {
  asm volatile("ld.volatile.global.v2.u64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "l"(p) : "memory");
}
__device__ __forceinline__ uint32_t lds32(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ void mma_bf16(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3]) : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void mma_f16(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3]) : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
template <bool F16> __device__ __forceinline__ float r16(float v) { return Op16<F16>::to(Op16<F16>::from(v)); }
template <bool F16> __device__ __forceinline__ uint32_t pack16(float lo, float hi) {
  const typename Op16<F16>::T2 p = Op16<F16>::pack(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&p);
}

template <int MT, bool F16 = false>      // m16 tiles per CTA: a row group is 16 MT poses
__global__ void __launch_bounds__(MGT, 1) mid_grid_kernel(const Args a) {
  using O = Op16<F16>;
  constexpr int RG = 16 * MT;
  extern __shared__ __align__(128) uint8_t mg_smem[];
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(mg_smem) + 127) & ~uintptr_t(127));
  const int nhid = a.nlayers - 2;
  uint8_t* wsm = base;                                        // [nhid][16 rows] hidden-layer weights
  uint8_t* wout = wsm + MAXHID * NF * PITCH;                   // [8 rows] output layer
  uint8_t* sact = wout + NOUT * PITCH;                         // [RG rows] input activations of the running layer (bf16) ...
  float* sred = reinterpret_cast<float*>(sact);                // ... and, after the MMAs, the warps' partial sums [8][RG][16]
  float* sres = reinterpret_cast<float*>(sact + RG * PITCH);   // [RG][16] this CTA's own block input (residual)
  uint64_t* wbar = reinterpret_cast<uint64_t*>(sres + RG * NF);   // [nhid + 1]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int fg = blockIdx.x % NFG, rg = blockIdx.x / NFG;
  const int row0 = rg * RG;
  const int live = min(RG, a.rows - row0);                     // poses of this row group that exist (>= 1 by the launch)
  const int nout_groups = (a.out + NOUT - 1) / NOUT;
  const bool has_out = fg < nout_groups;
  const int out_rows = has_out ? min(NOUT, a.out - fg * NOUT) : 0;

  MID_STAMP(0);
  const unsigned tag = xchg_tag(a.xchg);                       // in flight with the weight copies; first used by layer 0's stores
  unsigned arrived = 0;                                        // thread 0: CTAs that arrived before this one
  if (tid == 0) {
    for (int l = 0; l <= nhid; ++l) mbar_init(&wbar[l], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // unused rows must not hold NaN patterns: pad rows of the activations (poses that do not exist) and the missing rows of
  // a ragged output group only meet accumulator rows / columns that are never stored, but keep them finite anyway
  for (int i = tid; i < (RG * PITCH) / 16; i += MGT) reinterpret_cast<uint4*>(sact)[i] = make_uint4(0, 0, 0, 0);
  for (int i = tid; i < (NOUT * PITCH) / 16; i += MGT) reinterpret_cast<uint4*>(wout)[i] = make_uint4(0, 0, 0, 0);
  __syncthreads();
  // the CTA's whole share of the weights is requested now, row by row (padded pitch), by the last warp: lane 0 announces
  // the byte counts, every lane issues a few of the 72 row copies
  if (warp == MGT / 32 - 1) {
    if (lane == 0) {
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");        // the zero fill above vs the bulk copies below
      for (int l = 0; l < nhid; ++l) mbar_expect(&wbar[l], NF * 2048);
      if (has_out) mbar_expect(&wbar[nhid], out_rows * 2048);
    }
    __syncwarp();
    for (int i = lane; i < nhid * NF; i += 32) {
      const int l = i / NF, r = i % NF;
      bulk_row(wsm + i * PITCH, a.wt + (static_cast<size_t>(1 + l) * 1024 + fg * NF + r) * a.kpad, 2048, &wbar[l]);
    }
    if (lane < out_rows)
      bulk_row(wout + lane * PITCH, a.wt + (static_cast<size_t>(a.nlayers - 1) * 1024 + fg * NOUT + lane) * a.kpad, 2048, &wbar[nhid]);
  }
  auto words = [&](int l, int row) { return a.act + (static_cast<size_t>(l) * 64 + row) * 512; };
  // this thread's outputs in the epilogue of a hidden layer: pose er of the group, features 2 ej and 2 ej + 1 of the CTA's 16
  const int er = tid >> 3, ej = tid & 7;
  const bool epi = er < RG;

  // ---- layer 0 (K = 32): x and the weight rows straight from L2, fp32 FMA on bf16-rounded operands
  if (epi) {
    float acc0 = 0.f, acc1 = 0.f;
    const int n = fg * NF + 2 * ej;
    if (er < live) {
      const uint4* w0 = reinterpret_cast<const uint4*>(a.wt + static_cast<size_t>(n) * a.kpad);
      const uint4* w1 = reinterpret_cast<const uint4*>(a.wt + static_cast<size_t>(n + 1) * a.kpad);
      const float4* xr = reinterpret_cast<const float4*>(a.x + static_cast<size_t>(row0 + er) * kIn);
#pragma unroll
      for (int q = 0; q < 4; ++q) {                             // 8 inputs per step
        const uint4 u0 = __ldg(w0 + q), u1 = __ldg(w1 + q);
        const float4 xa = __ldg(xr + 2 * q), xb = __ldg(xr + 2 * q + 1);
        const float xs[8] = {r16<F16>(xa.x), r16<F16>(xa.y), r16<F16>(xa.z), r16<F16>(xa.w), r16<F16>(xb.x), r16<F16>(xb.y), r16<F16>(xb.z), r16<F16>(xb.w)};
        const typename O::T2* p0 = reinterpret_cast<const typename O::T2*>(&u0);
        const typename O::T2* p1 = reinterpret_cast<const typename O::T2*>(&u1);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          acc0 = fmaf(xs[2 * i], O::lo(p0[i]), acc0); acc0 = fmaf(xs[2 * i + 1], O::hi(p0[i]), acc0);
          acc1 = fmaf(xs[2 * i], O::lo(p1[i]), acc1); acc1 = fmaf(xs[2 * i + 1], O::hi(p1[i]), acc1);
        }
      }
    }
    const float v0 = r16<F16>(fmaxf(acc0 + __ldg(a.bias + n), 0.f)), v1 = r16<F16>(fmaxf(acc1 + __ldg(a.bias + n + 1), 0.f));
    sres[er * NF + 2 * ej] = v0; sres[er * NF + 2 * ej + 1] = v1;             // block input of the first residual block
    if (er < live) st_word(words(0, row0 + er) + fg * (NF / 2) + ej, pack16<F16>(v0, v1), tag);
  }
  MID_STAMP(1);

  // all of layer lp's outputs for this row group -> sact (bf16 rows): every thread polls the two words per pose it copies
  auto gather = [&](int lp) {
    // Polling all poses at once keeps the L2 busy with reads while the producers try to write (128 CTAs x 64 KB per poll
    // round; polling 32 poses at a time, a 64-pose call took 39 us instead of 25).  So every thread first polls ONE
    // sentinel - its two words of the group's first pose - and only when they carry the tag requests a batch of 16 poses:
    // the words of the other poses come from the same producer CTA and were stored by the same instruction, a few
    // warps apart, so the batch is almost always complete at the first try (it is re-polled until it is).  Poses that do
    // not exist are not loaded at all.  Measured alternatives (profiles/r2_mid_batch_latency.txt, 32 / 64 poses): no
    // sentinel 20.4 / 26.7 us; unconditional loads (absent poses re-reading live ones) 21.9 / 32.8 us, with the sentinel
    // 22.0 / 36.5 us; every CTA walking the poses from its own starting row 20.5 / 30.8 us; this form 18.4 / 26.6 us.
    const unsigned long long* src = words(lp, row0) + tid * 2;
    unsigned spins = 0;
    if (a.sentinel) {
      unsigned long long s0, s1;
      for (;;) {
        ld_words(src, s0, s1);
        if (static_cast<uint32_t>(s0 >> 32) == tag && static_cast<uint32_t>(s1 >> 32) == tag) break;
        if (++spins > (1u << 24)) { printf("p3d: mid-batch kernel: layer %d never arrived (block %d)\n", lp, (int)blockIdx.x); __trap(); }
      }
    }
#pragma unroll
    for (int b = 0; b < MT; ++b) {
      if (b * 16 >= live) break;
      unsigned long long w0[16], w1[16];
      for (;;) {
        bool ok = true;
#pragma unroll
        for (int r = 0; r < 16; ++r)
          if (b * 16 + r < live) ld_words(src + static_cast<size_t>(b * 16 + r) * 512, w0[r], w1[r]);
#pragma unroll
        for (int r = 0; r < 16; ++r)
          if (b * 16 + r < live) ok = ok && static_cast<uint32_t>(w0[r] >> 32) == tag && static_cast<uint32_t>(w1[r] >> 32) == tag;
        if (ok) break;
        if (++spins > (1u << 24)) { printf("p3d: mid-batch kernel: layer %d never arrived (block %d)\n", lp, (int)blockIdx.x); __trap(); }
      }
#pragma unroll
      for (int r = 0; r < 16; ++r)
        if (b * 16 + r < live)
          *reinterpret_cast<uint2*>(sact + (b * 16 + r) * PITCH + tid * 8) = make_uint2(static_cast<uint32_t>(w0[r]), static_cast<uint32_t>(w1[r]));
    }
  };
  // acc[mt][nt] += sact[16 mt .. +16][k range of this warp] x w[8 nt .. +8][same k]^T
  const int g = lane >> 2, t = lane & 3;
  auto mma_layer = [&](const uint8_t* w, int ntiles, float (&acc)[MT][2][4]) {
    const uint32_t sa = smem_addr(sact) + g * PITCH + (warp * 128 + 2 * t) * 2;
    const uint32_t sw = smem_addr(w) + g * PITCH + (warp * 128 + 2 * t) * 2;
#pragma unroll
    for (int ks = 0; ks < 8; ++ks) {
      uint32_t bf[2][2];
#pragma unroll
      for (int nt = 0; nt < 2; ++nt) {
        if (nt < ntiles) {
          bf[nt][0] = lds32(sw + nt * 8 * PITCH + ks * 32);
          bf[nt][1] = lds32(sw + nt * 8 * PITCH + ks * 32 + 16);
        } else { bf[nt][0] = 0; bf[nt][1] = 0; }
      }
#pragma unroll
      for (int mt = 0; mt < MT; ++mt) {
        const uint32_t ra = sa + mt * 16 * PITCH + ks * 32;
        const uint32_t a0 = lds32(ra), a1 = lds32(ra + 8 * PITCH), a2 = lds32(ra + 16), a3 = lds32(ra + 8 * PITCH + 16);
#pragma unroll
        for (int nt = 0; nt < 2; ++nt)
          if (nt < ntiles) {
            if constexpr (F16) mma_f16(acc[mt][nt], a0, a1, a2, a3, bf[nt][0], bf[nt][1]);
            else mma_bf16(acc[mt][nt], a0, a1, a2, a3, bf[nt][0], bf[nt][1]);
          }
      }
    }
  };
  // the warps' partial sums -> sred[warp][pose][16] (sact is dead by now: the caller put a block barrier in between)
  auto spill = [&](const float (&acc)[MT][2][4], int ntiles) {
#pragma unroll
    for (int mt = 0; mt < MT; ++mt)
#pragma unroll
      for (int nt = 0; nt < 2; ++nt) {
        if (nt >= ntiles) continue;
        float* d = sred + (static_cast<size_t>(warp) * RG + mt * 16 + g) * NF + nt * 8 + 2 * t;
        *reinterpret_cast<float2*>(d) = make_float2(acc[mt][nt][0], acc[mt][nt][1]);
        *reinterpret_cast<float2*>(d + 8 * NF) = make_float2(acc[mt][nt][2], acc[mt][nt][3]);
      }
  };

  // ---- hidden layers 1 .. nhid.  The residual of an even layer is the block input (output of layer l - 2), whose 16
  // features of this row group the CTA produced itself: sres.
  for (int l = 1; l <= nhid; ++l) {
    // every thread of the CTA has compared its tag in the first gather: arrive, while the outputs of layer 1 are on their way
    if (l == 2 && tid == 0) arrived = xchg_arrive(a.xchg);
    gather(l - 1);
    __syncthreads();
    mbar_wait(&wbar[l - 1], 0);
    float acc[MT][2][4];
#pragma unroll
    for (int mt = 0; mt < MT; ++mt)
#pragma unroll
      for (int nt = 0; nt < 2; ++nt)
#pragma unroll
        for (int i = 0; i < 4; ++i) acc[mt][nt][i] = 0.f;
    mma_layer(wsm + (l - 1) * NF * PITCH, 2, acc);
    __syncthreads();                                           // every warp has read sact: it becomes the reduction scratch
    spill(acc, 2);
    __syncthreads();
    if (epi) {
      float s0 = 0.f, s1 = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) {
        const float2 p = *reinterpret_cast<const float2*>(sred + (static_cast<size_t>(w) * RG + er) * NF + 2 * ej);
        s0 += p.x; s1 += p.y;
      }
      const int n = fg * NF + 2 * ej;
      float v0 = r16<F16>(fmaxf(s0 + __ldg(a.bias + l * 1024 + n), 0.f)), v1 = r16<F16>(fmaxf(s1 + __ldg(a.bias + l * 1024 + n + 1), 0.f));
      if (!(l & 1)) {
        if (a.residual) { v0 = r16<F16>(v0 + sres[er * NF + 2 * ej]); v1 = r16<F16>(v1 + sres[er * NF + 2 * ej + 1]); }
        sres[er * NF + 2 * ej] = v0; sres[er * NF + 2 * ej + 1] = v1;
      }
      if (er < live) st_word(words(l, row0 + er) + fg * (NF / 2) + ej, pack16<F16>(v0, v1), tag);
    }
    __syncthreads();                                           // the next gather overwrites the scratch
    MID_STAMP(1 + l);
  }
  // ---- output layer: feature group fg < ceil(out / 8) computes 8 features for its row group
  if (nhid < 2 && tid == 0) arrived = xchg_arrive(a.xchg);
  if (has_out) {
    gather(nhid);
    __syncthreads();
    mbar_wait(&wbar[nhid], 0);
    float acc[MT][2][4];
#pragma unroll
    for (int mt = 0; mt < MT; ++mt)
#pragma unroll
      for (int nt = 0; nt < 2; ++nt)
#pragma unroll
        for (int i = 0; i < 4; ++i) acc[mt][nt][i] = 0.f;
    mma_layer(wout, 1, acc);
    __syncthreads();
    spill(acc, 1);
    __syncthreads();
    for (int o = tid; o < RG * NOUT; o += MGT) {
      const int r = o >> 3, c = o & 7;
      float s = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) s += sred[(static_cast<size_t>(w) * RG + r) * NF + c];
      const int n = fg * NOUT + c;
      if (r < live && n < a.out) a.y[static_cast<size_t>(row0 + r) * a.out + n] = s + __ldg(a.bias + (a.nlayers - 1) * 1024 + n);
    }
  }
  if (tid == 0 && arrived == gridDim.x - 1) xchg_advance(a.xchg, tag);
  MID_STAMP(a.nlayers);
}

constexpr int smem_bytes(int mt) { return 128 + MAXHID * NF * PITCH + NOUT * PITCH + 16 * mt * PITCH + 16 * mt * NF * 4 + 8 * (MAXHID + 1) + 64; }

// 9 .. 64 poses, linear_size 1024, <= 4 hidden layers; returns 1 when this kernel cannot serve the call (another path takes it)
int forward(p3d_model* m, const float* x, float* y, int rows, cudaStream_t st) {
  static const bool on = [] { const char* e = getenv("P3D_MID_GRID"); return !(e && e[0] == '0'); }();     // P3D_MID_GRID=0: per-layer GEMMs instead
  const int nlayers = static_cast<int>(m->layers.size()), nhid = nlayers - 2;
  if (!on || m->L != 1024 || m->kpad != 1024 || nhid < 1 || nhid > MAXHID || m->out_size > 64 || rows < 1 || rows > 64) return 1;
  const int mt = rows > 32 ? 2 : 1;
  const int groups = (rows + 16 * mt - 1) / (16 * mt);
  if (m->num_sms < NFG * groups) return 1;
  if (!m->mid_act) return 1;                            // allocated (2 MB, zero) by p3d_model_create for width 1024 / bf16 / fp16
  static PerDeviceOnce attr;
  if (attr.needed()) {
    P3D_TRY(refuse_in_capture(st, "forward: first use of the 9-64 pose whole-chip kernel on this device"));
    P3D_CUDA(cudaFuncSetAttribute(mid_grid_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes(1)));
    P3D_CUDA(cudaFuncSetAttribute(mid_grid_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes(2)));
    P3D_CUDA(cudaFuncSetAttribute(mid_grid_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes(1)));
    P3D_CUDA(cudaFuncSetAttribute(mid_grid_kernel<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes(2)));
    attr.mark();
  }
  Args a;
  a.x = x; a.y = y; a.wt = m->wt_bf16; a.bias = m->bias_fold; a.act = static_cast<unsigned long long*>(m->mid_act); a.xchg = m->xchg;
  a.nlayers = nlayers; a.out = m->out_size; a.kpad = m->kpad; a.residual = m->cfg.residual; a.rows = rows;
  static const int sentinel = [] { const char* e = getenv("P3D_MID_SENTINEL"); return e ? atoi(e) : 1; }();
  a.sentinel = sentinel;
  a.stamps = nullptr;
  if (getenv("P3D_LAT_STAMPS")) a.stamps = m->lat_counter + 8;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(NFG * groups); cfg.blockDim = dim3(MGT); cfg.dynamicSmemBytes = smem_bytes(mt); cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeCooperative; at[0].val.cooperative = 1;     // every CTA polls what the others produce
  cfg.attrs = at; cfg.numAttrs = 1;
  const bool f16 = m->cfg.mode == P3D_MODE_FP16;
  if (mt == 1) P3D_CUDA(cudaLaunchKernelEx(&cfg, f16 ? mid_grid_kernel<1, true> : mid_grid_kernel<1>, a));
  else P3D_CUDA(cudaLaunchKernelEx(&cfg, f16 ? mid_grid_kernel<2, true> : mid_grid_kernel<2>, a));
  P3D_LAUNCH_CHECK();
  return P3D_OK;
}

}  // namespace mid
}  // namespace p3d
