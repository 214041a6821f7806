// Shared host-side plumbing for libp3d: error reporting, launch accounting, model state.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <atomic>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <string>
#include <vector>

#include "../../include/p3d.h"

namespace p3d {

void set_error(const char* fmt, ...);
void count_launch(int n = 1);
long long launch_count_now();

#define P3D_CUDA(expr)                                                                          \
  do {                                                                                          \
    cudaError_t e__ = (expr);                                                                   \
    if (e__ != cudaSuccess) {                                                                   \
      ::p3d::set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #expr, cudaGetErrorString(e__)); \
      return P3D_ERR_CUDA;                                                                      \
    }                                                                                           \
  } while (0)

#define P3D_LAUNCH_CHECK()                                                                      \
  do {                                                                                          \
    ::p3d::count_launch();                                                                      \
    cudaError_t e__ = cudaGetLastError();                                                       \
    if (e__ != cudaSuccess) {                                                                   \
      ::p3d::set_error("%s:%d: kernel launch failed: %s", __FILE__, __LINE__, cudaGetErrorString(e__)); \
      return P3D_ERR_CUDA;                                                                      \
    }                                                                                           \
  } while (0)

#define P3D_REQUIRE(cond, ...)          \
  do {                                  \
    if (!(cond)) {                      \
      ::p3d::set_error(__VA_ARGS__);    \
      return P3D_ERR_ARG;               \
    }                                   \
  } while (0)

#define P3D_TRY(expr)            \
  do {                           \
    int rc__ = (expr);           \
    if (rc__ != P3D_OK) return rc__; \
  } while (0)

// Function attributes (dynamic shared memory limit, cluster size) belong to the device's context, not to the process:
// a flag that remembers "already set" must be kept per device, or the second GPU used by one process launches with
// the 48 KB default and fails.  `if (once.needed()) { ...cudaFuncSetAttribute...; once.mark(); }`
struct PerDeviceOnce {
  std::atomic<unsigned long long> mask{0};
  static unsigned long long bit() { int d = 0; cudaGetDevice(&d); return 1ull << (d & 63); }
  bool needed() const { return (mask.load(std::memory_order_acquire) & bit()) == 0; }
  void mark() { mask.fetch_or(bit(), std::memory_order_release); }
};

// The 16-bit operand type of the inference kernels: bf16 (P3D_MODE_BF16) or fp16 (P3D_MODE_FP16).  Both modes round
// at the same points; the packed weights, packed input and 16-bit activations hold bf16 or fp16 bits accordingly.
template <bool F16> struct Op16;
template <> struct Op16<false> {
  using T = __nv_bfloat16; using T2 = __nv_bfloat162;
  static __device__ __forceinline__ T from(float v) { return __float2bfloat16_rn(v); }
  static __device__ __forceinline__ float to(T v) { return __bfloat162float(v); }
  static __device__ __forceinline__ T2 pack(float a, float b) { return __floats2bfloat162_rn(a, b); }
  static __device__ __forceinline__ float lo(T2 v) { return __low2float(v); }
  static __device__ __forceinline__ float hi(T2 v) { return __high2float(v); }
};
template <> struct Op16<true> {
  using T = __half; using T2 = __half2;
  static __device__ __forceinline__ T from(float v) { return __float2half_rn(v); }
  static __device__ __forceinline__ float to(T v) { return __half2float(v); }
  static __device__ __forceinline__ T2 pack(float a, float b) { return __floats2half2_rn(a, b); }
  static __device__ __forceinline__ float lo(T2 v) { return __low2float(v); }
  static __device__ __forceinline__ float hi(T2 v) { return __high2float(v); }
};

constexpr float kBnEps = 1e-3f;       // tf.layers.batch_normalization default
constexpr float kBnMomentum = 0.99f;  // idem
constexpr int kIn = 32;               // HUMAN_2D_SIZE (linear_model.py:60)

// One Linear(+BN) stage of the network, in graph order: w1 | (w2_i, w3_i)* | w4.
struct Layer {
  int K = 0, N = 0;
  bool has_bn = false;   // hidden layers when cfg.batch_norm
  bool hidden = true;    // false for the output layer (no BN/ReLU/dropout)
  // offsets (in floats) into the flat trainable buffer theta / grad / adam_m / adam_v
  size_t off_w = 0, off_b = 0, off_gamma = 0, off_beta = 0;
  // offsets into the flat non-trainable buffer (moving_mean | moving_variance)
  size_t off_mm = 0, off_mv = 0;
  // packed inference weights: row offset into wt_bf16 / bias_fold
  int row_off = 0;
  // fp32 folded weights [K,N] offset into wfold
  size_t off_wfold = 0;
  std::string wname, bname, bnscope;
};

struct NamedParam {
  std::string name;
  float* ptr;     // device
  size_t numel;
  bool affects_inference;
};

struct TrainWorkspace {
  int64_t cap_B = 0;
  float* z = nullptr;       // [nhidden][B][L] pre-BN activations
  float* h = nullptr;       // [nhidden][B][L] post-dropout(+residual) activations
  float* dh = nullptr;      // [B][L] gradient wrt current layer output
  float* dz = nullptr;      // [B][L]
  float* dres = nullptr;    // [B][L] residual-path gradient
  uint8_t* maskbuf = nullptr;  // [nhidden][B][L] dropout keep-masks
  float* dy = nullptr;      // [B][out]
  double* stats = nullptr;  // [nhidden][2][L] sum, sumsq (double) then mean,var
  float* mean = nullptr;    // [nhidden][L]
  float* rstd = nullptr;    // [nhidden][L]
  double* red = nullptr;    // [nhidden][2][L] backward sums (dgamma, dbeta) + misc scalars
  unsigned* gcount = nullptr;   // [2 nhidden][2] arrival counter + completion flag of the grid-synchronised fused epilogues
  float* scal = nullptr;    // small device scalars: loss, lr, clip dots...
  // bf16 operands of the tensor-core path (P3D_MODE_BF16)
  __nv_bfloat16* xb = nullptr;    // [B][32]
  __nv_bfloat16* hb = nullptr;    // [nhidden][B][L]
  __nv_bfloat16* dzb = nullptr;   // [B][L]
  __nv_bfloat16* dyb = nullptr;   // [B][48] (pad columns zero)
  __nv_bfloat16* wb = nullptr;    // weights [K][N] per layer at theta's offsets; W4 rows padded to 48
  // split-pair operands of the bf16x3 training route (P3D_TRAIN_MATMUL_BF16X3): every row [hi segment | lo segment],
  // segment = width rounded up to 64 columns (x, dy, W4: 64), padding zero.  Allocated zeroed.
  int64_t x3_B = 0;                // rows xs / hs / dzs / dys hold
  __nv_bfloat16* xs = nullptr;     // [B][128]
  __nv_bfloat16* hs = nullptr;     // [nhidden][B][2 seg]
  __nv_bfloat16* dzs = nullptr;    // [B][2 seg]
  __nv_bfloat16* dys = nullptr;    // [B][128]
  __nv_bfloat16* ws = nullptr;     // weights [K][2 seg_N] per layer at ws_off (unclipped; the clip scale is the GEMM's alpha)
  std::vector<size_t> ws_off;      // per layer, elements into ws
  void* tab = nullptr;            // device LayerTabEntry[nlayers]
  void* sc = nullptr;             // device StepScalars (per-step values: Adam step size, lr, dropout seed/step)
  // CUDA-graph replay of the step: fixed-address staging of x / t / y / (loss, lr) and one graph per (B, dropout)
  float* gx = nullptr; float* gt = nullptr; float* gy = nullptr; float* gscal = nullptr;
  struct GraphEntry { int64_t B; int dropout; int launches; void* exec; int64_t Bg; int64_t row0; };
  std::vector<GraphEntry> graphs;
  cudaStream_t cap_stream = nullptr;
  // the weight-gradient GEMMs of the fused small-batch step run on a side stream (a parallel branch of the graph)
  cudaStream_t side_stream = nullptr;
  cudaEvent_t ev[16] = {};
};

// Optional per-launch CUDA-event timing of the dominant kernel (bench.py's roofline figure):
// events are recorded on the launching stream right around the kernel.
namespace prof {
bool enabled();
void begin(cudaStream_t st, cudaEvent_t* e0, cudaEvent_t* e1);
void end(cudaStream_t st, cudaEvent_t e0, cudaEvent_t e1);
}  // namespace prof

namespace simt {
struct Epilogue {
  const float* bias = nullptr;        // [N] added to every row
  const float* res = nullptr;         // [M,N] (ldc) added after the activation
  int relu = 0;
  const float* alpha_dev = nullptr;   // optional device scalar multiplying the product (clip scale)
  float alpha = 1.f;
  float beta = 0.f;                   // C = alpha*AB + beta*C before bias/activation
};
// C[M,N] = epi(alpha * op(A)[M,K] op(B)[K,N]);  op(A)[m,k] = ta ? A[k*lda+m] : A[m*lda+k],
// op(B)[k,n] = tb ? B[n*ldb+k] : B[k*ldb+n]
int sgemm(bool ta, bool tb, int64_t M, int N, int K, const float* A, int lda, const float* B, int ldb, float* C,
          int ldc, const Epilogue& e, cudaStream_t st);
}  // namespace simt
namespace rt {
// Realtime front-end / back-end around the lifter (src/openpose_3dpose_sandbox_realtime.py:137-171): device tables.
struct Tables {
  double mu2[32], sd2[32];      // data_mean_2d[dim_to_use_2d], data_std_2d[dim_to_use_2d]
  int use2[32];                 // dim_to_use_2d (coordinate index into the 64-vector)
  double mu3[96], sd3[96];      // data_mean_3d, data_std_3d (all 96 dims)
  int use3[48];                 // dim_to_use_3d (first `out` entries)
  int pos3[96];                 // inverse: network output column of full dim j, or -1 (ignored dim)
  int out;
};
// Extra operands of the batch-1 cluster kernel when it runs the whole realtime step in one launch.
struct Fused {
  const Tables* tab = nullptr;                  // nullptr = plain forward
  const double* kp = nullptr;                   // [36] keypoints (host-mapped or device memory)
  float* enc = nullptr;                         // [32] normalised network input
  double* pose = nullptr;                       // [96] un-normalised prediction (only the used dims are written)
  unsigned long long* flag = nullptr;           // completion flag (host-mapped), set to seq after all outputs
  unsigned long long seq = 0;
};
}  // namespace rt
namespace simt {
int forward_latency_cluster_rt(p3d_model* m, const rt::Fused& f, float* y, cudaStream_t st);
}
namespace p2p {
// One rank's exchange buffer for the latency-bound reductions of the data-parallel step (SyncBN sums, loss), mapped by
// every rank of the node through CUDA IPC (p2p.cu).  Written by peers with NVLink stores, flags carry sequence numbers.
constexpr int NSLOTS = 4;
constexpr int MAXN = 8192;          // doubles per reduction (2 x linear_size <= 4096)
constexpr int MAXW = 16;
constexpr int YMAX = 1 << 19;       // floats of gathered step outputs (10922 rows of 48)
struct Layout {
  double data[NSLOTS][MAXW][MAXN];
  unsigned long long flag[NSLOTS][MAXW];
  unsigned long long seq;           // last completed sequence number (local)
  // gradient all-reduce (p2p.cu grad_allreduce_kernel): entry / exit flags per peer, sequence number, CTA counter
  unsigned long long gflag[2][MAXW];
  unsigned long long gseq;
  unsigned int gdone;
  // Low-latency form of `data` for the exchanges inside the fused GEMM epilogues: every double travels as two 8-byte
  // words {32 payload bits, 32-bit sequence tag}; a word is valid when its tag is the exchange's sequence number, so the
  // receiver polls the data itself - no release fence and no separate flag hop (one NVLink write latency per exchange).
  uint4 ll[NSLOTS][MAXW][MAXN + 8];
  // outputs of the last data-parallel step for the GLOBAL batch: every rank writes its rows into every rank's copy from
  // inside the gradient all-reduce kernel (between its handshakes), so model.step() needs no all-gather of its own
  float ybuf[YMAX];
};
struct Peers { Layout* p[MAXW]; };
struct GradPeers { float* g[MAXW]; };   // every rank's flat gradient buffer, peer-mapped
bool ready(const p3d_model* m);
bool grad_ready(const p3d_model* m);               // the gradient buffers of all ranks are mapped too
// m->grad <- sum over ranks, summed in rank order; y_local (may be null): this rank's [rows][out] step outputs, written to
// rows row0.. of every rank's Layout::ybuf on the way
int allreduce_grad(p3d_model* m, size_t n, const float* y_local, long long rows, long long row0, int out, cudaStream_t st);
const float* gathered_outputs(const p3d_model* m);          // this rank's Layout::ybuf
const Peers* device_peers(const p3d_model* m);     // device copy of the peer table (null until attached)
struct BnFinalize {                 // optional fused tail: BatchNorm statistics from the reduced [sum | sumsq]
  double invB = 0.0;
  float* mean = nullptr; float* rstd = nullptr; float* mm = nullptr; float* mv = nullptr;
};
int allreduce_small(p3d_model* m, double* buf, size_t n, cudaStream_t st, const BnFinalize* fin = nullptr);
void destroy(p3d_model* m);
}  // namespace p2p
namespace tcg {
// Extra operands of the fused training epilogues of tc_gemm.cu: the BatchNorm / ReLU / dropout arithmetic of a hidden
// layer inside the GEMM that produces its input, forward and backward.
//   mode 3, forward : acc = h_in W;  z = alpha acc + bias -> C;  BN batch statistics over the rows (mean / rstd /
//                     moving averages written), ReLU, dropout (Philox or injected mask), + residual -> h, hb, mask
//   mode 4, backward: acc = dz_next W^T;  dh = alpha acc (+ res) (-> dh_out);  da = dh * dropout * relu';  BN backward
//                     with the column sums of da and da * xhat -> dzb (bf16), dgamma / dbeta (or the bias gradient)
// The accumulator stays in TMEM between the two passes the column statistics need.  With one M tile (batch <= 128, one
// GPU) the column sums are CTA-local.  Otherwise (`gsum` set) every CTA adds its partial sums to gsum, the grid meets
// at an arrival counter (cooperative launch: all tiles are resident, so the grid must not exceed the SM count), and -
// data parallel - the CTA that arrives last pushes this rank's sums into every peer's exchange buffer over NVLink and
// raises the flags all CTAs of all ranks wait on: the SyncBN all-reduce happens INSIDE the GEMM, between its mainloop
// and its second epilogue pass, summed in rank order (bit-identical statistics on every rank).
struct FusedTrain {
  const void* sc = nullptr;               // train::StepScalars (device)
  const float* gamma = nullptr; const float* beta = nullptr;
  float* mean = nullptr; float* rstd = nullptr;            // [N] written by mode 3, read by mode 4
  float* mov_mean = nullptr; float* mov_var = nullptr;     // mode 3
  float* h = nullptr; void* hb = nullptr; uint8_t* mask = nullptr; const uint8_t* mask_in = nullptr; const float* hres = nullptr;   // mode 3, [M][N]
  const float* z = nullptr; float* dh_out = nullptr; void* dzb = nullptr;                                                       // mode 4, [M][N]
  float* ggamma = nullptr; float* gbeta = nullptr; float* gbias = nullptr;                                                      // mode 4, [N]
  int has_bn = 0, dropout = 0, layer = 0;
  float invB = 1.f;                       // 1 / GLOBAL batch
  double* gsum = nullptr;                 // [2][N] doubles, zero when the kernel starts (grid-synchronised form)
  unsigned* gcount = nullptr;             // [2]: arrival counter, completion flag; zero when the kernel starts
  const void* peers = nullptr;            // device p2p::Peers (world > 1)
  int rank = 0, world = 1;
  long long row0 = 0;                     // global row of this rank's row 0 (dropout counters use global rows)
  double* xsum = nullptr;                 // optional scalar summed over the ranks on the same exchange (the step's loss sum)
  float pg_scale = 1.f;                   // 1 / world: gradients every rank computes in full (dgamma, dbeta, bias) are
                                          // pre-divided so that the flat gradient all-reduce (a sum) restores them once
};
// tcgen05 GEMM (tc_gemm.cu): C[M,N] (+)= alpha * A B^T-form product of bf16 operands, fp32 result.
struct GemmArgs {
  int M = 0, N = 0, K = 0;
  const void* A = nullptr; int lda = 0; int a_mn = 0;   // a_mn ? [K][M] : [M][K]  (bf16)
  const void* B = nullptr; int ldb = 0; int b_mn = 0;   // b_mn ? [K][N] : [N][K]  (bf16)
  float* C = nullptr; int ldc = 0;
  const float* bias = nullptr;        // [N]
  const float* res = nullptr; int ldres = 0;
  const float* alpha_dev = nullptr;   // optional device scalar multiplied into alpha
  float alpha = 1.f;
  int split_k = 0;                    // split K over gridDim.z, fp32 atomics into C (C must hold the addend, e.g. zeros)
  int accumulate = 0;                 // C += (atomics) even when unsplit
  double* colsum = nullptr;           // optional [2][N] (+=): column sums of the result and of its square
  // bf16 result instead of C (inference layers): out = bf16(relu?(.)), then out = bf16(out + res_bf16)
  void* out_bf16 = nullptr; int ld_out_bf16 = 0;
  const void* res_bf16 = nullptr; int ld_res_bf16 = 0;
  int relu = 0;
  // fp16 operands (P3D_MODE_FP16 inference): A, B, out_bf16 and res_bf16 hold fp16; plain fp32 store or 16-bit output only
  int f16 = 0;
  // programmatic dependent launch: the kernel may start before its stream predecessor has finished; B (weights)
  // must not depend on that predecessor - its first tiles are fetched ahead of the dependency wait
  int pdl = 0;
  void* dbg = nullptr;                // diagnostics: [ctas][8] globaltimer stamps
  int fused_mode = 0;                 // 0, or 3 / 4: fused training epilogue (unsplit K; every tile resident at once)
  FusedTrain fused;
  // Segment schedule (bf16x3; 0 = off): A and B are split pairs, each row the hi segment then the lo segment from
  // column seg_a / seg_b (a multiple of 64) of the operand's contiguous dimension.  K-major: seg >= K rounded up to 64,
  // the columns between K and the lo segment must be zero.  MN-major: seg >= M (A) or N (B).  The K loop makes three
  // passes: A.hi B.hi + A.lo B.hi + A.hi B.lo; split K and the fp32 reduction epilogue are allowed.
  int seg_a = 0, seg_b = 0;
  // split-pair result (with the segment schedule): r = relu?(acc + bias) (+ res, fp32) -> C when C is set (may equal
  // res: in place), and bf16(r) | bf16(r - bf16(r)) -> out_bf16 columns n | out_lo + n
  int out_lo = 0;
};
// A planned GEMM: tensor maps + kernel parameters, built once (host cost of two cuTensorMapEncodeTiled calls)
// and launched many times while the operand pointers/shapes stay the same.
struct alignas(64) GemmPlan { unsigned char blob[1024]; int valid = 0; };
int plan(const GemmArgs& g, GemmPlan* out);
int launch(const GemmPlan& pl, cudaStream_t st);
int gemm(const GemmArgs& g, cudaStream_t st);
bool fused_fits(int M, int N, int K, int num_sms);   // can the fused training epilogues serve an M x N layer (all tiles resident)?
}  // namespace tcg
int sqerr_accumulate(const float* y, const float* t, size_t n, double* acc, cudaStream_t st);
int l2persist_acquire(int dev, size_t bytes);                // mlp_tc.cu: persisting-L2 set-aside for the fused inference kernel
int l2persist_release(int dev);                              // ... handed back (training steps want the whole L2)
bool l2persist_held(int dev, size_t bytes);                  // ... currently set aside, at least `bytes`
int mark_model_work(p3d_model* m, cudaStream_t st);          // record ev_done on st
int order_after_model_work(p3d_model* m, cudaStream_t st);   // st waits for the last recorded ev_done
// CUDA-graph capture (include/p3d.h, "CUDA graphs"): a call on a capturing stream may not allocate, free or
// synchronise.  capturing(st): st is capturing now.  refuse_in_capture(st, what): P3D_OK when st is not capturing,
// otherwise P3D_ERR_STATE with a message that names `what` and the warm-up rule.
bool capturing(cudaStream_t st);
int refuse_in_capture(cudaStream_t st, const char* what);
// a growable scratch buffer is being replaced by a larger one: freed at once while no graph can hold its address,
// kept until p3d_model_destroy once the model has been captured
void retire(p3d_model* m, void* p);
// new capacity (rows) of a growable scratch buffer that holds `cap` rows and must hold `need`: exactly `need` while
// superseded buffers are freed at once; once they are kept, at least twice the old capacity, so that what is kept
// stays below the live buffer's size
int64_t grown_cap(const p3d_model* m, int64_t cap, int64_t need);

// Exchange tags of the whole-chip inference kernels (p3d_model::xchg: [0] epoch, [32] arrival counter).  Every thread
// loads the epoch at kernel entry (xchg_tag: tag = epoch + 1, never 0).  Once every thread of a CTA has used its tag
// (compared it in the first gather), one thread arrives (xchg_arrive); the CTA that arrives last resets the counter and advances the epoch
// (xchg_advance).  All CTAs have read the epoch by then, and the next launch on the stream sees the new value, so no
// two launches - eager calls or graph replays, in any order - share a tag.
__device__ __forceinline__ unsigned xchg_tag(const unsigned* xchg) {
  unsigned e;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(e) : "l"(xchg) : "memory");
  return e + 1u;
}
// The compiler aggregates the arrival per warp and waits for its result at once: one contended L2 round trip for the
// arriving warp, so the kernels arrive just before a gather, where the warp waits for other CTAs' outputs anyway.
__device__ __forceinline__ unsigned xchg_arrive(unsigned* xchg) { return atomicAdd(xchg + 32, 1u); }
__device__ __forceinline__ void xchg_advance(unsigned* xchg, unsigned tag) {
  asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(xchg + 32), "r"(0u) : "memory");
  asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(xchg), "r"(tag == 0xFFFFFFFFu ? 0u : tag) : "memory");
}

}  // namespace p3d

struct p3d_model {
  p3d_cfg cfg;
  int out_size = 48;
  int L = 1024;
  std::vector<p3d::Layer> layers;
  std::vector<p3d::NamedParam> params;
  // flat parameter storage
  size_t n_train = 0, n_moving = 0;
  float* theta = nullptr;
  float* grad = nullptr;
  float* adam_m = nullptr;
  float* adam_v = nullptr;
  float* moving = nullptr;
  int64_t global_step = 0;
  // inference pack
  bool pack_valid = false;
  int rows_total = 0;      // sum of N over layers
  int kpad = 0;            // row pitch (elements) of wt_bf16 = max(L rounded up to 8, 64)
  __nv_bfloat16* wt_bf16 = nullptr;  // [rows_total][kpad], K-major, BN+clip folded; fp16 bits in P3D_MODE_FP16
  float* bias_fold = nullptr;        // [rows_total]
  float* wfold = nullptr;            // fp32 folded [K,N] per layer, concatenated
  double* norm2 = nullptr;           // [nlayers] ||W||_F^2
  // forward scratch
  int num_sms = 0;
  __nv_bfloat16* act_scratch = nullptr;  // [2][grid*128][L] bf16 (tcgen05 path)
  int act_grid = 0;
  __nv_bfloat16* xb = nullptr;           // packed input [cap][64]
  int64_t xb_cap = 0;
  // layered (one tcgen05 GEMM per layer) forward for small/medium batches: plans cached per batch size
  std::vector<p3d::tcg::GemmPlan> lay_plans;
  int64_t lay_B = -1;
  const void* lay_y = nullptr;
  const void* lay_x = nullptr;
  __nv_bfloat16* lay_act = nullptr;      // [2][lay_cap][L] bf16
  int64_t lay_cap = 0;
  unsigned long long* lat_counter = nullptr;   // grid-barrier counter of the latency kernel (monotonic), [8..] stamps
  unsigned long long lat_base = 0;
  void* lat_act = nullptr;               // 1 .. 8 poses whole-chip kernel (mlp_simt.cu): exchange words {value, tag}, 8 MB
  void* mid_act = nullptr;               // 9 .. 64 poses whole-chip kernel (mlp_mid.cu): exchange words {bf16 pair, tag} [8][64][512]
  // Exchange tags of both whole-chip kernels, in device memory: [0] epoch, [32] arrival counter.  Every CTA of a launch
  // reads the epoch at entry (tag = epoch + 1, never 0); the last CTA to finish resets the counter and advances the
  // epoch, so every launch - eager or a graph replay - uses a tag no earlier launch used.
  unsigned* xchg = nullptr;
  float* f32_a = nullptr;                // fp32-path activations [2][cap][L]
  int64_t f32_cap = 0;
  // bf16x3 mode (mlp_layered.cu forward_split): split pairs, every row [hi segment | lo segment], segment x3_seg =
  // L rounded up to 64 columns, padding zero
  int x3_seg = 0;
  __nv_bfloat16* wt_x3 = nullptr;        // folded W'^T split [rows_total][2 x3_seg], allocated at model creation
  __nv_bfloat16* x3_in = nullptr;        // input split [x3_cap][128]: hi columns 0..31, lo 64..95
  __nv_bfloat16* x3_act = nullptr;       // hidden activations split, [2][x3_cap][2 x3_seg]
  float* x3_res = nullptr;               // fp32 block input of the residual stream [x3_cap][L] (residual models)
  int64_t x3_cap = 0;
  struct X3Plans { int64_t rows = -1; const void* y = nullptr; std::vector<p3d::tcg::GemmPlan> pl; };
  X3Plans x3_plans[2];                   // full row chunks, the last (partial) chunk
  // growable scratch that a captured graph may still address (retire()): freed by p3d_model_destroy
  bool captured = false;                 // a call of this model has run on a capturing stream
  std::vector<void*> retired;
  // host-step pipeline
  cudaStream_t pipe_streams[3] = {nullptr, nullptr, nullptr};
  float* pipe_x[3] = {nullptr, nullptr, nullptr};
  float* pipe_t[3] = {nullptr, nullptr, nullptr};
  float* pipe_y[3] = {nullptr, nullptr, nullptr};
  double* pipe_loss = nullptr;                        // device accumulator (sum of squared errors)
  int64_t pipe_chunk = 0;
  cudaEvent_t pipe_ev[9] = {};                        // in / compute / out events of the three pipeline slots (cached)
  // Ordering between the caller's stream and the library's private streams: every asynchronous operation that writes
  // model state (training steps, epochs, forwards: weights, moving statistics, packed weights, scratch) records
  // `ev_done` on its stream; the host-buffer step and the realtime frame, which run on private non-blocking streams,
  // wait for it before they fold weights or launch (p3d::order_after_model_work).
  cudaEvent_t ev_done = nullptr;
  bool ev_done_recorded = false;
  // training
  int train_matmul = P3D_TRAIN_MATMUL_DEFAULT;   // p3d_model_set_train_matmul
  p3d::TrainWorkspace tw;
  void* nccl_comm = nullptr;
  int rank = 0, world = 1;
  void* p2p_state = nullptr;          // peer-memory exchange buffers of the small all-reduces (p2p.cu)
  // data parallel: what the gradient exchange of the current step gathers on the way (set by the step, read by p2p)
  const float* dp_y = nullptr; long long dp_rows = 0, dp_row0 = 0, dp_Bg = 0;
  bool dp_y_gathered = false;         // the last step left the global outputs in the exchange buffer
};
