// C ABI of libp3d.so (see include/p3d.h): model lifetime, variables by TF name, forward dispatch,
// the host-buffer evaluation step, misc.
#include <cstdlib>
#include <cstring>

#include "common.cuh"

namespace p3d {

static thread_local char g_err[1024] = "";
static std::atomic<long long>* launch_counter() {
  static std::atomic<long long> c{0};
  return &c;
}
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
void count_launch(int n) { launch_counter()->fetch_add(n); }
long long launch_count_now() { return launch_counter()->load(); }

namespace prep { int prepare(p3d_model*, cudaStream_t); int pack_input(const float*, __nv_bfloat16*, int64_t, bool, cudaStream_t); }
namespace tc { int forward_bf16(p3d_model*, const __nv_bfloat16*, float*, int64_t, cudaStream_t);
               int debug_umma_gemm(const void*, const void*, float*, int, int, cudaStream_t); }
namespace simt { int forward_fp32(p3d_model*, const float*, float*, int64_t, cudaStream_t);
                 int forward_small(p3d_model*, const float*, float*, int64_t, cudaStream_t);
                 int forward_latency(p3d_model*, const float*, float*, int64_t, cudaStream_t);
                 int forward_latency_grid(p3d_model*, const float*, float*, int, cudaStream_t);
                 int forward_latency_cluster(p3d_model*, const float*, float*, cudaStream_t); }
namespace mid { int forward(p3d_model*, const float*, float*, int, cudaStream_t); }
namespace tcg { int mma_rate(int, int, long long*, cudaStream_t); }
namespace layered { int forward(p3d_model*, const __nv_bfloat16*, float*, int64_t, cudaStream_t);
                    int forward_split(p3d_model*, const float*, float*, int64_t, cudaStream_t); }
namespace train { void free_workspace(p3d_model*); }

constexpr int kSmallBatchMax = 16;   // rows served by the latency (GEMV) path

__global__ void fill_kernel(float* p, size_t n, float v) {
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<size_t>(gridDim.x) * blockDim.x) p[i] = v;
}

// Streaming probe: reads n_read float4 and writes n_write float4 with fully coalesced streaming accesses - the HBM ceiling
// for a kernel with that read:write mix (the copy figure of MEASURED_PEAKS.json is 1:1; preprocessing writes 3.3x what
// it reads, evaluation only reads).
__global__ void stream_mix_kernel(const float4* __restrict__ src, float4* __restrict__ dst, long long n_read, long long n_write) {
  const long long n = n_read > n_write ? n_read : n_write;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n; i += static_cast<long long>(gridDim.x) * blockDim.x) {
    if (i < n_read) { const float4 v = __ldcs(src + i); acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w; }
    if (i < n_write) __stcs(dst + i, acc);
  }
  if (n_write == 0 && acc.x == 1.2345e38f) dst[0] = acc;      // keep the loads alive in the read-only case
}

// sum((y-t)^2) into a double accumulator
__global__ void sqerr_kernel(const float* __restrict__ y, const float* __restrict__ t, size_t n, double* __restrict__ acc) {
  double s = 0.0;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const float d = y[i] - t[i];
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
__global__ void finish_mse_kernel(const double* acc, double denom, float* loss) { *loss = static_cast<float>(*acc / denom); }

static int fill(float* p, size_t n, float v) {
  if (n == 0) return P3D_OK;
  int blocks = static_cast<int>((n + 255) / 256);
  if (blocks > 1024) blocks = 1024;
  fill_kernel<<<blocks, 256>>>(p, n, v);
  P3D_LAUNCH_CHECK();
  return P3D_OK;
}

int sqerr_accumulate(const float* y, const float* t, size_t n, double* acc, cudaStream_t st) {
  int blocks = static_cast<int>((n + 256 * 8 - 1) / (256 * 8));
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (blocks < 1) blocks = 1;
  sqerr_kernel<<<blocks, 256, 0, st>>>(y, t, n, acc);
  P3D_LAUNCH_CHECK();
  return P3D_OK;
}

namespace prof {
static bool g_on = false;
static std::vector<std::pair<cudaEvent_t, cudaEvent_t>> g_pending;
static double g_ms = 0.0;
static long long g_n = 0;
bool enabled() { return g_on; }
void begin(cudaStream_t st, cudaEvent_t* e0, cudaEvent_t* e1) {
  if (cudaEventCreate(e0) != cudaSuccess || cudaEventCreate(e1) != cudaSuccess) { *e0 = *e1 = nullptr; return; }
  cudaEventRecord(*e0, st);
}
void end(cudaStream_t st, cudaEvent_t e0, cudaEvent_t e1) {
  cudaEventRecord(e1, st);
  g_pending.emplace_back(e0, e1);
}
static void drain() {
  for (auto& pr : g_pending) {
    float ms = 0.f;
    if (cudaEventSynchronize(pr.second) == cudaSuccess && cudaEventElapsedTime(&ms, pr.first, pr.second) == cudaSuccess) {
      g_ms += ms; g_n += 1;
    }
    cudaEventDestroy(pr.first); cudaEventDestroy(pr.second);
  }
  g_pending.clear();
}
}  // namespace prof

bool capturing(cudaStream_t st) {
  cudaStreamCaptureStatus s = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &s) != cudaSuccess) {     // e.g. the legacy stream while another stream captures
    cudaGetLastError();
    return true;
  }
  return s != cudaStreamCaptureStatusNone;
}
int refuse_in_capture(cudaStream_t st, const char* what) {
  if (!capturing(st)) return P3D_OK;
  set_error("%s cannot happen inside a CUDA graph capture: warm up first - run the same call (same batch size) once "
            "outside the capture", what);
  return P3D_ERR_STATE;
}
void retire(p3d_model* m, void* p) {
  if (!p) return;
  if (m->captured) m->retired.push_back(p);
  else cudaFree(p);
}

int64_t grown_cap(const p3d_model* m, int64_t cap, int64_t need) {
  return (m->captured && 2 * cap > need) ? 2 * cap : need;
}

int mark_model_work(p3d_model* m, cudaStream_t st) {
  if (!m->ev_done) P3D_CUDA(cudaEventCreateWithFlags(&m->ev_done, cudaEventDisableTiming));
  if (capturing(st)) {
    // an external event-record node: every replay of the graph records ev_done, and the event itself never becomes
    // part of the capture (a plain record would leave it captured, and the next wait on it would be refused)
    m->captured = true;
    P3D_CUDA(cudaEventRecordWithFlags(m->ev_done, st, cudaEventRecordExternal));
  } else {
    P3D_CUDA(cudaEventRecord(m->ev_done, st));
  }
  m->ev_done_recorded = true;
  return P3D_OK;
}
int order_after_model_work(p3d_model* m, cudaStream_t st) {
  if (m->ev_done_recorded) P3D_CUDA(cudaStreamWaitEvent(st, m->ev_done, 0));
  return P3D_OK;
}

static NamedParam* find_param(p3d_model* m, const char* name) {
  for (auto& p : m->params)
    if (p.name == name) return &p;
  return nullptr;
}

}  // namespace p3d

using namespace p3d;

extern "C" {

const char* p3d_last_error(void) { return g_err; }
int p3d_version(void) { return 100; }
int64_t p3d_launch_count(void) { return launch_counter()->load(); }

int p3d_profile_enable(int on) {
  prof::drain();
  prof::g_on = on != 0;
  prof::g_ms = 0.0; prof::g_n = 0;
  return P3D_OK;
}
int p3d_profile_read(double* ms_total, int64_t* launches) {
  prof::drain();
  if (ms_total) *ms_total = prof::g_ms;
  if (launches) *launches = prof::g_n;
  return P3D_OK;
}

int p3d_host_alloc(void** out, size_t bytes) {
  P3D_REQUIRE(out, "host_alloc: null out");
  P3D_CUDA(cudaHostAlloc(out, bytes, cudaHostAllocPortable));
  return P3D_OK;
}
int p3d_host_free(void* p) {
  P3D_CUDA(cudaFreeHost(p));
  return P3D_OK;
}

int p3d_model_create(const p3d_cfg* cfg, p3d_model** out) {
  P3D_REQUIRE(cfg && out, "model_create: null argument");
  P3D_REQUIRE(cfg->linear_size >= 16 && cfg->linear_size % 4 == 0, "linear_size must be a positive multiple of 4");
  P3D_REQUIRE(cfg->num_layers >= 0 && cfg->num_layers <= 64, "num_layers out of range");
  P3D_REQUIRE(cfg->mode == P3D_MODE_BF16 || cfg->mode == P3D_MODE_FP32 || cfg->mode == P3D_MODE_BF16X3 || cfg->mode == P3D_MODE_FP16,
              "unknown mode %d", cfg->mode);
  int ndev = 0;
  P3D_CUDA(cudaGetDeviceCount(&ndev));
  P3D_REQUIRE(cfg->device >= 0 && cfg->device < ndev, "device %d not present (%d devices)", cfg->device, ndev);
  P3D_CUDA(cudaSetDevice(cfg->device));
  cudaDeviceProp prop;
  P3D_CUDA(cudaGetDeviceProperties(&prop, cfg->device));
  if (prop.major != 10) {
    set_error("libp3d is built for sm_100a only; device %d is sm_%d%d", cfg->device, prop.major, prop.minor);
    return P3D_ERR_CUDA;
  }
  p3d_model* m = new p3d_model();
  m->cfg = *cfg;
  m->L = cfg->linear_size;
  m->out_size = cfg->predict_14 ? 42 : 48;
  m->num_sms = prop.multiProcessorCount;
  const int L = m->L;
  const int nlay = 2 * cfg->num_layers + 2;
  m->layers.resize(nlay);
  // layer table + TF names (src/linear_model.py:106-107,121-122,176-193)
  for (int l = 0; l < nlay; ++l) {
    Layer& ly = m->layers[l];
    ly.K = (l == 0) ? kIn : L;
    ly.N = (l == nlay - 1) ? m->out_size : L;
    ly.hidden = (l != nlay - 1);
    ly.has_bn = ly.hidden && cfg->batch_norm;
    char buf[128];
    if (l == 0) { ly.wname = "linear_model/w1"; ly.bname = "linear_model/b1"; ly.bnscope = "linear_model/batch_normalization"; }
    else if (l == nlay - 1) { ly.wname = "linear_model/w4"; ly.bname = "linear_model/b4"; }
    else {
      const int blk = (l - 1) / 2, which = (l - 1) % 2;   // 0 -> w2/b2/bn1, 1 -> w3/b3/bn2
      snprintf(buf, sizeof(buf), "linear_model/two_linear_%d/w%d_%d", blk, which + 2, blk); ly.wname = buf;
      snprintf(buf, sizeof(buf), "linear_model/two_linear_%d/b%d_%d", blk, which + 2, blk); ly.bname = buf;
      snprintf(buf, sizeof(buf), "linear_model/two_linear_%d/batch_normalization%d%d", blk, which + 1, blk); ly.bnscope = buf;
    }
  }
  // flat layout: [all W][b, gamma, beta per layer]
  size_t off = 0, wf = 0;
  int row = 0;
  for (auto& ly : m->layers) {
    ly.off_w = off; off += static_cast<size_t>(ly.K) * ly.N;
    ly.off_wfold = wf; wf += static_cast<size_t>(ly.K) * ly.N;
    ly.row_off = row; row += ly.N;
  }
  const size_t n_w = off;
  size_t mo = 0;
  for (auto& ly : m->layers) {
    ly.off_b = off; off += ly.N;
    if (ly.has_bn) {
      ly.off_gamma = off; off += ly.N;
      ly.off_beta = off; off += ly.N;
      ly.off_mm = mo; mo += ly.N;
      ly.off_mv = mo; mo += ly.N;
    }
  }
  (void)n_w;
  m->n_train = off;
  m->n_moving = mo;
  m->rows_total = row + 16;   // slack so the padded output rows exist (zero)
  m->kpad = L < 64 ? 64 : (L + 7) / 8 * 8;   // rows start 16-byte aligned: the small-batch kernel loads 8 weights at a time
  auto fail = [&](int rc) { p3d_model_destroy(m); return rc; };
#define P3D_ALLOC(ptr, bytes)                                                                  \
  do {                                                                                         \
    cudaError_t e__ = cudaMalloc(reinterpret_cast<void**>(&(ptr)), (bytes));                   \
    if (e__ != cudaSuccess) { set_error("cudaMalloc(%zu) failed: %s", (size_t)(bytes), cudaGetErrorString(e__)); return fail(P3D_ERR_CUDA); } \
    cudaMemset((ptr), 0, (bytes));                                                             \
  } while (0)
  P3D_ALLOC(m->theta, sizeof(float) * m->n_train);
  P3D_ALLOC(m->grad, sizeof(float) * m->n_train);
  P3D_ALLOC(m->adam_m, sizeof(float) * m->n_train);
  P3D_ALLOC(m->adam_v, sizeof(float) * m->n_train);
  P3D_ALLOC(m->moving, sizeof(float) * (m->n_moving ? m->n_moving : 1));
  P3D_ALLOC(m->wt_bf16, sizeof(__nv_bfloat16) * static_cast<size_t>(m->rows_total) * m->kpad);
  P3D_ALLOC(m->bias_fold, sizeof(float) * m->rows_total);
  P3D_ALLOC(m->wfold, sizeof(float) * wf);
  P3D_ALLOC(m->norm2, sizeof(double) * nlay);
  P3D_ALLOC(m->pipe_loss, sizeof(double));
  // fixed-size forward scratch exists from the start, so that no forward has to allocate it (a graph capture could not)
  P3D_ALLOC(m->lat_counter, sizeof(unsigned long long) * 32);
  P3D_ALLOC(m->xchg, sizeof(unsigned) * 64);
  if (L == 1024 && (cfg->mode == P3D_MODE_BF16 || cfg->mode == P3D_MODE_FP16)) {   // the whole-chip kernels' exchange buffers (mlp_simt.cu, mlp_mid.cu)
    P3D_ALLOC(m->lat_act, sizeof(uint2) * 1024 * 8 * 128);
    P3D_ALLOC(m->mid_act, sizeof(unsigned long long) * 8 * 64 * 512);
  }
  if (cfg->mode == P3D_MODE_BF16X3 && L % 8 == 0) {    // the split weight pair of the bf16x3 GEMMs (zeroed: padding)
    m->x3_seg = (L + 63) / 64 * 64;
    P3D_ALLOC(m->wt_x3, sizeof(__nv_bfloat16) * static_cast<size_t>(m->rows_total) * 2 * m->x3_seg);
  }
#undef P3D_ALLOC
  // TF default BN state: gamma 1, beta 0, moving_mean 0, moving_variance 1
  for (auto& ly : m->layers) {
    if (!ly.has_bn) continue;
    if (fill(m->theta + ly.off_gamma, ly.N, 1.f) != P3D_OK) return fail(P3D_ERR_CUDA);
    if (fill(m->moving + ly.off_mv, ly.N, 1.f) != P3D_OK) return fail(P3D_ERR_CUDA);
  }
  for (auto& ly : m->layers) {
    m->params.push_back({ly.wname, m->theta + ly.off_w, static_cast<size_t>(ly.K) * ly.N, true});
    m->params.push_back({ly.bname, m->theta + ly.off_b, static_cast<size_t>(ly.N), true});
    if (ly.has_bn) {
      m->params.push_back({ly.bnscope + "/gamma", m->theta + ly.off_gamma, static_cast<size_t>(ly.N), true});
      m->params.push_back({ly.bnscope + "/beta", m->theta + ly.off_beta, static_cast<size_t>(ly.N), true});
      m->params.push_back({ly.bnscope + "/moving_mean", m->moving + ly.off_mm, static_cast<size_t>(ly.N), true});
      m->params.push_back({ly.bnscope + "/moving_variance", m->moving + ly.off_mv, static_cast<size_t>(ly.N), true});
    }
  }
  // Adam slots (tf.train.AdamOptimizer slot names "Adam" = m, "Adam_1" = v)
  const size_t nvars = m->params.size();
  for (size_t i = 0; i < nvars; ++i) {
    const NamedParam p = m->params[i];
    if (p.ptr < m->theta || p.ptr >= m->theta + m->n_train) continue;
    const size_t o = p.ptr - m->theta;
    m->params.push_back({p.name + "/Adam", m->adam_m + o, p.numel, false});
    m->params.push_back({p.name + "/Adam_1", m->adam_v + o, p.numel, false});
    // last computed gradient (what the reference exposes as model.gradients, src/linear_model.py:143-144)
    m->params.push_back({p.name + "/gradient", m->grad + o, p.numel, false});
  }
  if (cudaDeviceSynchronize() != cudaSuccess) { set_error("model_create: device error"); return fail(P3D_ERR_CUDA); }
  *out = m;
  return P3D_OK;
}

void p3d_model_destroy(p3d_model* m) {
  if (!m) return;
  cudaSetDevice(m->cfg.device);
  cudaDeviceSynchronize();
  train::free_workspace(m);
  cudaFree(m->theta); cudaFree(m->grad); cudaFree(m->adam_m); cudaFree(m->adam_v); cudaFree(m->moving);
  cudaFree(m->wt_bf16); cudaFree(m->bias_fold); cudaFree(m->wfold); cudaFree(m->norm2); cudaFree(m->pipe_loss);
  cudaFree(m->act_scratch); cudaFree(m->xb); cudaFree(m->f32_a); cudaFree(m->lat_counter); cudaFree(m->lay_act); cudaFree(m->lat_act); cudaFree(m->mid_act);
  cudaFree(m->xchg);
  cudaFree(m->wt_x3); cudaFree(m->x3_in); cudaFree(m->x3_act); cudaFree(m->x3_res);
  for (void* p : m->retired) cudaFree(p);
  if (m->ev_done) cudaEventDestroy(m->ev_done);
  for (auto& e : m->pipe_ev) if (e) cudaEventDestroy(e);
  for (int i = 0; i < 3; ++i) {
    if (m->pipe_streams[i]) cudaStreamDestroy(m->pipe_streams[i]);
    cudaFree(m->pipe_x[i]); cudaFree(m->pipe_t[i]); cudaFree(m->pipe_y[i]);
  }
  delete m;
}

int p3d_model_param_count(p3d_model* m) { return m ? static_cast<int>(m->params.size()) + 1 : 0; }

int p3d_model_param_name(p3d_model* m, int index, char* out, size_t cap, size_t* numel) {
  P3D_REQUIRE(m && out && cap > 0, "param_name: null argument");
  const int n = static_cast<int>(m->params.size());
  P3D_REQUIRE(index >= 0 && index <= n, "param_name: index %d out of range", index);
  if (index == n) { snprintf(out, cap, "global_step"); if (numel) *numel = 1; return P3D_OK; }
  snprintf(out, cap, "%s", m->params[index].name.c_str());
  if (numel) *numel = m->params[index].numel;
  return P3D_OK;
}

int p3d_model_set_param_host(p3d_model* m, const char* name, const float* host, size_t n) {
  P3D_REQUIRE(m && name && host, "set_param: null argument");
  P3D_CUDA(cudaSetDevice(m->cfg.device));
  if (strcmp(name, "global_step") == 0) {
    P3D_REQUIRE(n == 1, "global_step is a scalar");
    m->global_step = static_cast<int64_t>(host[0]);
    return P3D_OK;
  }
  if (strcmp(name, "learning_rate") == 0) {   // the base rate variable (src/linear_model.py:86); not enumerated
    P3D_REQUIRE(n == 1, "learning_rate is a scalar");
    m->cfg.learning_rate = host[0];
    return P3D_OK;
  }
  NamedParam* p = find_param(m, name);
  P3D_REQUIRE(p, "unknown variable '%s'", name);
  P3D_REQUIRE(p->numel == n, "variable '%s' has %zu elements, got %zu", name, p->numel, n);
  P3D_CUDA(cudaMemcpy(p->ptr, host, sizeof(float) * n, cudaMemcpyHostToDevice));
  if (p->affects_inference) m->pack_valid = false;
  return P3D_OK;
}

int p3d_model_get_param_host(p3d_model* m, const char* name, float* host, size_t n) {
  P3D_REQUIRE(m && name && host, "get_param: null argument");
  P3D_CUDA(cudaSetDevice(m->cfg.device));
  if (strcmp(name, "global_step") == 0) {
    P3D_REQUIRE(n == 1, "global_step is a scalar");
    host[0] = static_cast<float>(m->global_step);
    return P3D_OK;
  }
  if (strcmp(name, "learning_rate") == 0) {
    P3D_REQUIRE(n == 1, "learning_rate is a scalar");
    host[0] = m->cfg.learning_rate;
    return P3D_OK;
  }
  NamedParam* p = find_param(m, name);
  P3D_REQUIRE(p, "unknown variable '%s'", name);
  P3D_REQUIRE(p->numel == n, "variable '%s' has %zu elements, got %zu", name, p->numel, n);
  P3D_CUDA(cudaDeviceSynchronize());
  P3D_CUDA(cudaMemcpy(host, p->ptr, sizeof(float) * n, cudaMemcpyDeviceToHost));
  return P3D_OK;
}

int64_t p3d_model_global_step(p3d_model* m) { return m ? m->global_step : -1; }

int p3d_model_prepare_inference(p3d_model* m, void* stream) {
  P3D_REQUIRE(m, "prepare_inference: null model");
  P3D_CUDA(cudaSetDevice(m->cfg.device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  // the fold rewrites the packed weights in place (graphs captured earlier read the new ones); captured itself, it
  // would leave pack_valid set before any replay had computed it
  if (capturing(st)) {
    set_error("prepare_inference cannot be captured into a CUDA graph: call it outside the capture");
    return P3D_ERR_STATE;
  }
  P3D_TRY(prep::prepare(m, st));
  return mark_model_work(m, st);
}

// packed input buffer [cap][64] bf16 of the tensor-core paths
static int ensure_xb(p3d_model* m, int64_t B, cudaStream_t st) {
  if (m->xb_cap < B) {
    P3D_TRY(refuse_in_capture(st, "forward: growing the packed-input buffer"));
    const int64_t cap = grown_cap(m, m->xb_cap, B < 1024 ? 1024 : B);
    retire(m, m->xb);
    m->xb = nullptr; m->xb_cap = 0;
    P3D_CUDA(cudaMalloc(&m->xb, sizeof(__nv_bfloat16) * 64ull * cap));
    m->xb_cap = cap;
  }
  return P3D_OK;
}
// the tensor-core forward from the packed input m->xb
static int forward_packed(p3d_model* m, float* y, int64_t B, cudaStream_t st) {
  // One tile of the fused persistent kernel takes ~100 us to walk all layers (a single SM pair streams every
  // weight); below the crossover (measured: 77 vs 97 us at 4096 poses, 135 vs 101 us at 8192) the per-layer GEMMs,
  // which split each layer over N, are faster.
  static const int64_t layered_max = [] { const char* e = getenv("P3D_LAYERED_MAX"); return e ? atoll(e) : 6144LL; }();
  const bool fused_ok = (m->L % 256) == 0 && m->L <= 4096;
  if (!fused_ok || B < layered_max) return layered::forward(m, m->xb, y, B, st);
  return tc::forward_bf16(m, m->xb, y, B, st);
}

static int forward_on(p3d_model* m, const float* x, float* y, int64_t B, cudaStream_t st) {
  if (!m->pack_valid) {
    if (capturing(st)) {
      set_error("forward: the variables changed since the last weight fold, and the fold cannot be captured into a "
                "CUDA graph: call prepare_inference outside the capture first");
      return P3D_ERR_STATE;
    }
    P3D_TRY(prep::prepare(m, st));
  }
  if (m->cfg.mode == P3D_MODE_FP32) return simt::forward_fp32(m, x, y, B, st);
  if (m->cfg.mode == P3D_MODE_BF16X3) {
    // widths no tensor-core tiling covers: the FFMA chain, which keeps the same precision contract
    if ((m->L % 8) != 0) return simt::forward_fp32(m, x, y, B, st);
    return layered::forward_split(m, x, y, B, st);
  }
  const int L = m->L;
  // fp16 mode: bf16 mode's paths on fp16 operands; widths no tensor-core tiling covers take the FFMA chain, whose
  // contract is stricter (the bf16-only forward_small is not ported)
  if (m->cfg.mode == P3D_MODE_FP16 && (L % 8) != 0) return simt::forward_fp32(m, x, y, B, st);
  if (B == 1 && L == 1024) {                            // single pose: whole-chip kernel (or the 16-CTA cluster kernel), one launch
    const int rc = simt::forward_latency_cluster(m, x, y, st);
    if (rc <= 0) return rc;                              // 1 = not schedulable here -> fall through
  }
  if (B >= 2 && B <= 8 && L == 1024) {                  // a handful of poses: the same whole-chip kernel, fp32 activations
    const int rc = simt::forward_latency_grid(m, x, y, static_cast<int>(B), st);
    if (rc <= 0) return rc;
  }
  if (B >= 9 && B <= 64 && L == 1024) {                 // the reference's batch size: one whole-chip launch, mma.sync tiles, bf16 activations
    const int rc = mid::forward(m, x, y, static_cast<int>(B), st);
    if (rc <= 0) return rc;
  }
  if ((L % 8) != 0) {                                    // widths no tensor-core tiling covers
    if (B <= kSmallBatchMax) return simt::forward_small(m, x, y, B, st);
    return simt::forward_fp32(m, x, y, B, st);
  }
  P3D_TRY(ensure_xb(m, B, st));
  P3D_TRY(prep::pack_input(x, m->xb, B, m->cfg.mode == P3D_MODE_FP16, st));
  return forward_packed(m, y, B, st);
}

int p3d_model_forward(p3d_model* m, const float* x, float* y, int64_t B, void* stream) {
  P3D_REQUIRE(m && x && y, "forward: null argument");
  P3D_REQUIRE(B >= 0, "forward: negative batch");
  if (B == 0) return P3D_OK;
  P3D_CUDA(cudaSetDevice(m->cfg.device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  P3D_TRY(forward_on(m, x, y, B, st));
  return mark_model_work(m, st);     // the host-buffer step / realtime frame (private streams) order themselves behind this
}

int p3d_model_mse(p3d_model* m, const float* y, const float* t, int64_t B, float* loss, void* stream) {
  P3D_REQUIRE(m && y && t && loss && B > 0, "mse: bad argument");
  P3D_CUDA(cudaSetDevice(m->cfg.device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  P3D_CUDA(cudaMemsetAsync(m->pipe_loss, 0, sizeof(double), st));
  P3D_TRY(sqerr_accumulate(y, t, static_cast<size_t>(B) * m->out_size, m->pipe_loss, st));
  finish_mse_kernel<<<1, 1, 0, st>>>(m->pipe_loss, static_cast<double>(B) * m->out_size, loss);
  P3D_LAUNCH_CHECK();
  return mark_model_work(m, st);     // pipe_loss is the host-buffer step's accumulator too
}

int p3d_model_step_eval_host(p3d_model* m, const float* x_host, const float* t_host, float* y_host, float* loss_host, int64_t B) {
  P3D_REQUIRE(m && x_host && y_host, "step_eval_host: null argument");
  P3D_REQUIRE(B >= 0, "step_eval_host: negative batch");
  if (loss_host) *loss_host = 0.f;
  if (B == 0) return P3D_OK;
  P3D_CUDA(cudaSetDevice(m->cfg.device));
  const int out = m->out_size;
  // Chunk size of the H2D -> forward -> D2H pipeline (P3D_PIPE_CHUNK overrides).  Measured on 2^20 poses: 65536 and 32768
  // give 130 M poses/s end to end, 16384 gives 123, 8192 gives 77 (below ~16 K poses the fused kernel no longer fills
  // the machine).  The steady state is bound by the host->device copy: 320 B per pose at the ~45 GB/s this box's PCIe
  // link sustains with the device->host copy running the other way (tools/probe_pcie.py: 47.5 GB/s per direction).
  static const int64_t chunk_max = [] { const char* e = getenv("P3D_PIPE_CHUNK"); const long long v = e ? atoll(e) : 0; return v >= 1024 ? v : 65536LL; }();
  const int64_t chunk = B < chunk_max ? B : chunk_max;
  if (!m->pipe_streams[0])
    for (int i = 0; i < 3; ++i) P3D_CUDA(cudaStreamCreateWithFlags(&m->pipe_streams[i], cudaStreamNonBlocking));
  if (m->pipe_chunk < chunk) {
    for (int i = 0; i < 3; ++i) {
      cudaFree(m->pipe_x[i]); cudaFree(m->pipe_t[i]); cudaFree(m->pipe_y[i]);
      m->pipe_x[i] = m->pipe_t[i] = m->pipe_y[i] = nullptr;
    }
    m->pipe_chunk = 0;
    for (int i = 0; i < 3; ++i) {
      P3D_CUDA(cudaMalloc(&m->pipe_x[i], sizeof(float) * chunk * kIn));
      P3D_CUDA(cudaMalloc(&m->pipe_t[i], sizeof(float) * chunk * out));
      P3D_CUDA(cudaMalloc(&m->pipe_y[i], sizeof(float) * chunk * out));
    }
    m->pipe_chunk = chunk;
  }
  cudaStream_t s_in = m->pipe_streams[0], s_cmp = m->pipe_streams[1], s_out = m->pipe_streams[2];
  for (auto& e : m->pipe_ev) if (!e) P3D_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  cudaEvent_t* ev_in = m->pipe_ev; cudaEvent_t* ev_cmp = m->pipe_ev + 3; cudaEvent_t* ev_out = m->pipe_ev + 6;
  // a training step / epoch / forward still running on the caller's stream owns the weights, the moving statistics and
  // the forward scratch: the pipeline's streams start behind it
  P3D_TRY(order_after_model_work(m, s_in));
  P3D_TRY(order_after_model_work(m, s_cmp));
  int rc = P3D_OK;
  cudaError_t ce = cudaSuccess;
#define P3D_PIPE(call) do { if (rc == P3D_OK && ce == cudaSuccess) ce = (call); } while (0)
  if (!m->pack_valid) rc = prep::prepare(m, s_cmp);
  P3D_PIPE(cudaMemsetAsync(m->pipe_loss, 0, sizeof(double), s_cmp));
  // Tapered schedule (P3D_PIPE_TAPER=0 switches it off): the first upload and the last forward + download are not
  // overlapped by anything, so the pipeline starts and ends on quarter / half chunks (16 K poses still fill the fused
  // kernel) and runs full chunks in between.  Measured on 2^20 poses, same box: 130.9 -> 134.3 M poses/s end to end.
  static const bool taper = [] { const char* e = getenv("P3D_PIPE_TAPER"); return !(e && e[0] == '0'); }();
  int64_t head[2] = {0, 0}, tail[2] = {0, 0};
  if (taper && B >= 4 * chunk && chunk >= 4096) { head[0] = chunk / 4; head[1] = chunk / 2; tail[0] = chunk / 2; tail[1] = chunk / 4; }
  const int64_t body_end = B - tail[0] - tail[1];
  int64_t done = 0;
  for (int it = 0; rc == P3D_OK && ce == cudaSuccess && done < B; ++it) {
    const int slot = it % 3;
    int64_t n;
    if (it < 2 && head[it]) n = head[it];
    else if (done < body_end) n = (body_end - done < chunk) ? (body_end - done) : chunk;
    else n = (done == body_end && tail[0]) ? tail[0] : B - done;
    if (it >= 3) P3D_PIPE(cudaStreamWaitEvent(s_in, ev_out[slot], 0));      // slot buffers free again
    P3D_PIPE(cudaMemcpyAsync(m->pipe_x[slot], x_host + done * kIn, sizeof(float) * n * kIn, cudaMemcpyHostToDevice, s_in));
    if (t_host) P3D_PIPE(cudaMemcpyAsync(m->pipe_t[slot], t_host + done * out, sizeof(float) * n * out, cudaMemcpyHostToDevice, s_in));
    P3D_PIPE(cudaEventRecord(ev_in[slot], s_in));
    P3D_PIPE(cudaStreamWaitEvent(s_cmp, ev_in[slot], 0));
    if (ce != cudaSuccess) break;
    rc = forward_on(m, m->pipe_x[slot], m->pipe_y[slot], n, s_cmp);
    if (rc != P3D_OK) break;
    if (t_host) rc = sqerr_accumulate(m->pipe_y[slot], m->pipe_t[slot], static_cast<size_t>(n) * out, m->pipe_loss, s_cmp);
    P3D_PIPE(cudaEventRecord(ev_cmp[slot], s_cmp));
    P3D_PIPE(cudaStreamWaitEvent(s_out, ev_cmp[slot], 0));
    P3D_PIPE(cudaMemcpyAsync(y_host + done * out, m->pipe_y[slot], sizeof(float) * n * out, cudaMemcpyDeviceToHost, s_out));
    P3D_PIPE(cudaEventRecord(ev_out[slot], s_out));
    done += n;
  }
#undef P3D_PIPE
  cudaError_t e1 = cudaStreamSynchronize(s_in), e2 = cudaStreamSynchronize(s_cmp), e3 = cudaStreamSynchronize(s_out);
  if (rc != P3D_OK) return rc;
  if (ce != cudaSuccess || e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess) {
    cudaError_t e = ce != cudaSuccess ? ce : (e1 != cudaSuccess ? e1 : (e2 != cudaSuccess ? e2 : e3));
    set_error("step_eval_host: %s", cudaGetErrorString(e));
    return P3D_ERR_CUDA;
  }
  if (t_host && loss_host) {
    double acc = 0;
    P3D_CUDA(cudaMemcpy(&acc, m->pipe_loss, sizeof(double), cudaMemcpyDeviceToHost));
    *loss_host = static_cast<float>(acc / (static_cast<double>(B) * out));
  }
  return P3D_OK;
}

// CRC-32C (Castagnoli, reflected polynomial 0x82F63B78), slice-by-8 on the host: the checksum of TensorFlow's
// checkpoint files (p3d/checkpoint.py).  `init` is the CRC of the bytes that came before (0 to start).
uint32_t p3d_crc32c(const void* data_host, size_t n, uint32_t init) {
  static uint32_t T[8][256];
  static const bool ready = [] {
    for (uint32_t i = 0; i < 256; ++i) {
      uint32_t c = i;
      for (int k = 0; k < 8; ++k) c = (c & 1) ? (c >> 1) ^ 0x82F63B78u : c >> 1;
      T[0][i] = c;
    }
    for (uint32_t i = 0; i < 256; ++i)
      for (int t = 1; t < 8; ++t) T[t][i] = (T[t - 1][i] >> 8) ^ T[0][T[t - 1][i] & 0xFF];
    return true;
  }();
  (void)ready;
  const uint8_t* p = static_cast<const uint8_t*>(data_host);
  uint32_t c = ~init;
  while (n && (reinterpret_cast<uintptr_t>(p) & 7)) { c = (c >> 8) ^ T[0][(c ^ *p++) & 0xFF]; --n; }
  while (n >= 8) {
    uint64_t w;
    memcpy(&w, p, 8);
    w ^= c;
    c = T[7][w & 0xFF] ^ T[6][(w >> 8) & 0xFF] ^ T[5][(w >> 16) & 0xFF] ^ T[4][(w >> 24) & 0xFF] ^
        T[3][(w >> 32) & 0xFF] ^ T[2][(w >> 40) & 0xFF] ^ T[1][(w >> 48) & 0xFF] ^ T[0][(w >> 56) & 0xFF];
    p += 8; n -= 8;
  }
  while (n--) c = (c >> 8) ^ T[0][(c ^ *p++) & 0xFF];
  return ~c;
}

int p3d_debug_stream_mix(const void* src, void* dst, int64_t n_read_f4, int64_t n_write_f4, void* stream) {
  P3D_REQUIRE(src && dst && n_read_f4 >= 0 && n_write_f4 >= 0, "debug_stream_mix: bad argument");
  const int64_t n = n_read_f4 > n_write_f4 ? n_read_f4 : n_write_f4;
  if (n == 0) return P3D_OK;
  stream_mix_kernel<<<148 * 8, 256, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const float4*>(src), static_cast<float4*>(dst), n_read_f4, n_write_f4);
  P3D_LAUNCH_CHECK();
  return P3D_OK;
}

int p3d_debug_latency_stamps(p3d_model* m, uint64_t* out_host, int n) {
  P3D_REQUIRE(m && out_host && n >= 1 && n <= 24, "latency_stamps: bad argument");
  P3D_REQUIRE(m->lat_counter, "latency_stamps: the batch-1 kernel has not run (set P3D_LAT_STAMPS=1)");
  P3D_CUDA(cudaDeviceSynchronize());
  P3D_CUDA(cudaMemcpy(out_host, m->lat_counter + 8, sizeof(uint64_t) * n, cudaMemcpyDeviceToHost));
  return P3D_OK;
}

int p3d_debug_tc_gemm(const void* A, int lda, int a_mn, const void* B, int ldb, int b_mn, float* C, int ldc, int M, int N, int K,
                      const float* bias, const float* res, float alpha, int split_k, double* colsum, void* stream) {
  tcg::GemmArgs g;
  { const char* e = getenv("P3D_GEMM_DBG_PTR"); if (e) g.dbg = reinterpret_cast<void*>(strtoull(e, nullptr, 0)); }
  g.M = M; g.N = N; g.K = K; g.A = A; g.lda = lda; g.a_mn = a_mn; g.B = B; g.ldb = ldb; g.b_mn = b_mn; g.C = C; g.ldc = ldc;
  g.bias = bias; g.res = res; g.ldres = ldc; g.alpha = alpha; g.split_k = split_k; g.colsum = colsum;
  return tcg::gemm(g, static_cast<cudaStream_t>(stream));
}

int p3d_debug_tc_gemm_seg(const void* A, int lda, int a_mn, int seg_a, const void* B, int ldb, int b_mn, int seg_b, float* C, int ldc,
                          int M, int N, int K, const float* res, float alpha, int split_k, void* stream) {
  P3D_REQUIRE(seg_a > 0 && seg_b > 0, "debug_tc_gemm_seg: both operands are split pairs (seg_a, seg_b > 0)");
  tcg::GemmArgs g;
  g.M = M; g.N = N; g.K = K; g.A = A; g.lda = lda; g.a_mn = a_mn; g.seg_a = seg_a; g.B = B; g.ldb = ldb; g.b_mn = b_mn; g.seg_b = seg_b;
  g.C = C; g.ldc = ldc; g.res = res; g.ldres = ldc; g.alpha = alpha; g.split_k = split_k;
  return tcg::gemm(g, static_cast<cudaStream_t>(stream));
}

int p3d_debug_mma_rate(int N, int iters, int64_t* out_dev, void* stream) {
  P3D_REQUIRE(out_dev, "debug_mma_rate: null argument");
  return tcg::mma_rate(N, iters, reinterpret_cast<long long*>(out_dev), static_cast<cudaStream_t>(stream));
}

int p3d_debug_umma_gemm(const void* A, const void* W, float* C, int N, int K, void* stream) {
  P3D_REQUIRE(A && W && C, "debug_umma_gemm: null argument");
  return tc::debug_umma_gemm(A, W, C, N, K, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
