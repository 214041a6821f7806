// Realtime front-end and back-end around the lifter: the arithmetic of the frame loop of
// src/openpose_3dpose_sandbox_realtime.py:137-171
//   keypoints (18 OpenPose/COCO joints) -> H3.6M joint order + synthesised Hip / Neck / Thorax (:137-154)
//   -> enc_in[:, dim_to_use_2d], (enc_in - mu) / sigma (:160-163) -> model.step(isTraining=False) (:168)
//   -> data_utils.unNormalizeData of the prediction (:171, src/data_utils.py:283-311).
//
// One frame (batch 1, host buffers) is ONE kernel launch: the 16-CTA cluster kernel of mlp_simt.cu reads the
// keypoints from mapped pinned memory, runs the front-end on load, the six layers, the un-normalisation on store,
// writes the results straight into mapped pinned memory and raises a flag there; the host spins on the flag.  No
// cudaMemcpy and no stream synchronise on the frame's critical path.  Batches of frames (device buffers) run as
// front-end kernel -> p3d_model_forward -> back-end kernel.
#include <chrono>
#include <cstring>

#include "common.cuh"
#include "math_hd.h"

namespace p3d {
namespace prep { int prepare(p3d_model* m, cudaStream_t st); }
namespace simt { int forward_latency_cluster_rt_people(p3d_model* m, const rt::Fused& f, float* y, int people, cudaStream_t st); }
namespace rt {

constexpr int kMaxPeople = 8;        // people of one frame the cluster kernel serves in one launch

struct HostIO {                      // one mapped pinned block shared with the kernel: up to kMaxPeople people
  double kp[kMaxPeople][36];
  double pose[kMaxPeople][96];
  float enc[kMaxPeople][32];
  float y[kMaxPeople * 48];          // [P][out]
  unsigned long long flag;
};

}  // namespace rt
}  // namespace p3d

struct p3d_realtime {
  p3d_model* model = nullptr;
  p3d::rt::Tables host_tab;
  p3d::rt::Tables* dev_tab = nullptr;
  p3d::rt::HostIO* io = nullptr;     // cudaHostAlloc'ed, mapped
  cudaStream_t stream = nullptr;
  unsigned long long seq = 0;
  // staging of the generic path (width != 1024 / fp32 mode / no 16-CTA cluster / more than kMaxPeople people)
  double* d_kp = nullptr; float* d_enc = nullptr; float* d_y = nullptr; double* d_pose = nullptr;
  int64_t d_cap = 0;                 // rows the staging buffers hold
};

namespace p3d {
namespace rt {

// enc_in[b, i] = (h36m(kp[b])[use2[i]] - mu2[i]) / sd2[i], fp64 arithmetic, fp32 result (the TF feed's cast)
__global__ void frontend_kernel(const double* __restrict__ kp, const Tables* __restrict__ tab, float* __restrict__ enc, long long B) {
  const long long total = B * 32;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long b = i >> 5;
    const int c = static_cast<int>(i & 31);
    const double v = (openpose_h36m_coord(kp + b * 36, tab->use2[c]) - tab->mu2[c]) / tab->sd2[c];
    enc[i] = static_cast<float>(v);
  }
}

// pose[b, j] = float32(y[b, pos3[j]]) * sd3[j] + mu3[j]   (ignored dims: 0 * sd + mu), data_utils.py:299-311
__global__ void backend_kernel(const float* __restrict__ y, const Tables* __restrict__ tab, double* __restrict__ pose, long long B) {
  const long long total = B * 96;
  const int out = tab->out;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long b = i / 96;
    const int j = static_cast<int>(i - b * 96);
    const int s = tab->pos3[j];
    const double v = s >= 0 ? static_cast<double>(y[b * out + s]) : 0.0;
    pose[i] = __dadd_rn(__dmul_rn(v, tab->sd3[j]), tab->mu3[j]);
  }
}

// grow the staging buffers to B rows (the previous call synchronised its stream, nothing still reads them)
static int ensure_staging(p3d_realtime* r, int64_t B) {
  if (B <= r->d_cap) return P3D_OK;
  cudaFree(r->d_kp); cudaFree(r->d_enc); cudaFree(r->d_y); cudaFree(r->d_pose);
  r->d_kp = nullptr; r->d_enc = nullptr; r->d_y = nullptr; r->d_pose = nullptr; r->d_cap = 0;
  P3D_CUDA(cudaMalloc(&r->d_kp, sizeof(double) * 36 * B));
  P3D_CUDA(cudaMalloc(&r->d_enc, sizeof(float) * 32 * B));
  P3D_CUDA(cudaMalloc(&r->d_y, sizeof(float) * 48 * B));
  P3D_CUDA(cudaMalloc(&r->d_pose, sizeof(double) * 96 * B));
  r->d_cap = B;
  return P3D_OK;
}

// spin on the mapped flag until the kernel raised it to seq; look at the stream now and then so that a failed launch
// cannot hang the caller
static int wait_flag(p3d_realtime* r, unsigned long long seq, const char* who) {
  volatile unsigned long long* flag = &r->io->flag;
  const auto t0 = std::chrono::steady_clock::now();
  unsigned spins = 0;
  while (*flag != seq) {
    if ((++spins & 0xFFFF) == 0) {
      const cudaError_t q = cudaStreamQuery(r->stream);
      if (q != cudaSuccess && q != cudaErrorNotReady) { set_error("%s: %s", who, cudaGetErrorString(q)); return P3D_ERR_CUDA; }
      if (q == cudaSuccess && *flag != seq) { set_error("%s: the kernel finished without raising its flag", who); return P3D_ERR_CUDA; }
      if (std::chrono::steady_clock::now() - t0 > std::chrono::seconds(10)) { set_error("%s: timed out", who); return P3D_ERR_CUDA; }
    }
  }
  __sync_synchronize();
  return P3D_OK;
}

static inline int grid_for(long long n) { long long g = (n + 255) / 256; if (g > 148 * 8) g = 148 * 8; return static_cast<int>(g < 1 ? 1 : g); }

static int step_device(p3d_realtime* r, const double* kp, float* enc, float* y, double* pose, int64_t B, cudaStream_t st) {
  frontend_kernel<<<grid_for(B * 32), 256, 0, st>>>(kp, r->dev_tab, enc, B);
  P3D_LAUNCH_CHECK();
  P3D_TRY(p3d_model_forward(r->model, enc, y, B, st));
  if (pose) {
    backend_kernel<<<grid_for(B * 96), 256, 0, st>>>(y, r->dev_tab, pose, B);
    P3D_LAUNCH_CHECK();
  }
  return P3D_OK;
}

}  // namespace rt
}  // namespace p3d

using namespace p3d;

extern "C" {

int p3d_realtime_create(p3d_model* m, const double* mean2d, const double* std2d, const int32_t* use2d, const double* mean3d,
                        const double* std3d, const int32_t* use3d, p3d_realtime** out) {
  P3D_REQUIRE(m && mean2d && std2d && use2d && mean3d && std3d && use3d && out, "realtime_create: null argument");
  P3D_REQUIRE(m->out_size <= 48, "realtime_create: output width above 48");
  P3D_CUDA(cudaSetDevice(m->cfg.device));
  rt::Tables t;
  memset(&t, 0, sizeof(t));
  for (int i = 0; i < 32; ++i) {
    P3D_REQUIRE(use2d[i] >= 0 && use2d[i] < 64, "realtime_create: dim_to_use_2d entry outside 0..63");
    P3D_REQUIRE(std2d[use2d[i]] != 0.0, "realtime_create: zero 2D standard deviation on a used dimension");
    t.use2[i] = use2d[i]; t.mu2[i] = mean2d[use2d[i]]; t.sd2[i] = std2d[use2d[i]];
  }
  for (int j = 0; j < 96; ++j) { t.mu3[j] = mean3d[j]; t.sd3[j] = std3d[j]; t.pos3[j] = -1; }
  t.out = m->out_size;
  for (int g = 0; g < t.out; ++g) {
    P3D_REQUIRE(use3d[g] >= 0 && use3d[g] < 96, "realtime_create: dim_to_use_3d entry outside 0..95");
    P3D_REQUIRE(t.pos3[use3d[g]] < 0, "realtime_create: dim_to_use_3d repeats a dimension");
    t.use3[g] = use3d[g]; t.pos3[use3d[g]] = g;
  }
  p3d_realtime* r = new p3d_realtime();
  r->model = m; r->host_tab = t;
  auto fail = [&](const char* what) {
    set_error("realtime_create: %s: %s", what, cudaGetErrorString(cudaGetLastError()));
    p3d_realtime_destroy(r);
    return P3D_ERR_CUDA;
  };
  if (cudaMalloc(&r->dev_tab, sizeof(rt::Tables)) != cudaSuccess) return fail("cudaMalloc");
  if (cudaMemcpy(r->dev_tab, &t, sizeof(t), cudaMemcpyHostToDevice) != cudaSuccess) return fail("cudaMemcpy");
  if (cudaHostAlloc(reinterpret_cast<void**>(&r->io), sizeof(rt::HostIO), cudaHostAllocMapped) != cudaSuccess) return fail("cudaHostAlloc");
  memset(r->io, 0, sizeof(rt::HostIO));
  for (int b = 0; b < rt::kMaxPeople; ++b)          // ignored dims never change (data_utils.py:305-310)
    for (int j = 0; j < 96; ++j) r->io->pose[b][j] = 0.0 * t.sd3[j] + t.mu3[j];
  if (cudaStreamCreateWithFlags(&r->stream, cudaStreamNonBlocking) != cudaSuccess) return fail("cudaStreamCreate");
  if (rt::ensure_staging(r, 1) != P3D_OK) return fail("cudaMalloc");
  *out = r;
  return P3D_OK;
}

void p3d_realtime_destroy(p3d_realtime* r) {
  if (!r) return;
  if (r->stream) { cudaStreamSynchronize(r->stream); cudaStreamDestroy(r->stream); }
  cudaFree(r->dev_tab); cudaFree(r->d_kp); cudaFree(r->d_enc); cudaFree(r->d_y); cudaFree(r->d_pose);
  if (r->io) cudaFreeHost(r->io);
  delete r;
}

int p3d_realtime_step(p3d_realtime* r, const double* xy36, float* enc_in, float* y, double* pose3d_or_null, int64_t B, void* stream) {
  P3D_REQUIRE(r && xy36 && enc_in && y, "realtime_step: null argument");
  P3D_REQUIRE(B >= 0, "realtime_step: negative batch");
  if (B == 0) return P3D_OK;
  P3D_CUDA(cudaSetDevice(r->model->cfg.device));
  return rt::step_device(r, xy36, enc_in, y, pose3d_or_null, B, static_cast<cudaStream_t>(stream));
}

int p3d_realtime_step_host(p3d_realtime* r, const double* xy36_host, float* enc_in_host_or_null, float* y_host_or_null,
                           double* pose3d_host) {
  P3D_REQUIRE(r && xy36_host && pose3d_host, "realtime_step_host: null argument");
  p3d_model* m = r->model;
  P3D_CUDA(cudaSetDevice(m->cfg.device));
  const int out = m->out_size;
  P3D_TRY(order_after_model_work(m, r->stream));     // a training step still running on the caller's stream owns the weights
  if (!m->pack_valid) { P3D_TRY(prep::prepare(m, r->stream)); }
  rt::HostIO* io = r->io;
  memcpy(io->kp[0], xy36_host, sizeof(double) * 36);
  rt::Fused f;
  f.tab = r->dev_tab; f.kp = io->kp[0]; f.enc = io->enc[0]; f.pose = io->pose[0]; f.flag = &io->flag; f.seq = ++r->seq;
  int rc = simt::forward_latency_cluster_rt(m, f, io->y, r->stream);
  if (rc < 0) return rc;
  if (rc == 0) {
    P3D_TRY(rt::wait_flag(r, f.seq, "realtime_step_host"));
    memcpy(pose3d_host, io->pose[0], sizeof(double) * 96);
    if (enc_in_host_or_null) memcpy(enc_in_host_or_null, io->enc, sizeof(float) * 32);
    if (y_host_or_null) memcpy(y_host_or_null, io->y, sizeof(float) * out);
    return P3D_OK;
  }
  // generic route (width != 1024, fp32 mode, or a 16-CTA cluster cannot be scheduled): staged copies around the kernels
  P3D_TRY(order_after_model_work(r->model, r->stream));
  P3D_CUDA(cudaMemcpyAsync(r->d_kp, io->kp[0], sizeof(double) * 36, cudaMemcpyHostToDevice, r->stream));
  P3D_TRY(rt::step_device(r, r->d_kp, r->d_enc, r->d_y, r->d_pose, 1, r->stream));
  P3D_CUDA(cudaMemcpyAsync(io->pose[0], r->d_pose, sizeof(double) * 96, cudaMemcpyDeviceToHost, r->stream));
  P3D_CUDA(cudaMemcpyAsync(io->enc[0], r->d_enc, sizeof(float) * 32, cudaMemcpyDeviceToHost, r->stream));
  P3D_CUDA(cudaMemcpyAsync(io->y, r->d_y, sizeof(float) * out, cudaMemcpyDeviceToHost, r->stream));
  P3D_CUDA(cudaStreamSynchronize(r->stream));
  memcpy(pose3d_host, io->pose[0], sizeof(double) * 96);
  if (enc_in_host_or_null) memcpy(enc_in_host_or_null, io->enc, sizeof(float) * 32);
  if (y_host_or_null) memcpy(y_host_or_null, io->y, sizeof(float) * out);
  return P3D_OK;
}

int p3d_realtime_step_people_host(p3d_realtime* r, const double* xy36_host, int P, float* enc_in_host_or_null,
                                  float* y_host_or_null, double* pose3d_host) {
  P3D_REQUIRE(r && xy36_host && pose3d_host, "realtime_step_people_host: null argument");
  P3D_REQUIRE(P >= 0, "realtime_step_people_host: negative number of people");
  if (P == 0) return P3D_OK;
  p3d_model* m = r->model;
  P3D_CUDA(cudaSetDevice(m->cfg.device));
  const int out = m->out_size;
  P3D_TRY(order_after_model_work(m, r->stream));     // a training step still running on the caller's stream owns the weights
  if (!m->pack_valid) { P3D_TRY(prep::prepare(m, r->stream)); }
  rt::HostIO* io = r->io;
  if (P <= rt::kMaxPeople) {
    memcpy(io->kp, xy36_host, sizeof(double) * 36 * P);
    rt::Fused f;
    f.tab = r->dev_tab; f.kp = io->kp[0]; f.enc = io->enc[0]; f.pose = io->pose[0]; f.flag = &io->flag; f.seq = ++r->seq;
    const int rc = simt::forward_latency_cluster_rt_people(m, f, io->y, P, r->stream);
    if (rc < 0) return rc;
    if (rc == 0) {
      P3D_TRY(rt::wait_flag(r, f.seq, "realtime_step_people_host"));
      memcpy(pose3d_host, io->pose, sizeof(double) * 96 * P);
      if (enc_in_host_or_null) memcpy(enc_in_host_or_null, io->enc, sizeof(float) * 32 * P);
      if (y_host_or_null) memcpy(y_host_or_null, io->y, sizeof(float) * out * P);
      return P3D_OK;
    }
  }
  // staged route: one upload of all P people, the batched device step, the downloads, one synchronise
  P3D_TRY(rt::ensure_staging(r, P));
  P3D_CUDA(cudaMemcpyAsync(r->d_kp, xy36_host, sizeof(double) * 36 * P, cudaMemcpyHostToDevice, r->stream));
  P3D_TRY(rt::step_device(r, r->d_kp, r->d_enc, r->d_y, r->d_pose, P, r->stream));
  P3D_CUDA(cudaMemcpyAsync(pose3d_host, r->d_pose, sizeof(double) * 96 * P, cudaMemcpyDeviceToHost, r->stream));
  if (enc_in_host_or_null)
    P3D_CUDA(cudaMemcpyAsync(enc_in_host_or_null, r->d_enc, sizeof(float) * 32 * P, cudaMemcpyDeviceToHost, r->stream));
  if (y_host_or_null)
    P3D_CUDA(cudaMemcpyAsync(y_host_or_null, r->d_y, sizeof(float) * out * P, cudaMemcpyDeviceToHost, r->stream));
  P3D_CUDA(cudaStreamSynchronize(r->stream));
  return P3D_OK;
}

}  // extern "C"
