/* p3d.h - C ABI of libp3d.so: the B200 (sm_100a) implementation of 3d-pose-baseline's hot path.
 *
 * The reference (EsauPR/3d-pose-baseline) is pure Python: it has no FFI/plugin layer, every device
 * op runs inside TensorFlow and every geometry op inside NumPy.  The drop-in boundary is therefore
 * the reference's Python surface (mirrored in 3d-pose-baseline_b200/p3d/*.py); this header is the
 * C ABI that mirror binds through ctypes.  Each entry cites the reference interface it replaces
 * (paths relative to the reference repository).
 *
 * Conventions
 *   - every call returns 0 on success, <0 on error; p3d_last_error() gives a thread-local message.
 *   - pointers are DEVICE pointers unless the name ends in _host.  The caller owns every buffer it
 *     passes; the library keeps no caller pointer after return.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  Calls are
 *     asynchronous on that stream unless they take/return host data.
 *   - handles are not thread-safe; distinct handles may be used from distinct threads.
 *   - there is NO CPU fallback: without a CUDA device every compute call fails with P3D_ERR_CUDA.
 *
 * CUDA graphs
 *   - capturable on a stream in capture (cudaStreamBeginCapture, torch.cuda.graph): p3d_model_forward,
 *     p3d_model_mse and p3d_realtime_step, at any batch size, width and mode.  Every other call that takes a
 *     model returns P3D_ERR_STATE on a capturing stream (training steps and epochs, prepare_inference) or is
 *     synchronous and must not be called during a capture (host-buffer steps, the realtime host frame).
 *   - warm-up: a call may allocate or grow scratch, or set up a kernel, the first time it meets a batch size.  On
 *     a capturing stream it cannot, and returns P3D_ERR_STATE instead; run the same call once outside the capture
 *     first (PyTorch's warm-up convention).
 *   - weights: a graph reads the packed inference weights in place.  After set_param_host, a checkpoint restore
 *     or a training step, call p3d_model_prepare_inference outside the capture before the next replay (a capture
 *     while the fold is stale returns P3D_ERR_STATE rather than capturing the fold).
 *   - the caller's buffers (x, y, t, loss, the realtime inputs and outputs) must outlive the graph; the library's
 *     scratch does (buffers a graph may address are freed by p3d_model_destroy only; once a model has been
 *     captured, growing scratch at least doubles, so what is kept stays below the size of the live buffer).
 *   - a replay is ordered before later host-buffer steps and realtime host frames of the model, as eager calls
 *     are.  Replays of graphs of ONE model must not run concurrently (they share the model's scratch): replay
 *     them on one stream, or order them.  A replay after a training step has handed the fused kernel's
 *     persisting-L2 set-aside back is slower, not different.
 */
#ifndef P3D_H_
#define P3D_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define P3D_OK 0
#define P3D_ERR_ARG (-1)
#define P3D_ERR_CUDA (-2)
#define P3D_ERR_STATE (-3)
#define P3D_ERR_NCCL (-4)

#define P3D_MODE_BF16 0 /* tcgen05 bf16 x bf16 -> fp32 accumulate (headline path) */
#define P3D_MODE_FP32 1 /* fp32 FFMA path, <=1e-4 relative to the fp64 oracle */
/* fp32-class (<=1e-4 relative to the fp64 oracle): inference on tcgen05 as three split-bf16 products per MatMul
 * (hi*hi + lo*hi + hi*lo, fp32 accumulation, fp32 activations); linear_size % 8 != 0 runs the FFMA path.  Training
 * steps and epochs are those of P3D_MODE_FP32 unless p3d_model_set_train_matmul(P3D_TRAIN_MATMUL_BF16X3) puts their
 * MatMuls on the tensor cores too; the whole-chip bf16 kernels and the one-launch realtime frame are not used (frames
 * take the staged route). */
#define P3D_MODE_BF16X3 2
/* fp16 operands wherever P3D_MODE_BF16 uses bf16: every inference path of bf16 mode (the fused kernel, the per-layer
 * GEMMs, the whole-chip kernels for 1-64 poses and the one-launch realtime frame), the same rounding points, fp32
 * accumulation, the same tensor-core rate.  Contract: <= 2e-3 row-wise relative error against the fp64 oracle (bf16
 * mode: ~6e-3), provided every folded weight, input and activation stays inside fp16's range (|v| <= 65504).
 * linear_size % 8 != 0 runs the fp32 FFMA path.  Training steps and epochs are those of P3D_MODE_BF16 (the same
 * kernels on the bf16 tensor cores); p3d_model_set_train_matmul returns P3D_ERR_ARG. */
#define P3D_MODE_FP16 3

const char* p3d_last_error(void);
int p3d_version(void);
/* number of kernels this library has launched so far in this process (bench.py's gpu_launches) */
int64_t p3d_launch_count(void);

/* Per-launch CUDA-event timing of the dominant kernel (the fused tcgen05 forward), recorded on the
 * launching stream.  enable(1) resets the counters; read() waits for the recorded events and returns
 * the summed device time and the number of launches since enable. */
int p3d_profile_enable(int on);
int p3d_profile_read(double* ms_total, int64_t* launches);

/* pinned host memory for the end-to-end path (cudaHostAlloc / cudaFreeHost) */
int p3d_host_alloc(void** out_host, size_t bytes);
int p3d_host_free(void* host);

/* ---------------------------------------------------------------- LinearModel -----------------
 * linear_model.LinearModel.__init__ (src/linear_model.py:34-151): same flags. */
typedef struct p3d_model p3d_model;
typedef struct {
  int linear_size; /* src/linear_model.py:35 */
  int num_layers;  /* :36 number of two_linear blocks */
  int residual;    /* :37 */
  int batch_norm;  /* :38 */
  int max_norm;    /* :39 tf.clip_by_norm(w,1): whole-matrix Frobenius clip inside the graph */
  int predict_14;  /* :43 output width 42 instead of 48 */
  int mode;        /* P3D_MODE_* */
  int device;      /* CUDA ordinal */
  float learning_rate; /* :41 */
} p3d_cfg;

int p3d_model_create(const p3d_cfg* cfg, p3d_model** out);
void p3d_model_destroy(p3d_model* m);

/* Variables by their TensorFlow names (what tf.train.Saver stores, src/linear_model.py:151):
 * "linear_model/w1", "linear_model/b1", "linear_model/batch_normalization/{gamma,beta,moving_mean,
 * moving_variance}", "linear_model/two_linear_<i>/{w2_<i>,b2_<i>,batch_normalization1<i>/...,w3_<i>,
 * b3_<i>,batch_normalization2<i>/...}", "linear_model/w4", "linear_model/b4"; optimizer state as
 * "<var>/Adam" (m) and "<var>/Adam_1" (v); "global_step" (as float); "learning_rate" (the base
 * rate variable, src/linear_model.py:86) is settable/gettable by name but not enumerated.  Weights are [in,out] row-major. */
int p3d_model_set_param_host(p3d_model* m, const char* tf_name, const float* host, size_t n);
int p3d_model_get_param_host(p3d_model* m, const char* tf_name, float* host, size_t n);
int p3d_model_param_count(p3d_model* m);
int p3d_model_param_name(p3d_model* m, int index, char* out, size_t cap, size_t* numel);

/* Fold clip_by_norm + moving-statistics BN into per-layer W',b' and pack them for the forward
 * kernels (src/linear_model.py:108-112,178-193,123).  Called lazily by forward if params changed. */
int p3d_model_prepare_inference(p3d_model* m, void* stream);

/* model.step(..., isTraining=False) forward (src/linear_model.py:237-245): y[B,out] = f(x[B,32]).
 * x, y fp32 row-major on the device; any B >= 1. */
int p3d_model_forward(p3d_model* m, const float* x, float* y, int64_t B, void* stream);
/* mean((y-t)^2) over all B*out elements (src/linear_model.py:129); loss is a DEVICE float. */
int p3d_model_mse(p3d_model* m, const float* y, const float* t, int64_t B, float* loss, void* stream);
/* the same step with HOST buffers (what a NumPy caller of step() passes): chunked, pipelined
 * H2D -> forward -> D2H inside.  x_host/t_host/y_host may be pageable or pinned.  t_host may be NULL
 * (loss_host then receives 0).  Synchronous. */
int p3d_model_step_eval_host(p3d_model* m, const float* x_host, const float* t_host, float* y_host,
                             float* loss_host, int64_t B);

/* model.step(..., isTraining=True) (src/linear_model.py:226-235): forward with batch statistics and
 * dropout, MSE, backward, BN moving-average update, TF-Adam with exponential lr decay; y receives the
 * pre-update outputs, loss/lr_used are DEVICE floats.  mask_or_null: optional uint8 [nhidden][B][L]
 * dropout keep-mask (1 = keep) injected for tests; otherwise a Philox4x32-10 mask is generated from
 * (seed, global_step, layer, global_row0 + row, col).  global_B/row0 describe this rank's shard when
 * data-parallel (global_B = B, row0 = 0 on one GPU). */
int p3d_model_train_step(p3d_model* m, const float* x, const float* t, int64_t B, float keep_prob,
                         uint64_t seed, const uint8_t* mask_or_null, int64_t global_B, int64_t row0,
                         float* loss, float* lr_used, float* y, void* stream);

/* The batch loop of predict_3dpose.train() (src/predict_3dpose.py:231-259) over a DEVICE-resident training set:
 * X[n,32] / T[n,out] are what LinearModel.get_all_batches concatenates (src/linear_model.py:266-300),
 * perm_or_null[n] its np.random.permutation (int64, device; NULL = natural order), the n % batch_size tail is
 * dropped (:311-313).  Every batch is gathered on the device and stepped as a replayed CUDA graph - no host
 * synchronisation inside.  losses[n / batch_size] (device) receives each step's loss, lr_last_or_null the last
 * learning rate.  Single GPU (data-parallel models call p3d_model_train_step per batch). */
int p3d_model_train_epoch(p3d_model* m, const float* X, const float* T, int64_t n, const int64_t* perm_or_null, int64_t batch_size,
                          float keep_prob, uint64_t seed, float* losses, float* lr_last_or_null, void* stream);

/* Which arithmetic runs the MatMuls of a training step (steps and epochs), chosen per model:
 *   P3D_TRAIN_MATMUL_DEFAULT: the mode's own route - tcgen05 bf16 (P3D_MODE_BF16, P3D_MODE_FP16), FFMA (P3D_MODE_FP32,
 *                             P3D_MODE_BF16X3).
 *   P3D_TRAIN_MATMUL_BF16X3 : every MatMul of the step (forward, data and weight gradients) on tcgen05 as three split-bf16
 *                             products hi*hi + lo*hi + hi*lo with fp32 accumulation; activations, BatchNorm, dropout,
 *                             the loss and Adam stay fp32 as on the FFMA route.  fp32-class, not bit-equal to FFMA: at
 *                             batch 64 gradients are within 2e-5 of each tensor's max of the fp64 graph; at batch 4096
 *                             the split operands move pre-activations by ~1e-5 relative, which flips the ReLU of a few
 *                             dozen units near zero (gradients within ~3e-3 relative L2) - hence opt-in.  Widths with
 *                             linear_size % 8 != 0 keep the FFMA route.
 * Valid on P3D_MODE_FP32 and P3D_MODE_BF16X3 models; a P3D_MODE_BF16 or P3D_MODE_FP16 model returns P3D_ERR_ARG.  A host call without a
 * stream: it must not be made while a training step of the model is in flight.  Switching drops the model's captured
 * training-step graphs (the next step captures again).  Data-parallel ranks must all set the same kind. */
#define P3D_TRAIN_MATMUL_DEFAULT 0
#define P3D_TRAIN_MATMUL_BF16X3 1
int p3d_model_set_train_matmul(p3d_model* m, int kind);
/* Data parallel: a NCCL communicator owned by the library (SyncBN statistics + one gradient
 * all-reduce per step).  id_host = 128-byte ncclUniqueId made by rank 0 and broadcast by the caller. */
int p3d_nccl_unique_id(uint8_t* id_host /*[128]*/);
int p3d_model_attach_nccl(p3d_model* m, const uint8_t* id_host, int rank, int world);

/* Optional, after attach_nccl, ranks of ONE node: the latency-bound reductions of a data-parallel step (SyncBN sums
 * forward and backward, loss) then travel over NVLink peer memory instead of NCCL calls - inside the GEMM kernels that
 * need them (fused training epilogues: batches whose tiles all fit the SMs) or as single kernels; and the flat gradient
 * all-reduce becomes one pull / sum-in-rank-order / push kernel over the peer-mapped gradient buffers instead of
 * ncclAllReduce (P3D_P2P_GRAD=0 keeps NCCL).  Every rank exports two CUDA IPC handles (exchange buffer, gradient buffer:
 * 128 bytes), the host layer all-gathers them, every rank attaches all `world` entries (rank-major, 128 bytes each).  If a peer is not reachable attach fails, closes what it had opened and
 * the step keeps using NCCL; p3d_model_p2p_detach does the same on request (the host layer calls it on every rank when
 * ANY rank failed to attach, so that all ranks take the same path).  The exchange waits for its peers like an NCCL
 * collective (no timeout; P3D_SYNC_TIMEOUT_S=<s> makes a longer wait trap): ranks must step in lockstep. */
int p3d_model_p2p_handle(p3d_model* m, uint8_t* handle128_host);   /* [exchange buffer | flat gradient buffer] */
int p3d_model_p2p_attach(p3d_model* m, const uint8_t* handles_host, int rank, int world);
int p3d_model_p2p_detach(p3d_model* m);
/* Data parallel, after p3d_model_train_step: the outputs of the GLOBAL batch [global_B, out] (device pointer).  When the
 * gradient travelled over peer memory, every rank's rows were written into every rank's exchange buffer on the way and
 * this is one device-to-device copy; returns 1 (and copies nothing) when they are not available - NCCL gradient path,
 * or a global batch beyond the buffer (10922 rows) - and the caller all-gathers the per-rank outputs itself. */
int p3d_model_gathered_outputs(p3d_model* m, float* y_global, int64_t global_B, void* stream);
/* Measurement aid (bench.py `secondary.train_dp`): one exchange of a data-parallel step on its own, on `stream`.
 * what = 0: the flat fp32 gradient all-reduce; 1: one SyncBN-sized (2 x linear_size doubles) sum - both over peer memory
 * when it is attached (the step's own path), over NCCL otherwise.  The buffers hold whatever the last step left; they are summed in place. */
int p3d_debug_dp_part(p3d_model* m, int what, void* stream);
int64_t p3d_model_global_step(p3d_model* m);

/* CRC-32C of a HOST buffer (host code, slice-by-8): the checksum TensorFlow's checkpoint format uses for table blocks
 * and tensors (tf.train.Saver, src/linear_model.py:151) - see p3d/checkpoint.py.  init = CRC of the preceding bytes. */
uint32_t p3d_crc32c(const void* data_host, size_t n, uint32_t init);

/* ---------------------------------------------------------------- realtime front-end ----------
 * The per-frame arithmetic of src/openpose_3dpose_sandbox_realtime.py:137-171 around model.step():
 *   xy36 = the first 18 OpenPose/COCO keypoints as (x,y) pairs (:137-142, fp64 like the JSON floats)
 *   -> scatter into H3.6M joint order (order = [15,12,25,26,27,17,18,19,1,2,3,6,7,8], :20,:144-147),
 *      Hip = (RHip+LHip)/2, Neck/Nose = (Head+Spine)/2, Thorax = 2*Spine - Neck/Nose (:148-154)
 *   -> enc_in = (enc_in[dim_to_use_2d] - mean) / std in fp64 (:160-163), cast to fp32 by the feed
 *   -> y = model.step(enc_in, isTraining=False) (:168)
 *   -> pose3d[96] = data_utils.unNormalizeData(y, mean3d, std3d, ignore) (:171; src/data_utils.py:283-311).
 * create() copies the statistics: mean2d/std2d[64], use2d[32] = dim_to_use_2d, mean3d/std3d[96],
 * use3d[out] = dim_to_use_3d (all HOST pointers, as returned by normalization_stats). */
typedef struct p3d_realtime p3d_realtime;
int p3d_realtime_create(p3d_model* m, const double* mean2d_host, const double* std2d_host, const int32_t* use2d_host,
                        const double* mean3d_host, const double* std3d_host, const int32_t* use3d_host, p3d_realtime** out);
void p3d_realtime_destroy(p3d_realtime* r);
/* One frame, HOST buffers, synchronous.  With linear_size 1024 in bf16 or fp16 mode this is a single kernel launch that reads
 * the keypoints from and writes the results to mapped pinned memory (no cudaMemcpy, no stream synchronise).
 * enc_in_host[32] and y_host[out] (the normalised input / prediction) are optional. */
int p3d_realtime_step_host(p3d_realtime* r, const double* xy36_host, float* enc_in_host_or_null, float* y_host_or_null,
                           double* pose3d_host /*[96]*/);
/* B frames, DEVICE buffers, asynchronous on `stream`: xy36[B,36] fp64 -> enc_in[B,32], y[B,out], pose3d[B,96] (optional). */
int p3d_realtime_step(p3d_realtime* r, const double* xy36, float* enc_in, float* y, double* pose3d_or_null, int64_t B,
                      void* stream);

/* ---------------------------------------------------------------- cameras ---------------------
 * One H36M camera as loaded by cameras.load_camera_params (src/cameras.py:92-120). */
typedef struct {
  double R[9]; /* row-major 3x3 */
  double T[3];
  double f[2];
  double c[2];
  double k[3];
  double p[2];
} p3d_camera;

/* cameras.project_point_radial (src/cameras.py:13-53).  P[npts,3] -> proj[npts,2], and optionally
 * D, radial, tan, r2 [npts] (NULL = not wanted).  f64 variant = reference precision. */
int p3d_project_point_radial_f64(const double* P, const p3d_camera* cam_host, double* proj, double* D,
                                 double* radial, double* tan_, double* r2, int64_t npts, void* stream);
int p3d_project_point_radial_f32(const float* P, const p3d_camera* cam_host, float* proj, float* D,
                                 float* radial, float* tan_, float* r2, int64_t npts, void* stream);
/* cameras.world_to_camera_frame / camera_to_world_frame (src/cameras.py:55-90) */
int p3d_world_to_camera_f64(const double* P, const p3d_camera* cam_host, double* out, int64_t npts, void* stream);
int p3d_camera_to_world_f64(const double* P, const p3d_camera* cam_host, double* out, int64_t npts, void* stream);

/* Fused camera_frame preprocessing for ncams (<=8) cameras:
 *   2D: data_utils.project_to_cameras (src/data_utils.py:339-364) + normalize_data (:260-280)
 *   3D: transform_world_to_camera (:233-257) + postprocess_3d (:474-494) + normalize_data
 * world[N,96] fp32 -> x2d[ncams,N,32] and/or y3d[ncams,N,48 or 42] fp32 (either may be NULL).
 * mean/std are full-width (64 / 96) host vectors; the dims_to_use tables are built in. */
int p3d_project_normalize(const float* world, const p3d_camera* cams_host, int ncams, const double* mean2d_host,
                          const double* std2d_host, const double* mean3d_host, const double* std3d_host,
                          int predict_14, float* x2d, float* y3d, int64_t N, void* stream);

/* data_utils.normalize_data / unNormalizeData for one array (src/data_utils.py:260-311).
 * dim = 2 or 3.  normalize: in[N,64|96] -> out[N,32|48|42];  unnormalize: the inverse, ignored
 * dims come out as the mean.  f64 I/O like the reference (unnormalize rounds its input to fp32 first,
 * as the reference does at :299-303). */
int p3d_normalize_f64(const double* in, const double* mean_host, const double* std_host, int dim, int predict_14,
                      double* out, int64_t N, void* stream);
int p3d_unnormalize_f64(const double* in, const double* mean_host, const double* std_host, int dim, int predict_14,
                        double* out, int64_t N, void* stream);

/* data_utils.normalization_stats (src/data_utils.py:211-212): column mean and population std of
 * data[N,D] (f64).  work = 2*D device doubles of scratch. */
int p3d_column_stats_f64(const double* data, int64_t N, int D, double* mean, double* stdv, double* work, void* stream);
/* data_utils.postprocess_3d (src/data_utils.py:474-494) for one array: out = in - tile(in[:, :3]);
 * roots_or_null[N,3] receives the root positions.  Out of place. */
int p3d_root_center_f64(const double* in, double* out, double* roots_or_null, int64_t N, int D, void* stream);

/* ---------------------------------------------------------------- evaluation ------------------
 * predict_3dpose.evaluate_batches arithmetic (src/predict_3dpose.py:399-442) + per-pose
 * procrustes.compute_similarity_transform(gt, out, compute_optimal_scale=True) (src/procrustes.py:2-63).
 * pred_n, gt_n: normalised [N,48|42] fp32.  dists_or_null[N,J] (J=17|14) per-joint errors in mm;
 * joint_sum[J] DEVICE doubles are ACCUMULATED into (caller zeroes them), so that joint_err =
 * joint_sum/N and total_err = sum(joint_sum)/(N*J).
 * p3d_procrustes_mpjpe is the HBM-bound fp32 kernel (MPJPE / per-joint means within 1e-5 mm of the NumPy
 * float64 reference, single per-pose distances within 1e-3 mm); p3d_procrustes_mpjpe_f64 does all alignment
 * arithmetic in fp64 (distances within 1e-6 mm, ~3x slower).  pred_n / gt_n must be 16-byte aligned. */
int p3d_procrustes_mpjpe(const float* pred_n, const float* gt_n, const double* mean3d_host, const double* std3d_host,
                         int predict_14, int use_procrustes, int64_t N, float* dists_or_null, double* joint_sum,
                         void* stream);
int p3d_procrustes_mpjpe_f64(const float* pred_n, const float* gt_n, const double* mean3d_host, const double* std3d_host,
                             int predict_14, int use_procrustes, int64_t N, float* dists_or_null, double* joint_sum,
                             void* stream);
/* Batched procrustes.compute_similarity_transform on raw poses X,Y[N,J,3] f64 (J<=17):
 * d[N], Z[N,J,3], T[N,9], b[N], c[N,3]; any output may be NULL. */
int p3d_similarity_transform_f64(const double* X, const double* Y, int J, int compute_optimal_scale, int64_t N,
                                 double* d, double* Z, double* T, double* b, double* c, void* stream);

/* Streaming probe (diagnostics): reads n_read_f4 and writes n_write_f4 16-byte words with coalesced streaming accesses;
 * timed by tools/bench_aux.py to give the HBM ceiling at the read:write mix of the preprocessing / evaluation kernels. */
int p3d_debug_stream_mix(const void* src, void* dst, int64_t n_read_f4, int64_t n_write_f4, void* stream);

/* ---------------------------------------------------------------- debug / self-test -----------
 * One-CTA tcgen05 GEMM: C[128,N] = A[128,K] * W[N,K]^T, A/W bf16 row-major (K contiguous),
 * K % 64 == 0, N % 16 == 0, N <= 256.  Exercises TMA + UMMA descriptors + TMEM load in isolation. */
/* globaltimer stamps (ns) of the batch-1 cluster kernel's last run (P3D_LAT_STAMPS=1): [0] entry, [1] after layer 0,
 * [1+l] after hidden layer l, [nlayers] exit. */
int p3d_debug_latency_stamps(p3d_model* m, uint64_t* out_host, int n);
/* Diagnostics: the generic tcgen05 GEMM of the training step (csrc/tc_gemm.cu).  A: a_mn ? [K][M] : [M][K],
 * B: b_mn ? [K][N] : [N][K], both bf16 with pitches lda/ldb (elements); C fp32 [M][ldc].
 * C = alpha * A.B (+bias[n]) (+res[m][n]); split_k != 0 splits K over the grid with fp32 atomics (C must be
 * zeroed); colsum (optional, [2][N] doubles, +=) receives the column sums of C and C^2. */
int p3d_debug_tc_gemm(const void* A, int lda, int a_mn, const void* B, int ldb, int b_mn, float* C, int ldc, int M, int N, int K,
                      const float* bias, const float* res, float alpha, int split_k, double* colsum, void* stream);
/* Diagnostics: the same GEMM under the segment schedule of the bf16x3 GEMMs.  A and B are split pairs: along the
 * operand's contiguous dimension (K of a K-major operand, M / N of an MN-major one) every row holds the hi halves from
 * column 0 and the lo halves from column seg_a / seg_b (multiples of 64); C = alpha * (A.hi B.hi + A.lo B.hi + A.hi B.lo)
 * (+res[m][n]); split_k != 0 splits K over the grid with fp32 atomics (C must be zeroed). */
int p3d_debug_tc_gemm_seg(const void* A, int lda, int a_mn, int seg_a, const void* B, int ldb, int b_mn, int seg_b, float* C, int ldc,
                          int M, int N, int K, const float* res, float alpha, int split_k, void* stream);
/* Diagnostics: cycles of `iters` back-to-back tcgen05.mma 128 x N x 16 on resident shared-memory operands (one CTA).
 * out_dev[0] = cycles to issue, out_dev[1] = cycles until the commit completes. */
int p3d_debug_mma_rate(int N, int iters, int64_t* out_dev, void* stream);
int p3d_debug_umma_gemm(const void* A_bf16, const void* W_bf16, float* C, int N, int K, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* P3D_H_ */
