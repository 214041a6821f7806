#!/usr/bin/env python
"""bench.py - headline benchmark of the B200 hot path (BASELINE.json: "poses/sec (fused MLP inference,
bf16) at 1/2/4/8 B200; batch-1 p50 latency").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one pass of LinearModel(1024, 2, residual, batch_norm, max_norm) inference over one
batch of 2^20 synthetic poses per GPU (configs[1]).  N > 1 is launched by torch.distributed.run, one
process per GPU; the pose batch is sharded by rows (weak scaling: 2^20 poses per GPU), there is no
data-path collective (SURVEY 8e), timing is CUDA events, max over ranks.  Rank 0 prints ONE JSON line.

The same line carries `secondary`: at N = 1 the other BASELINE.json configs (batch sweep, training step, preprocessing,
evaluation, realtime frame); at N > 1 `train_dp` - the data-parallel training step (configs[3]: global batch 64 / 4096 and
4096 rows per GPU, SyncBN + gradient exchange, with the exchange split out) - and `stress_width4096` (configs[4]: 2^21
poses per GPU, 8 x 2^21 = 16 M).

--impl reference times the reference's own CPU implementation of the path.  TensorFlow is not
installable here (no network, SURVEY 8c), so this is the NumPy restatement of linear_model.py's graph
(oracle/mlp_ref.py, "port"), fp32, all host threads, on a bounded sample of the same workload.

--dump-outputs DIR writes, after the timed steps, predictions y of the last timed step as DIR/y.npy (float32; with
N > 1 one file per rank, DIR/y_rank<r>.npy): the same rows in every run, so that two builds run with the same arguments
can be compared output for output (the inputs are seeded too).  Our arm writes a fixed, seeded sample of DUMP_ROWS of
its 2^20 rows; the reference arm writes its first REF_DUMP_ROWS rows, which its sample always holds (the sample size
follows the host's speed, its first rows do not).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "3d-pose-baseline_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

METRIC = "poses/sec (fused MLP inference, bf16)"
UNIT = "poses/s"
L, NL, IN, OUT = 1024, 2, 32, 48
FLOP_PER_POSE = 2 * (IN * L + 2 * NL * L * L + L * OUT)       # 8,552,448 (SURVEY 8d)
B_PER_GPU = 1 << 20
WORKLOAD = "LinearModel(linear_size=1024,num_layers=2,residual,batch_norm,max_norm) inference, batch 2^20 poses/GPU"
DUMP_ROWS = 32768           # 6.3 MB of float32 predictions per rank: 8 ranks stay under 64 MB
REF_DUMP_ROWS = 4096        # the reference arm's smallest sample


def dump_rows(n):
    """Row indices --dump-outputs writes out of n predictions: the same seeded sample in every run."""
    return np.sort(np.random.RandomState(0).choice(n, min(n, DUMP_ROWS), replace=False))


def write_dump(dirname, name, arr):
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, name + ".npy"), np.ascontiguousarray(arr, dtype=np.float32))


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return {"hbm_gbs": d.get("hbm_gbs", 6650.0), "bf16_tflops": d.get("bf16_tflops", 1590.0),
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", 1400.0), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler(threading.Thread):
    """Samples SM clock, power and throttle reasons through NVML every ~5 ms while the timed region runs
    (the nvidia-smi CLI takes ~100 ms per query, longer than a whole step)."""

    def __init__(self, index=0, period=0.005):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.stop_flag = [], threading.Event()
        self.nv = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        while not self.stop_flag.is_set():
            try:
                self.samples.append((nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM),
                                     nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h),
                                     nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0))
            except Exception:
                pass
            self.stop_flag.wait(self.period)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=2)
        if self.nv is None or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "note": "NVML unavailable"}
        nv = self.nv
        bits = 0
        for s in self.samples:
            bits |= s[1]
        names = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                 "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                 "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        return {"sm_mhz": statistics.median(s[0] for s in self.samples), "sm_max_mhz": self.max_sm,
                "reasons": [k for k, v in names.items() if bits & v], "samples": len(self.samples),
                "power_w_max": max(s[2] for s in self.samples)}


# ------------------------------------------------------------------------------------------ reference arm
def cpu_forward(M, p, x, cfg, threads, block=2048):
    """The CPU restatement with ALL host threads busy.  One NumPy call per op over the whole sample keeps only the
    MatMuls multi-threaded (BLAS); the elementwise ops of the graph (BatchNorm, ReLU, residual) run on one core and
    take most of the time (measured here: 10.0 K poses/s).  At inference every pose is independent, so the sample is
    cut into row blocks that are pushed through the same forward by a thread pool, BLAS single-threaded inside a block
    (NumPy releases the GIL in BLAS and ufuncs): 48.6 K poses/s on the same 8 cores, bit-identical outputs."""
    if threads <= 1 or x.shape[0] <= block:
        return M.forward(p, x, cfg, training=False)
    try:
        from threadpoolctl import threadpool_limits
    except Exception:
        return M.forward(p, x, cfg, training=False)
    from concurrent.futures import ThreadPoolExecutor
    with threadpool_limits(limits=1):
        with ThreadPoolExecutor(max_workers=threads) as ex:
            parts = list(ex.map(lambda lo: M.forward(p, x[lo:lo + block], cfg, training=False), range(0, x.shape[0], block)))
    return np.concatenate(parts, axis=0)


def cpu_port_rate(sample, threads, repeats=1):
    """poses/s of the CPU restatement of the reference graph (fp32, op by op like the TF graph)."""
    from oracle import mlp_ref as M
    from oracle import synth
    cfg = M.Config(L, NL, True, True, True)
    p = {k: v.astype(np.float32) for k, v in M.init_params(L, NL, seed=1, bn="trained").items()}
    x, _ = synth.mlp_inputs(sample, seed=0)
    best = None
    for _ in range(repeats):
        t0 = time.perf_counter()
        y = cpu_forward(M, p, x, cfg, threads)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    assert y.dtype == np.float32 and np.isfinite(y).all()
    return sample / best, best


def use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1 to every rank, which would silently run the CPU arm's BLAS on one core:
    raise the BLAS / OpenMP pools back to every core this process may use.  Returns the thread count in effect."""
    want = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        from threadpoolctl import threadpool_info, threadpool_limits
        threadpool_limits(limits=want)
        got = [int(i.get("num_threads", 1)) for i in threadpool_info()]
        return max(got) if got else want
    except Exception:
        return int(os.environ.get("OMP_NUM_THREADS", want))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    threads = use_all_host_threads()
    rate0, _ = cpu_port_rate(16384, threads)
    # size the per-step sample so that the whole run stays within ~4 minutes: at the ~170 K poses/s of a 16-core host
    # that is the full 2^20-pose batch of our arm's config (same_config), fewer poses on a smaller host
    budget = float(os.environ.get("P3D_BENCH_REF_BUDGET_S", "240")) / max(1, args.steps + args.warmup)
    sample = int(min(B_PER_GPU, max(REF_DUMP_ROWS, (rate0 * budget) // 4096 * 4096)))
    from oracle import mlp_ref as M
    from oracle import synth
    cfg = M.Config(L, NL, True, True, True)
    p = {k: v.astype(np.float32) for k, v in M.init_params(L, NL, seed=1, bn="trained").items()}
    x, _ = synth.mlp_inputs(sample, seed=0)
    for _ in range(args.warmup):
        cpu_forward(M, p, x, cfg, threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        y = cpu_forward(M, p, x, cfg, threads)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        write_dump(args.dump_outputs, "y", y[:REF_DUMP_ROWS])
    value = sample * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "note": "TensorFlow not installable (no network): NumPy restatement of the "
                   "reference graph (oracle/mlp_ref.py) on the host cores; each step = a bounded sample",
                   "sample_poses": sample, "full_batch": sample == B_PER_GPU},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{sample} poses per step (of 2^20), fp32, NumPy restatement of the TF graph, row blocks of 2048 "
                                   f"poses over {threads} threads"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------ our arm
def bind_to_gpu_numa(local_rank):
    """Pin this rank's host threads (and with them the pinned staging buffers it is about to allocate: first touch) to the
    NUMA node its GPU hangs off.  With every rank on node 0 the host-buffer step of 8 ranks crosses the socket
    interconnect for half of the GPUs (round 1: end-to-end efficiency 0.27 at N = 8).  Returns what was done."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        with open(f"/sys/bus/pci/devices/{bus}/numa_node") as f:
            node = int(f.read().strip())
        nodes = [d for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit()]
        if node < 0 or len(nodes) <= 1:
            return {"numa_nodes": len(nodes), "gpu_node": node, "bound": False}
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            spec = f.read().strip()
        cpus = set()
        for part in spec.split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return {"numa_nodes": len(nodes), "gpu_node": node, "bound": False}
        os.sched_setaffinity(0, cpus)
        return {"numa_nodes": len(nodes), "gpu_node": node, "bound": True, "cpus": len(cpus)}
    except Exception as e:          # no NVML / sysfs: leave the affinity alone
        return {"bound": False, "error": str(e)[:80]}


def train_dp_measurements(torch, dist, lib, _lib, dev, local_rank, rank, world):
    """BASELINE configs[3] under data parallelism (all ranks take part): LinearModel(1024, 2, residual, batch_norm,
    max_norm) training step, dropout 0.5, Adam, SyncBN, rows of the global batch split over the ranks.  Per case:
    the step (CUDA events, max over ranks), the same rows per GPU WITHOUT any exchange (a single-GPU model on the local
    shard: what the GPU itself needs), the flat gradient all-reduce alone and one standalone SyncBN-sized peer-memory
    exchange; `exchange_us_derived` = step - local step - gradient all-reduce = the SyncBN / loss exchanges as they sit
    inside the step (in-kernel over NVLink peer memory when the tiles fit, waits for the slowest rank included)."""
    from p3d import LinearModel

    def timed(fn, iters, warm=5):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record(); torch.cuda.synchronize()
        ms = torch.tensor([a.elapsed_time(b) / iters], device=dev, dtype=torch.float64)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()) * 1e3          # us

    runs = []
    g = torch.Generator(device=dev).manual_seed(11)
    sptr = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for label, Bg in (("global 64", 64), ("global 4096", 4096), ("4096 rows per GPU", 4096 * world)):
        m = LinearModel(L, NL, True, True, True, Bg, 1e-3, mode="bf16", device=local_rank, seed=1, dist=dist)
        x = torch.randn((Bg, IN), device=dev, generator=g); t = torch.randn((Bg, OUT), device=dev, generator=g)
        dist.broadcast(x, 0); dist.broadcast(t, 0)
        us = timed(lambda: m.step(None, x, t, 0.5, isTraining=True), 20)
        ar = timed(lambda: _lib.check(lib.p3d_debug_dp_part(m._handle, 0, sptr)), 20)
        ex = timed(lambda: _lib.check(lib.p3d_debug_dp_part(m._handle, 1, sptr)), 50)
        peer = bool(getattr(m, "p2p", False))
        m.close()
        rows = Bg // world
        ml = LinearModel(L, NL, True, True, True, rows, 1e-3, mode="bf16", device=local_rank, seed=1)
        xl, tl = x[:rows].contiguous(), t[:rows].contiguous()
        local = timed(lambda: ml.step(None, xl, tl, 0.5, isTraining=True), 20)
        ml.close()
        runs.append({"case": label, "global_batch": Bg, "rows_per_gpu": rows, "us_per_step": round(us, 1),
                     "poses_per_s": round(Bg / (us * 1e-6)), "tflops": round(Bg * 25_591_808 / (us * 1e-6) / 1e12, 2),
                     "local_step_us_no_exchange": round(local, 1), "grad_allreduce_us": round(ar, 1),
                     "one_syncbn_exchange_us_standalone": round(ex, 1),
                     "exchange_us_derived": round(us - local - ar, 1), "peer_memory_exchange": peer})
    return {"config": "dropout keep 0.5, max_norm, Adam, SyncBN; bf16 tcgen05 GEMMs, fp32 master weights; 17.2 MB fp32 gradient",
            "n_gpus": world, "runs": runs}


def stress_measurement(torch, lib, _lib, peaks, dev, local_rank, world, dist):
    """BASELINE configs[4]: linear_size=4096, num_layers=4 (269 MB of bf16 weights > L2), 2^21 poses per GPU (8 GPUs: 16 M
    poses), rows sharded, no collective.  CUDA events, max over ranks."""
    from p3d import LinearModel
    ms_model = LinearModel(4096, 4, True, True, True, 64, 1e-3, seed=3, mode="bf16", device=local_rank)
    Bs = 1 << 21
    g = torch.Generator(device=dev).manual_seed(21)
    xs = torch.randn((Bs, IN), device=dev, generator=g); ys = torch.empty((Bs, OUT), device=dev)
    sptr = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for _ in range(2):
        _lib.check(lib.p3d_model_forward(ms_model._handle, xs.data_ptr(), ys.data_ptr(), Bs, sptr))
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(3):
        _lib.check(lib.p3d_model_forward(ms_model._handle, xs.data_ptr(), ys.data_ptr(), Bs, sptr))
    b.record(); torch.cuda.synchronize()
    ms = torch.tensor([a.elapsed_time(b) / 3], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    flop = 2 * (IN * 4096 + 2 * 4 * 4096 * 4096 + 4096 * OUT)
    ms_model.close()
    del xs, ys
    return {"config": f"linear_size=4096, num_layers=4, residual, batch_norm, max_norm; 2^21 poses per GPU x {world} GPUs = {world << 21} poses",
            "ms": round(ms, 3), "poses_per_s": round(world * Bs / (ms * 1e-3)),
            "tflops_per_gpu": round(Bs * flop / (ms * 1e-3) / 1e12, 1),
            "frac_of_bf16_peak": round(Bs * flop / (ms * 1e-3) / 1e12 / peaks["bf16_tflops"], 4)}


def pinned_array(lib, shape, dtype=np.float32):
    n = int(np.prod(shape)) * np.dtype(dtype).itemsize
    ptr = C.c_void_p()
    rc = lib.p3d_host_alloc(C.byref(ptr), max(n, 16))
    if rc != 0:
        raise RuntimeError("p3d_host_alloc failed")
    arr = np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_byte)), shape=(max(n, 16),))[:n].view(dtype).reshape(shape)
    return arr, ptr


def secondary_measurements(torch, model, lib, _lib, peaks, dev, stream, sptr):
    """The other BASELINE.json configs, measured in the same run (N = 1, rank 0; a few seconds in total):
    inference batch sweep, training step (batch 64 / 4096, both modes), camera-frame preprocessing and
    Procrustes/MPJPE evaluation against the HBM roofline.  CUDA events around back-to-back calls."""
    from oracle import synth
    from p3d import LinearModel, data_utils

    def timed(fn, iters, warm=3):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(iters):
            fn()
        b.record(stream)
        torch.cuda.synchronize()
        return a.elapsed_time(b) / iters          # ms

    out = {}
    g = torch.Generator(device=dev).manual_seed(7)
    sweep = []
    for lg in (0, 1, 3, 4, 6, 8, 10, 12, 14, 16, 18):
        Bs = 1 << lg
        xs = torch.randn((Bs, IN), device=dev, generator=g); ys = torch.empty((Bs, OUT), device=dev)
        ms = timed(lambda: lib.p3d_model_forward(model._handle, xs.data_ptr(), ys.data_ptr(), Bs, sptr), 100 if lg <= 12 else 10)
        tf = Bs * FLOP_PER_POSE / (ms * 1e-3) / 1e12
        sweep.append({"batch": Bs, "us_per_call": round(ms * 1e3, 2), "poses_per_s": round(Bs / (ms * 1e-3)),
                      "frac_of_bf16_peak": round(tf / peaks["bf16_tflops"], 4)})
    out["inference_batch_sweep"] = sweep

    out["stress_width4096"] = stress_measurement(torch, lib, _lib, peaks, dev, dev.index or 0, 1, None)

    train = []
    for Bt, mode in ((64, "bf16"), (4096, "bf16"), (32768, "bf16"), (64, "fp32"), (4096, "fp32")):
        mt = LinearModel(L, NL, True, True, True, Bt, 1e-3, seed=1, mode=mode)
        xt = torch.randn((Bt, IN), device=dev, generator=g); tt = torch.randn((Bt, OUT), device=dev, generator=g)
        ms = timed(lambda: mt.step(None, xt, tt, 0.5, isTraining=True), 20 if mode == "bf16" else 5)
        train.append({"batch": Bt, "mode": mode, "gemms": "tcgen05 bf16, fp32 master weights" if mode == "bf16" else "fp32 FFMA",
                      "us_per_step": round(ms * 1e3, 1), "poses_per_s": round(Bt / (ms * 1e-3)),
                      "tflops": round(Bt * 25_591_808 / (ms * 1e-3) / 1e12, 2)})
        mt.close()
    out["training_step"] = {"config": "dropout keep 0.5, max_norm, Adam, BN batch statistics", "runs": train}

    N = 1 << 20
    cams = synth.cameras(4, seed=3)
    root = torch.randn((N, 1, 3), device=dev, generator=g) * 500
    world_p = (root + torch.randn((N, 32, 3), device=dev, generator=g) * 300).reshape(N, 96).contiguous()
    m2, s2 = np.full(64, 500.0), np.full(64, 150.0)
    m3, s3 = np.zeros(96), np.full(96, 200.0)
    ms = timed(lambda: data_utils.camera_frame_dataset(world_p, cams, m2, s2, m3, s3), 10)
    bts = N * (384 + 512 + 768)
    out["preprocess"] = {"workload": "project_point_radial + world_to_camera + root-centre + normalise, 2^20 poses x 4 cameras",
                         "ms": round(ms, 4), "poses_per_s": round(N / (ms * 1e-3)),
                         "roofline": {"bound": "hbm", "achieved": round(bts / (ms * 1e-3) / 1e9, 1), "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                      "frac": round(bts / (ms * 1e-3) / 1e9 / peaks["hbm_gbs"], 4), "algorithmic_bytes": bts}}
    NE = 4 * N
    gt = torch.randn((NE, 48), device=dev, generator=g)
    pr = gt + 0.2 * torch.randn((NE, 48), device=dev, generator=g)
    sums = torch.zeros(18, dtype=torch.float64, device=dev)
    m3h, s3h = np.ascontiguousarray(m3), np.ascontiguousarray(s3)
    ev = {}
    for use_proc in (1, 0):
        ms = timed(lambda: _lib.check(lib.p3d_procrustes_mpjpe(pr.data_ptr(), gt.data_ptr(), _lib.np_ptr(m3h), _lib.np_ptr(s3h), 0, use_proc,
                                                               NE, None, sums.data_ptr(), sptr)), 10)
        bts = NE * 384
        ev["procrustes_mpjpe" if use_proc else "plain_mpjpe"] = {
            "ms": round(ms, 4), "poses_per_s": round(NE / (ms * 1e-3)),
            "roofline": {"bound": "hbm", "achieved": round(bts / (ms * 1e-3) / 1e9, 1), "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": round(bts / (ms * 1e-3) / 1e9 / peaks["hbm_gbs"], 4), "algorithmic_bytes": bts}}
    ev["workload"] = "un-normalise + (Procrustes) + MPJPE, 4 x 2^20 poses, fp32 kernel"
    out["evaluation"] = ev

    # one realtime frame end to end (openpose_3dpose_sandbox_realtime.py:137-171): host keypoints -> host 3D pose, one
    # cluster-kernel launch over mapped pinned memory; host wall clock through the public Python call
    import time
    from p3d.realtime import RealtimeLifter
    rs = np.random.RandomState(5)
    use2 = np.array([0, 1, 2, 3, 4, 5, 6, 7, 12, 13, 14, 15, 16, 17, 24, 25, 26, 27, 30, 31, 34, 35, 36, 37, 38, 39, 50, 51, 52, 53, 54, 55])
    use3 = np.array([c for j in (1, 2, 3, 6, 7, 8, 12, 13, 14, 15, 17, 18, 19, 25, 26, 27) for c in (3 * j, 3 * j + 1, 3 * j + 2)])
    lifter = RealtimeLifter(model, np.full(64, 500.0), np.full(64, 150.0), use2, m3, s3, use3)
    frames = rs.uniform(100, 900, size=(64, 36)).tolist()
    for i in range(200):
        lifter.step(frames[i % 64])
    lat = []
    for i in range(2000):
        t0 = time.perf_counter()
        lifter.step(frames[i % 64])
        lat.append((time.perf_counter() - t0) * 1e6)
    lat.sort()
    out["realtime_frame"] = {"workload": "OpenPose keypoints (host) -> normalise -> lifter -> un-normalised 3D pose (host), batch 1",
                             "launches_per_frame": 1, "p50_us_wall": round(lat[len(lat) // 2], 2), "p99_us_wall": round(lat[int(0.99 * len(lat))], 2),
                             "frames": len(lat)}
    lifter.close()
    return out


def timed_model(local_rank):
    """The model of the timed path: random-init weights (the model's own kaiming init) + non-trivial BN statistics so
    that the folding is real."""
    from p3d import LinearModel
    model = LinearModel(L, NL, True, True, True, 64, 1e-3, mode="bf16", device=local_rank, seed=1)
    rng = np.random.RandomState(2)
    for name, shape in model.variable_shapes().items():
        leaf = name.rsplit("/", 1)[-1]
        if "Adam" in name or name.endswith("/gradient"):
            continue
        if leaf == "gamma":
            model.set_variable(name, rng.uniform(0.5, 1.5, shape))
        elif leaf == "beta":
            model.set_variable(name, rng.normal(0, 0.1, shape))
        elif leaf == "moving_mean":
            model.set_variable(name, rng.normal(0, 0.5, shape))
        elif leaf == "moving_variance":
            model.set_variable(name, rng.uniform(0.5, 2.0, shape))
    return model


def timed_inputs(torch, dev, rank):
    """The B_PER_GPU input poses of the timed path on this rank."""
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    return torch.randn((B_PER_GPU, IN), device=dev, generator=g)


def run_ours(args):
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: libp3d has no CPU fallback"}))
        return 2
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    numa = bind_to_gpu_numa(local_rank) if world > 1 else {"bound": False, "note": "single rank: affinity left alone"}
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from p3d import _lib
    lib = _lib.lib
    peaks = load_peaks()

    model = timed_model(local_rank)
    B = B_PER_GPU
    x = timed_inputs(torch, dev, rank)
    t = torch.zeros((B, OUT), device=dev)
    y = torch.empty((B, OUT), device=dev)
    stream = torch.cuda.current_stream()
    sptr = C.c_void_p(stream.cuda_stream)

    def step():
        _lib.check(lib.p3d_model_forward(model._handle, x.data_ptr(), y.data_ptr(), B, sptr))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    warm = max(3, args.warmup)
    for _ in range(warm):
        step()
    # ---- device-resident timing (value): K steps between two events, max over ranks
    sampler = ClockSampler(local_rank) if rank == 0 else None
    barrier()
    if sampler:
        sampler.start()
    lib.p3d_profile_enable(1)
    launches0 = lib.p3d_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    barrier()
    elapsed_ms = e0.elapsed_time(e1)
    launches = int(lib.p3d_launch_count() - launches0)
    kms, kn = C.c_double(), C.c_int64()
    lib.p3d_profile_read(C.byref(kms), C.byref(kn))
    lib.p3d_profile_enable(0)
    dumped = y[torch.from_numpy(dump_rows(B)).to(dev)].cpu().numpy() if args.dump_outputs else None
    clocks = sampler.summary() if sampler else None
    el = torch.tensor([elapsed_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(el, op=dist.ReduceOp.MAX)
    elapsed_ms = float(el.item())
    value = world * B * args.steps / (elapsed_ms * 1e-3)

    # ---- end-to-end: model.step() with pinned HOST buffers, H2D of x and decoder_outputs + D2H of y inside
    xh, xh_ptr = pinned_array(lib, (B, IN))
    th, th_ptr = pinned_array(lib, (B, OUT))
    yh_buf, yh_ptr = pinned_array(lib, (B, OUT))
    xh[:] = x.cpu().numpy()
    th[:] = 0.0
    e2e_steps = max(2, min(args.steps, 5))
    model.step(None, xh, th, 1.0, isTraining=False, out=yh_buf)   # warm (allocates the pipeline buffers)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        loss, _, yh = model.step(None, xh, th, 1.0, isTraining=False, out=yh_buf)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    e2 = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(e2, op=dist.ReduceOp.MAX)
    e2e_value = world * B * e2e_steps / float(e2.item())
    mine = torch.tensor([B * (IN + OUT) * 4 * e2e_steps / e2e_s / 1e9, (B * OUT * 4) * e2e_steps / e2e_s / 1e9], device=dev, dtype=torch.float64)
    per_rank = [torch.zeros(2, device=dev, dtype=torch.float64) for _ in range(world)]
    if world > 1:
        dist.all_gather(per_rank, mine)
    else:
        per_rank = [mine]
    per_rank = [{"rank": r, "h2d_gbs": round(float(v[0]), 2), "d2h_gbs": round(float(v[1]), 2)} for r, v in enumerate(per_rank)]
    ok = bool(np.isfinite(yh[:1024]).all()) and bool(np.allclose(yh[:4096], y[:4096].cpu().numpy(), atol=1e-5))
    # the same call without a target (decoder_outputs=None, an extension of the reference contract: its callers pass
    # zeros when they only want predictions): 128 B per pose up instead of 320
    model.step(None, xh, None, 1.0, isTraining=False, out=yh_buf)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        model.step(None, xh, None, 1.0, isTraining=False, out=yh_buf)
    torch.cuda.synchronize()
    e3 = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(e3, op=dist.ReduceOp.MAX)
    e2e_nt_value = world * B * e2e_steps / float(e3.item())
    ok = ok and bool(np.allclose(yh_buf[:4096], y[:4096].cpu().numpy(), atol=1e-5))

    # ---- batch-1 latency (p50) of the same model: CUDA events per call + host wall clock
    lat = None
    if rank == 0:
        x1, t1 = x[:1].contiguous(), t[:1].contiguous()
        y1 = torch.empty((1, OUT), device=dev)
        for _ in range(200):
            _lib.check(lib.p3d_model_forward(model._handle, x1.data_ptr(), y1.data_ptr(), 1, sptr))
        torch.cuda.synchronize()
        ev, wall = [], []
        LAT_ITERS = 10000                                   # SURVEY 8d: >= 10 k iterations after warm-up
        for _ in range(LAT_ITERS):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            w0 = time.perf_counter()
            a.record(stream)
            _lib.check(lib.p3d_model_forward(model._handle, x1.data_ptr(), y1.data_ptr(), 1, sptr))
            b.record(stream)
            b.synchronize()
            wall.append((time.perf_counter() - w0) * 1e6)
            ev.append(a.elapsed_time(b) * 1e3)
        # ... and back to back (no host in between): what one call occupies the device for
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(2000):
            lib.p3d_model_forward(model._handle, x1.data_ptr(), y1.data_ptr(), 1, sptr)
        b.record(stream); b.synchronize()
        lat = {"p50_us_device": statistics.median(ev), "p50_us_wall": statistics.median(wall),
               "p99_us_wall": sorted(wall)[int(0.99 * len(wall))], "iters": LAT_ITERS,
               "back_to_back_us_per_call": a.elapsed_time(b) * 1e3 / 2000,
               "kernel": "latency_grid_kernel<1>: 128 CTAs (cooperative), 8.56 MB of bf16 weights pulled by the whole chip, "
                         "activations exchanged through self-validating {value, tag} words",
               "note": "p50_us_device brackets ONE call with two CUDA events (includes the launch); back_to_back is the "
                       "device time per call"}

    # ---- CPU baseline (rank 0, N == 1 only): the oracle port on the host cores, bounded sample
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = use_all_host_threads()
        r0, _ = cpu_port_rate(16384, threads)
        sample = int(min(B, max(4096, (r0 * 15.0) // 4096 * 4096)))          # ~15 s of CPU work
        rate, secs = cpu_port_rate(sample, threads)
        cpu = {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": f"{sample} of 2^20 poses, fp32 NumPy restatement of the TF graph, row blocks of 2048 poses over "
                         f"{threads} threads, {secs:.1f} s"}

    secondary = None
    if rank == 0 and world == 1 and not args.no_secondary:
        secondary = secondary_measurements(torch, model, lib, _lib, peaks, dev, stream, sptr)
    if world > 1 and not args.no_secondary:          # every rank takes part; rank 0 reports
        secondary = {"train_dp": train_dp_measurements(torch, dist, lib, _lib, dev, local_rank, rank, world),
                     "stress_width4096": stress_measurement(torch, lib, _lib, peaks, dev, local_rank, world, dist)}

    if rank == 0:
        k_ms = kms.value / max(1, kn.value)
        achieved = B * FLOP_PER_POSE / (k_ms * 1e-3) / 1e12
        # dram__bytes of ONE launch of the timed kernel from an ncu capture (tools/capture_traffic.sh); the file names the
        # source it was captured from - a capture of another version of the kernel is refused
        traffic, traffic_note = None, "no capture"
        tpath = os.path.join(ROOT, "profiles", "mlp_tc_traffic.json")
        if os.path.exists(tpath):
            import hashlib
            with open(tpath) as f:
                tj = json.load(f)
            with open(os.path.join(ROOT, "3d-pose-baseline_b200", "csrc", "mlp_tc.cu"), "rb") as f:
                sha = hashlib.sha256(f.read()).hexdigest()[:16]
            if tj.get("kernel_src_sha16") == sha:
                traffic, traffic_note = tj.get("dram_bytes_per_launch"), f"ncu capture of {tj.get('when', '?')} ({tj.get('capture', '')})"
            else:
                traffic_note = f"stale capture refused (made from mlp_tc.cu {tj.get('kernel_src_sha16')}, built from {sha})"
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm,
            "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": WORKLOAD, "global_batch": world * B, "sharding": f"rows, {world} x 2^20, no collective",
                       "l2": "x (134 MB) + y (201 MB) per step exceed the 126 MB L2; no flush needed",
                       "weights": "random init (kaiming), BN statistics non-trivial and folded"},
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
                         "frac": achieved / peaks["bf16_tflops"], "traffic": traffic, "traffic_source": traffic_note,
                         "algorithmic_bytes_per_launch": B * (128 + 192),
                         "peak_source": peaks["source"] + " burst bf16 (MEASURED_PEAKS.json)",
                         "frac_of_sustained": achieved / peaks["bf16_tflops_sustained"],
                         "kernel": "mlp_forward_tc_kernel", "kernel_ms": k_ms, "kernel_launches": int(kn.value),
                         "flop_per_launch": B * FLOP_PER_POSE},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": B * (IN + OUT) * 4,
                    "d2h_bytes_per_step": B * OUT * 4 + 4, "steps": e2e_steps, "outputs_match_device_path": ok,
                    "per_rank": per_rank, "host_numa": numa,
                    "predictions_only": {"value": e2e_nt_value, "unit": UNIT, "h2d_bytes_per_step": B * IN * 4,
                                         "api": "LinearModel.step(None, x_pinned, None, 1.0, isTraining=False, out=y_pinned)"},
                    "api": "LinearModel.step(None, x_pinned, dec_out_pinned, 1.0, isTraining=False, out=y_pinned)"},
            "gpu_launches": launches,
            "clocks": clocks,
            "latency_batch1": lat,
        }
        if cpu:
            line["cpu_baseline"] = cpu
        if secondary:
            line["secondary"] = secondary
        print(json.dumps(line))
    if dumped is not None:
        write_dump(args.dump_outputs, "y" if world == 1 else f"y_rank{rank}", dumped)
    lib.p3d_host_free(yh_ptr)
    lib.p3d_host_free(xh_ptr)
    lib.p3d_host_free(th_ptr)
    model.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the batch sweep / training / preprocessing / evaluation lines")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a fixed sample of the last timed step's predictions to DIR/y.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    # The contract is ONE JSON line on stdout: libraries (NCCL's version banner, torchrun notices) also write to
    # fd 1, so fd 1 is pointed at stderr for the duration of the run and the line goes to the saved descriptor.
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    real_stdout = os.fdopen(saved, "w")
    import builtins
    _print = builtins.print

    def emit(*a, **k):
        if a and isinstance(a[0], str) and a[0].startswith("{"):
            _print(*a, file=real_stdout, **k)
            real_stdout.flush()
        else:
            _print(*a, **k)
    builtins.print = emit
    try:
        if args.impl == "reference":
            return run_reference(args)
        return run_ours(args)
    finally:
        builtins.print = _print


if __name__ == "__main__":
    sys.exit(main())
