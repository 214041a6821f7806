"""Drop-in for the reference's `linear_model.LinearModel` (src/linear_model.py:31-300) on B200.

Same constructor flags, same `step()` / `get_all_batches()` contract; the TensorFlow graph and session
are replaced by libp3d.so (hand-written sm_100a CUDA).  There is no TensorFlow, Triton or CPU path.

Differences that are visible to a caller, all additive:
  * `session` is accepted and ignored (there is no tf.Session).
  * keyword-only extras: `mode` ('bf16' tensor-core path, 'fp32', 'bf16x3': fp32 accuracy on the tensor cores
    for inference, trained like 'fp32', or 'fp16': bf16's paths on fp16 operands, <= 2e-3 row-wise error,
    trained like 'bf16'), `train_matmul` (None: the mode's own training route; 'bf16x3' with mode
    'fp32' or 'bf16x3': the training step's MatMuls as three split-bf16 tensor-core products), `device`, `seed`, `dist`.
  * `step()` also accepts torch CUDA tensors (fp32) and then returns torch tensors without any host copy.
  * summaries are `Summary(tag, value)` tuples that serialize to the TF `Summary` protobuf on demand; with a
    `summaries_dir` the train/test writers append real TensorBoard event files (p3d/summary.py), without one they
    only collect what they are given.
"""
from __future__ import annotations

import collections
import ctypes as C
import math
import os

import numpy as np

from . import _lib
from ._lib import lib, check
from .summary import FileWriter, Summary


class _Evaluable:
    """Stands in for a tf.Variable/Tensor that callers `.eval()` (predict_3dpose.py:228,288)."""

    def __init__(self, getter):
        self._getter = getter

    def eval(self, session=None):
        return self._getter()

    def __float__(self):
        return float(self._getter())

    def __int__(self):
        return int(self._getter())


class _NullWriter:
    """train_writer/test_writer when no summaries_dir was given: summaries are collected, nothing is written."""

    def __init__(self, path):
        self.path = path
        self.events = []

    def add_summary(self, summary, step=None):
        self.events.append((step, summary))

    def add_graph(self, graph, global_step=None):
        pass

    def flush(self):
        pass

    def close(self):
        pass


def kaiming(shape, rng: np.random.RandomState, dtype=np.float32):
    """linear_model.py:17-29: truncated_normal(shape) * sqrt(2/shape[0]); samples beyond 2 sigma re-drawn."""
    v = rng.standard_normal(int(np.prod(shape)))
    bad = np.abs(v) > 2.0
    while bad.any():
        v[bad] = rng.standard_normal(int(bad.sum()))
        bad = np.abs(v) > 2.0
    return (v.reshape(shape) * math.sqrt(2.0 / float(shape[0]))).astype(dtype)


def shard_rows(n_rows: int, rank: int, world: int):
    """Contiguous row block of `rank` when n_rows poses are split over `world` GPUs (SURVEY 8e)."""
    base, rem = divmod(n_rows, world)
    start = rank * base + min(rank, rem)
    return start, start + base + (1 if rank < rem else 0)


class _Saver(object):
    """tf.train.Saver(tf.global_variables(), max_to_keep=10) of the reference (linear_model.py:151) writing and
    reading TensorFlow's checkpoint format without TensorFlow (p3d/checkpoint.py):
        model.saver.save(sess, os.path.join(train_dir, 'checkpoint'), global_step=step)   # predict_3dpose.py:328
        model.saver.restore(sess, ckpt.model_checkpoint_path)                             # predict_3dpose.py:180
    Variables carry the TF1 graph's names; `global_step` is an int32 scalar, `learning_rate` the base rate,
    `beta1_power` / `beta2_power` the optimizer's non-slot variables (beta^(global_step + 1))."""

    def __init__(self, model, max_to_keep=10):
        self._model, self.max_to_keep = model, max_to_keep

    def save(self, sess, save_path, global_step=None):
        from . import checkpoint
        m = self._model
        prefix = save_path if global_step is None else "{0}-{1}".format(save_path, int(global_step))
        t = {}
        for name, v in m.get_variables(include_optimizer=True).items():
            t[name] = np.int32(int(v)) if name == "global_step" else np.asarray(v, dtype=np.float32)
        g = int(m.global_step.eval())
        t["learning_rate"] = np.float32(m._lr0)
        t["beta1_power"] = np.float32(0.9 ** (g + 1))
        t["beta2_power"] = np.float32(0.999 ** (g + 1))
        checkpoint.write_bundle(prefix, t)
        checkpoint.update_checkpoint_state(os.path.dirname(os.path.abspath(prefix)), prefix, self.max_to_keep)
        return prefix

    def restore(self, sess, save_path):
        from . import checkpoint
        m = self._model
        t = checkpoint.read_bundle(save_path)          # ValueError if <save_path>.index is missing (predict_3dpose.py:175)
        shapes = m.variable_shapes()
        wanted = [n for n in m.get_variable_names(include_optimizer=True)]
        missing = [n for n in wanted if n not in t and "Adam" not in n]
        if missing:
            raise ValueError("checkpoint {0} lacks variables: {1}".format(save_path, ", ".join(missing[:4])))
        for n in wanted:
            if n not in t:
                continue                                 # a checkpoint saved without optimizer slots keeps the fresh ones
            a = np.asarray(t[n])
            if n != "global_step" and tuple(a.shape) != tuple(shapes[n]):
                raise ValueError("variable {0}: checkpoint shape {1} != model shape {2}".format(n, a.shape, shapes[n]))
            m.set_variable(n, a.astype(np.float32))      # fp16 checkpoints (--use_fp16) widen here
        if "learning_rate" in t:
            m._set_base_learning_rate(float(np.asarray(t["learning_rate"])))


class LinearModel(object):
    """A simple Linear+RELU model (linear_model.py:31)."""

    def __init__(self, linear_size, num_layers, residual, batch_norm, max_norm, batch_size, learning_rate,
                 summaries_dir=None, predict_14=False, dtype=np.float32, *, mode="bf16", device=0, seed=None,
                 dist=None, train_matmul=None):
        self.HUMAN_2D_SIZE = 16 * 2                                  # linear_model.py:60
        self.HUMAN_3D_SIZE = 14 * 3 if predict_14 else 16 * 3         # :69
        self.input_size = self.HUMAN_2D_SIZE
        self.output_size = self.HUMAN_3D_SIZE
        self.linear_size = int(linear_size)
        self.num_layers = int(num_layers)
        self.residual, self.batch_norm, self.max_norm = bool(residual), bool(batch_norm), bool(max_norm)
        self.batch_size = int(batch_size)
        self.predict_14 = bool(predict_14)
        self.mode = mode
        self.device = int(device)
        self._lr0 = float(learning_rate)
        self._seed = int(seed) if seed is not None else int.from_bytes(os.urandom(4), "little")
        self._handle = None
        modes = {"bf16": _lib.MODE_BF16, "fp32": _lib.MODE_FP32, "bf16x3": _lib.MODE_BF16X3, "fp16": _lib.MODE_FP16}
        if mode not in modes:
            raise ValueError("mode must be 'bf16', 'fp32', 'bf16x3' or 'fp16'")
        # the arithmetic of the training step's MatMuls (p3d_model_set_train_matmul); with `dist`, every rank passes the
        # same value
        if train_matmul not in (None, "bf16x3"):
            raise ValueError("train_matmul must be None or 'bf16x3'")
        if train_matmul is not None and mode in ("bf16", "fp16"):
            raise ValueError("train_matmul='bf16x3' needs mode 'fp32' or 'bf16x3' (bf16 and fp16 models train on bf16 tensor cores)")
        self.train_matmul = train_matmul
        # Summary writers for train and test runs (linear_model.py:80-82)
        if summaries_dir:
            self.train_writer = FileWriter(os.path.join(summaries_dir, "train"))
            self.test_writer = FileWriter(os.path.join(summaries_dir, "test"))
        else:
            self.train_writer, self.test_writer = _NullWriter("train"), _NullWriter("test")

        cfg = _lib.Cfg(self.linear_size, self.num_layers, int(self.residual), int(self.batch_norm),
                       int(self.max_norm), int(self.predict_14),
                       modes[mode], self.device, self._lr0)
        h = C.c_void_p()
        check(lib.p3d_model_create(C.byref(cfg), C.byref(h)))
        self._handle = h
        if train_matmul == "bf16x3":
            check(lib.p3d_model_set_train_matmul(self._handle, _lib.TRAIN_MATMUL_BF16X3))
        self.global_step = _Evaluable(lambda: int(lib.p3d_model_global_step(self._handle)))
        self.learning_rate = _Evaluable(self._decayed_lr)
        self._names = self._query_names()
        self._init_variables(np.random.RandomState(self._seed))
        self.saver = _Saver(self, max_to_keep=10)                     # linear_model.py:151
        self.err_mm = np.float32(0.0)                                  # :133, the 'error_mm' placeholder
        # data parallel (one process per GPU, torch.distributed for the rendezvous only)
        self.rank, self.world = 0, 1
        if dist is not None:
            self._attach_dist(dist)

    # ------------------------------------------------------------------ variables
    def _query_names(self):
        out = collections.OrderedDict()
        n = lib.p3d_model_param_count(self._handle)
        buf = C.create_string_buffer(256)
        numel = C.c_size_t()
        for i in range(n):
            check(lib.p3d_model_param_name(self._handle, i, buf, 256, C.byref(numel)))
            out[buf.value.decode()] = int(numel.value)
        return out

    def variable_shapes(self):
        """TF variable name -> shape, weights [in,out] (what tf.train.Saver would hold)."""
        L, shapes = self.linear_size, collections.OrderedDict()
        for name, numel in self._names.items():
            base = name.replace("/Adam_1", "").replace("/Adam", "").replace("/gradient", "")
            leaf = base.rsplit("/", 1)[-1]
            if leaf == "w1":
                shapes[name] = (self.input_size, L)
            elif leaf == "w4":
                shapes[name] = (L, self.output_size)
            elif leaf.startswith("w"):
                shapes[name] = (L, L)
            elif name == "global_step":
                shapes[name] = ()
            else:
                shapes[name] = (numel,)
        return shapes

    def _init_variables(self, rng):
        """kaiming for every weight AND bias (linear_model.py:106-107,121-122,176-188); BN at TF defaults."""
        for name, shape in self.variable_shapes().items():
            leaf = name.rsplit("/", 1)[-1]
            if "Adam" in name or name == "global_step" or name.endswith("/gradient"):
                continue
            if leaf[0] in "wb" and "batch_normalization" not in name:
                self.set_variable(name, kaiming(shape, rng))

    def set_variable(self, name, value):
        a = np.ascontiguousarray(np.asarray(value, dtype=np.float32)).reshape(-1)
        check(lib.p3d_model_set_param_host(self._handle, name.encode(), _lib.np_ptr(a), a.size))

    def get_variable(self, name):
        shape = self.variable_shapes()[name]
        a = np.empty(self._names[name], dtype=np.float32)
        check(lib.p3d_model_get_param_host(self._handle, name.encode(), _lib.np_ptr(a), a.size))
        return a.reshape(shape) if shape != () else a[0]

    def get_variables(self, include_optimizer=False):
        return {n: self.get_variable(n) for n in self._names
                if not n.endswith("/gradient") and (include_optimizer or ("Adam" not in n and n != "global_step"))}

    def get_variable_names(self, include_optimizer=False):
        return [n for n in self._names
                if not n.endswith("/gradient") and (include_optimizer or ("Adam" not in n and n != "global_step"))]

    def get_gradients(self):
        """Gradients of the last training step by variable name (model.gradients, linear_model.py:143-144)."""
        return {n[:-len("/gradient")]: self.get_variable(n) for n in self._names if n.endswith("/gradient")}

    def set_variables(self, values):
        for n, v in values.items():
            self.set_variable(n, v)

    def prepare_inference(self):
        """Fold clip_by_norm and the BatchNorm statistics into the packed inference weights now, on the current torch
        stream (p3d_model_prepare_inference).  Inference does this by itself after set_variable, restore or a training
        step, but not inside a CUDA graph capture; the fold rewrites the packed weights in place, so graphs captured
        earlier see the new weights on their next replay.  Call it outside any capture."""
        torch = _lib.require_cuda()
        with torch.cuda.device(self.device):
            check(lib.p3d_model_prepare_inference(self._handle, _lib.current_stream()))

    # tf.train.Saver stand-in (linear_model.py:151; predict_3dpose.py:158-186,328): one .npz keyed by TF names
    def save(self, path):
        path = path if path.endswith(".npz") else path + ".npz"      # np.savez would append it silently
        np.savez(path, **{k.replace("/", "|"): v for k, v in self.get_variables(include_optimizer=True).items()})
        return path

    def restore(self, path):
        path = path if path.endswith(".npz") or os.path.exists(path) else path + ".npz"
        if not os.path.exists(path):
            raise ValueError("Asked to load checkpoint {0}, but it does not seem to exist".format(path))
        with np.load(path) as z:
            for k in z.files:
                self.set_variable(k.replace("|", "/"), z[k])

    def _set_base_learning_rate(self, lr):
        """The `learning_rate` variable of a restored checkpoint replaces the constructor's value (linear_model.py:86)."""
        a = np.array([lr], dtype=np.float32)
        check(lib.p3d_model_set_param_host(self._handle, b"learning_rate", _lib.np_ptr(a), 1))
        self._lr0 = float(a[0])

    def _decayed_lr(self):
        """tf.train.exponential_decay(lr, global_step, 100000, 0.96) (linear_model.py:86-90)."""
        return np.float32(self._lr0) * np.float32(0.96) ** np.float32(int(self.global_step) / 100000.0)

    # ------------------------------------------------------------------ distributed
    def _attach_dist(self, dist):
        torch = _lib.require_cuda()
        self.rank, self.world = dist.get_rank(), dist.get_world_size()
        if self.world == 1:
            return
        ident = np.zeros(128, dtype=np.uint8)
        if self.rank == 0:
            check(lib.p3d_nccl_unique_id(_lib.np_ptr(ident)))
        t = torch.from_numpy(ident).cuda(self.device) if dist.get_backend() == "nccl" else torch.from_numpy(ident)
        dist.broadcast(t, src=0)
        ident = t.cpu().numpy().copy()
        # one dropout seed for the whole job: masks are keyed by (seed, step, layer, GLOBAL row, column), so with rank 0's
        # seed a data-parallel step draws exactly the mask of the single-device step on the global batch
        sd = torch.tensor([self._seed], dtype=torch.int64)
        sd = sd.cuda(self.device) if dist.get_backend() == "nccl" else sd
        dist.broadcast(sd, src=0)
        self._seed = int(sd.item())
        # identical initial variables on every rank
        for name in self._names:
            if name == "global_step" or name.endswith("/gradient"):
                continue
            v = torch.from_numpy(np.asarray(self.get_variable(name), dtype=np.float32).copy())
            if dist.get_backend() == "nccl":
                v = v.cuda(self.device)
            dist.broadcast(v, src=0)
            self.set_variable(name, v.cpu().numpy())
        check(lib.p3d_model_attach_nccl(self._handle, _lib.np_ptr(ident), self.rank, self.world))
        self._dist = dist
        # single node: the small SyncBN / loss reductions go over NVLink peer memory (CUDA IPC); NCCL otherwise
        self.p2p = False
        if os.environ.get("P3D_P2P", "1") != "0" and int(os.environ.get("LOCAL_WORLD_SIZE", self.world)) == self.world:
            mine = np.zeros(128, dtype=np.uint8)
            check(lib.p3d_model_p2p_handle(self._handle, _lib.np_ptr(mine)))
            hs = [torch.zeros(128, dtype=torch.uint8, device=torch.device("cuda", self.device) if dist.get_backend() == "nccl" else "cpu")
                  for _ in range(self.world)]
            src = torch.from_numpy(mine)
            dist.all_gather(hs, src.cuda(self.device) if dist.get_backend() == "nccl" else src)
            allh = np.ascontiguousarray(np.concatenate([h.cpu().numpy() for h in hs]))
            self.p2p = lib.p3d_model_p2p_attach(self._handle, _lib.np_ptr(allh), self.rank, self.world) == 0
            ok = torch.tensor([1 if self.p2p else 0], device=torch.device("cuda", self.device) if dist.get_backend() == "nccl" else "cpu")
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)          # all ranks or none: every rank acts on the reduced flag
            if int(ok.item()) == 0:
                check(lib.p3d_model_p2p_detach(self._handle))   # closes what this rank had opened; the step keeps NCCL
                self.p2p = False

    # ------------------------------------------------------------------ step
    def step(self, session, encoder_inputs, decoder_outputs, dropout_keep_prob, isTraining=True, *,
             dropout_mask=None, out=None):
        """Run a step of the model feeding the given inputs (linear_model.py:203-245).

        Returns (loss, loss_summary, learning_rate_summary, outputs) when isTraining else
        (loss, loss_summary, outputs).  NumPy in -> NumPy out; torch CUDA tensors in -> torch out.
        `out`: optional preallocated fp32 [B,out] NumPy array for the evaluation outputs (e.g. pinned
        memory from p3d_host_alloc, which lets the device->host copy overlap the compute)."""
        torch = _lib.require_cuda()
        is_torch = hasattr(encoder_inputs, "is_cuda")
        # Extension of the reference contract: decoder_outputs=None for isTraining=False (the reference's callers pass
        # zeros when they only want predictions, openpose_3dpose_sandbox_realtime.py:166-168): nothing is uploaded for
        # it and the returned loss is 0.
        no_target = decoder_outputs is None
        if no_target and isTraining:
            raise ValueError("decoder_outputs is required for a training step")
        if is_torch:
            x, t = encoder_inputs, decoder_outputs
            if not (x.is_cuda and x.dtype == torch.float32) or not (no_target or (t.is_cuda and t.dtype == torch.float32)):
                raise ValueError("torch inputs must be float32 CUDA tensors")
            x = x.contiguous()
            t = None if no_target else t.contiguous()
        else:
            x = np.ascontiguousarray(np.asarray(encoder_inputs, dtype=np.float32))   # the TF feed casts fp64 -> fp32
            t = None if no_target else np.ascontiguousarray(np.asarray(decoder_outputs, dtype=np.float32))
        if x.ndim != 2 or x.shape[1] != self.input_size:
            raise ValueError("encoder_inputs must be [B,%d]" % self.input_size)
        if not no_target and (t.ndim != 2 or t.shape[1] != self.output_size or t.shape[0] != x.shape[0]):
            raise ValueError("decoder_outputs must be [B,%d]" % self.output_size)
        B = int(x.shape[0])

        if not isTraining:
            if is_torch:
                with torch.cuda.device(self.device):
                    y = torch.empty((B, self.output_size), dtype=torch.float32, device=x.device)
                    loss = torch.zeros((), dtype=torch.float32, device=x.device)
                    st = _lib.current_stream()
                    check(lib.p3d_model_forward(self._handle, x.data_ptr(), y.data_ptr(), B, st))
                    if B and not no_target:
                        check(lib.p3d_model_mse(self._handle, y.data_ptr(), t.data_ptr(), B, loss.data_ptr(), st))
                self._last_outputs, self._last_loss = y, loss
                return loss, Summary("loss/loss", loss), y
            if out is not None:
                if out.shape != (B, self.output_size) or out.dtype != np.float32 or not out.flags.c_contiguous:
                    raise ValueError("out must be a C-contiguous float32 [B,%d] array" % self.output_size)
                y = out
            else:
                y = np.empty((B, self.output_size), dtype=np.float32)
            loss = C.c_float(0.0)
            check(lib.p3d_model_step_eval_host(self._handle, _lib.np_ptr(x), None if no_target else _lib.np_ptr(t),
                                               _lib.np_ptr(y), C.byref(loss), B))
            self._last_outputs, self._last_loss = y, np.float32(loss.value)
            return np.float32(loss.value), Summary("loss/loss", np.float32(loss.value)), y

        # ---- training
        keep = float(dropout_keep_prob)
        with torch.cuda.device(self.device):
            dev = torch.device("cuda", self.device)
            xd = x if is_torch else torch.from_numpy(x).to(dev)
            td = t if is_torch else torch.from_numpy(t).to(dev)
            gB, row0 = B, 0
            if self.world > 1:          # every rank is handed the global batch; it trains on its row block
                lo, hi = shard_rows(B, self.rank, self.world)
                xd, td, row0 = xd[lo:hi].contiguous(), td[lo:hi].contiguous(), lo
            Bl = int(xd.shape[0])
            y = torch.empty((Bl, self.output_size), dtype=torch.float32, device=dev)
            scal = torch.zeros(2, dtype=torch.float32, device=dev)
            mask_ptr = None
            if dropout_mask is not None:      # tests inject the keep-mask: uint8 [nhidden][B][L]
                md = torch.as_tensor(np.ascontiguousarray(dropout_mask, dtype=np.uint8)).to(dev)
                if self.world > 1:
                    md = md[:, row0:row0 + Bl].contiguous()
                mask_ptr = md.data_ptr()
            check(lib.p3d_model_train_step(self._handle, xd.data_ptr(), td.data_ptr(), Bl, keep,
                                           C.c_uint64(self._seed & 0xFFFFFFFFFFFFFFFF), mask_ptr, gB, row0,
                                           scal.data_ptr(), scal.data_ptr() + 4, y.data_ptr(), _lib.current_stream()))
            if self.world > 1:
                # the outputs of the global batch: normally they travelled with the gradient exchange (one D2D copy)
                yg = torch.empty((B, self.output_size), dtype=torch.float32, device=dev)
                rc = lib.p3d_model_gathered_outputs(self._handle, yg.data_ptr(), B, _lib.current_stream())
                if rc == 1:
                    parts = [torch.empty((shard_rows(B, r, self.world)[1] - shard_rows(B, r, self.world)[0],
                                          self.output_size), dtype=torch.float32, device=dev) for r in range(self.world)]
                    self._dist.all_gather(parts, y)
                    yg = torch.cat(parts, 0)
                else:
                    check(rc)
                y = yg
            if is_torch:
                self._last_outputs, self._last_loss = y, scal[0]
                return scal[0], Summary("loss/loss", scal[0]), Summary("learning_rate/learning_rate", scal[1]), y
            s = scal.cpu().numpy()
            yh = y.cpu().numpy()
            self._last_outputs, self._last_loss = yh, np.float32(s[0])
            return (np.float32(s[0]), Summary("loss/loss", np.float32(s[0])),
                    Summary("learning_rate/learning_rate", np.float32(s[1])), yh)

    def train_epoch(self, encoder_inputs, decoder_outputs, dropout_keep_prob, shuffle=True, perm=None):
        """The batch loop of the reference's train() (src/predict_3dpose.py:231-259) without the host in it:
        `encoder_inputs` [n,32] / `decoder_outputs` [n,out] are the concatenated training set (what
        get_all_batches builds, linear_model.py:266-300; NumPy or torch CUDA), permuted (np.random.permutation
        as in :309 unless `perm` is given or shuffle=False), cut into n // batch_size batches (the tail is
        dropped, :311-313) and stepped on the device, one replayed CUDA graph per batch.
        Returns (losses[n_batches], last learning rate) - NumPy for NumPy inputs, torch otherwise."""
        torch = _lib.require_cuda()
        if self.world > 1:
            raise RuntimeError("train_epoch is single-GPU; data-parallel training steps through step()")
        is_torch = hasattr(encoder_inputs, "is_cuda")
        dev = torch.device("cuda", self.device)
        with torch.cuda.device(self.device):
            X = (encoder_inputs if is_torch else torch.from_numpy(np.ascontiguousarray(encoder_inputs, dtype=np.float32))).to(dev, torch.float32).contiguous()
            T = (decoder_outputs if is_torch else torch.from_numpy(np.ascontiguousarray(decoder_outputs, dtype=np.float32))).to(dev, torch.float32).contiguous()
            n = int(X.shape[0])
            if X.dim() != 2 or X.shape[1] != self.input_size or T.shape != (n, self.output_size):
                raise ValueError("expected [n,%d] inputs and [n,%d] outputs" % (self.input_size, self.output_size))
            nb = n // self.batch_size
            pd = None
            if perm is not None:
                pd = torch.as_tensor(np.asarray(perm, dtype=np.int64)).to(dev)
            elif shuffle:
                pd = torch.from_numpy(np.random.permutation(n).astype(np.int64)).to(dev)
            losses = torch.zeros(max(nb, 1), dtype=torch.float32, device=dev)
            lr = torch.zeros(1, dtype=torch.float32, device=dev)
            if nb:
                check(lib.p3d_model_train_epoch(self._handle, X.data_ptr(), T.data_ptr(), n, pd.data_ptr() if pd is not None else None,
                                                self.batch_size, float(dropout_keep_prob), C.c_uint64(self._seed & 0xFFFFFFFFFFFFFFFF),
                                                losses.data_ptr(), lr.data_ptr(), _lib.current_stream()))
            losses = losses[:nb]
        if is_torch:
            return losses, lr[0]
        return losses.cpu().numpy(), float(lr.item())

    # ------------------------------------------------------------------ batching (host side, linear_model.py:247-300)
    def get_all_batches(self, data_x, data_y, camera_frame, training=True):
        """Obtain a list of all the batches, randomly permuted when training (linear_model.py:247-300)."""
        n = sum(v.shape[0] for v in data_x.values())
        encoder_inputs = np.zeros((n, self.input_size), dtype=float)
        decoder_outputs = np.zeros((n, self.output_size), dtype=float)
        idx = 0
        for key2d in data_x.keys():
            (subj, b, fname) = key2d
            key3d = key2d if camera_frame else (subj, b, "{0}.h5".format(fname.split(".")[0]))
            key3d = (subj, b, fname[:-3]) if fname.endswith("-sh") and camera_frame else key3d
            n2d = data_x[key2d].shape[0]
            encoder_inputs[idx:idx + n2d, :] = data_x[key2d]
            decoder_outputs[idx:idx + n2d, :] = data_y[key3d]
            idx += n2d
        if training:
            perm = np.random.permutation(n)
            encoder_inputs, decoder_outputs = encoder_inputs[perm, :], decoder_outputs[perm, :]
        n_extra = n % self.batch_size
        if n_extra > 0:
            encoder_inputs, decoder_outputs = encoder_inputs[:-n_extra, :], decoder_outputs[:-n_extra, :]
        n_batches = n // self.batch_size
        return np.split(encoder_inputs, n_batches), np.split(decoder_outputs, n_batches)

    # ------------------------------------------------------------------ graph handles (linear_model.py:128-148)
    # The reference's callers hold on to graph tensors of the model.  There is no graph here; the attributes exist and
    # carry what a `session.run` on them would have returned for the LAST step:
    #   model.outputs   (:128)      predictions of the last step() [B, out]
    #   model.loss      (:129)      its loss
    #   model.gradients (:143-144)  [[gradient, variable name], ...] of the last training step, in the order of the
    #                               trainable variables (the reference stores [grad, var] pairs)
    #   model.updates   (:145)      the train op: a callable that runs one training step, `model.updates(x, t, keep)`
    #   model.err_mm    (:133)      the 'error_mm' placeholder: a settable slot; `model.err_mm_summary` (:134) is BOTH
    #                               callable with a value (this repo's callers) and, called without one, the summary
    #                               of whatever model.err_mm holds (what sess.run(model.err_mm_summary,
    #                               {model.err_mm: e}) returns, predict_3dpose.py:295,322)
    @property
    def outputs(self):
        return getattr(self, "_last_outputs", None)

    @property
    def loss(self):
        return getattr(self, "_last_loss", None)

    @property
    def gradients(self):
        g = self.get_gradients()
        return [[g[n], n] for n in self.get_variable_names() if n in g]

    @property
    def updates(self):
        return lambda encoder_inputs, decoder_outputs, dropout_keep_prob: self.step(
            None, encoder_inputs, decoder_outputs, dropout_keep_prob, isTraining=True)

    def err_mm_summary(self, err_mm=None):
        """The 'loss/error_mm' summary of linear_model.py:133-134.  The reference evaluates it with
        `sess.run(model.err_mm_summary, {model.err_mm: total_err})` (predict_3dpose.py:295,322); without a session
        it is a call: `model.test_writer.add_summary(model.err_mm_summary(total_err), current_step)`, or
        `model.err_mm = total_err; model.err_mm_summary()`."""
        if err_mm is None:
            err_mm = self.err_mm
        return Summary("loss/error_mm", np.float32(err_mm))

    def close(self):
        if self._handle is not None:
            lib.p3d_model_destroy(self._handle)
            self._handle = None
        for w in (getattr(self, "train_writer", None), getattr(self, "test_writer", None)):
            if w is not None:
                w.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class PoseBase(object):
    """Facade with the call signature of the reference's TF2 twin `PoseBase` (src/top_vae_3d_pose/models.py:287-481):
    `PoseBase(units=1024, input_size=32, output_size=48)`, `model(inputs, training=False)` -> [B, output_size].
    It is LinearModel(units, 2, residual, batch_norm, max_norm) - the layer chain of `call` (:442-481) - so the VAE
    scripts can use the B200 lifter as their frozen `pose3d` network.  Variables carry the same names
    ("linear_model/w1", "linear_model/two_linear_0/w2_0", ...; :295-439) and are reachable as attributes w1, b1,
    w2_0, ... (NumPy copies) or through `model.linear`.  Only inference (`training=False`, moving statistics) is
    served: `training=True` in the reference is a forward with batch statistics inside a tf.GradientTape, which
    belongs to LinearModel.step(isTraining=True) here."""

    def __init__(self, units=1024, input_size=32, output_size=48, **kw):
        if input_size != 32 or output_size not in (48, 42):
            raise ValueError("PoseBase lifts 32-d 2D poses to 48-d (or 42-d) 3D poses")
        self.linear_size, self.input_size, self.output_size = units, input_size, output_size
        self.linear = LinearModel(units, 2, True, True, True, 64, 1e-3, predict_14=(output_size == 42), **kw)

    def __call__(self, inputs, training=True):
        return self.call(inputs, training=training)

    def call(self, inputs, training=True):
        if training:
            raise NotImplementedError("PoseBase facade serves training=False; train through LinearModel.step")
        is_torch = hasattr(inputs, "is_cuda")
        if is_torch:
            torch = _lib.require_cuda()
            zeros = torch.zeros((inputs.shape[0], self.output_size), dtype=torch.float32, device=inputs.device)
        else:
            zeros = np.zeros((np.asarray(inputs).shape[0], self.output_size), dtype=np.float32)
        return self.linear.step(None, inputs, zeros, 1.0, isTraining=False)[2]

    def __getattr__(self, name):                      # w1, b1, w2_0, b3_1, w4, ... (models.py:296-439)
        if name in ("linear", "linear_size", "input_size", "output_size"):
            raise AttributeError(name)
        full = None
        if name in ("w1", "b1", "w4", "b4"):
            full = "linear_model/" + name
        elif len(name) == 4 and name[0] in "wb" and name[1] in "23" and name[2] == "_" and name[3] in "01":
            full = "linear_model/two_linear_{0}/{1}".format(name[3], name)
        if full is None:
            raise AttributeError(name)
        return self.linear.get_variable(full)

    def load_weights(self, values):
        """{TF variable name: array} (e.g. checkpoint.read_bundle(prefix)) -> the model's variables."""
        have = set(self.linear.get_variable_names(include_optimizer=True))
        self.linear.set_variables({k: v for k, v in values.items() if k in have})

    def close(self):
        self.linear.close()
