"""Shared machinery behind the model contract.

The reference duplicates ~300 lines of iteration protocol in every model file
(``alex_net.py:300-585``, ``googlenet.py:650-950``, ``cifar10.py:254-493`` …): shared
input buffers + sub-batch slicing, the loader handshake, ``train_iter`` / ``val_iter``
/ ``reset_iter`` / ``adjust_hyperp`` / ``cleanup`` and the compile helpers.
:class:`ModelBase` implements that protocol once; a concrete model only provides
hyper-parameters, its data object and ``build_model()`` / ``forward()``.

Contract exposed (ref ``helper_funcs.py:163-205``, ``README.md:54-67``):
``params`` (list of torch tensors — views into the flat arena), ``data``,
``compile_iter_fns(sync_type)``, ``train_iter(count, recorder)``,
``val_iter(count, recorder)``, ``reset_iter(mode)``, ``adjust_hyperp(epoch)``,
``cleanup()``, ``n_epochs``, ``epoch``, ``n_subb``; plus ``vels``/``vels2``,
``shared_lr``, ``get_vel``/``descent_vel``/``train_iter_fn``/``val_iter_fn``.

B200-native pieces: bf16 NHWC activations with fp32 master weights in the arena;
the whole step (H2D hand-off excluded) can be captured in a CUDA graph
(``config['cuda_graph']``); lr/momentum live in device memory so the graph never
needs re-capture; costs/errors stay on the device until the recorder prints.
"""
from __future__ import annotations

import time

import numpy as np
import torch

from .. import ops
from ..parallel.arena import FlatArena
from ..utils import nvtx
from ..utils.opt import FlatAdam, FlatSGD, SharedScalar, pre_model_iter_fn
from .layers2 import BatchNormal, Crop, Dropout, count_params


def pick_device(config):
    dev = config.get("device")
    if dev is not None:
        return torch.device(dev)
    if torch.cuda.is_available():
        return torch.device("cuda", torch.cuda.current_device())
    return torch.device("cpu")


class ModelBase(object):
    # ---- hyper-parameter defaults (override per model)
    n_epochs = 1
    momentum = 0.9
    weight_decay = 0.0
    batch_size = 128
    file_batch_size = 128
    learning_rate = 0.01
    lr_policy = "step"
    lr_step = ()
    lr_gamma = 0.1
    use_momentum = True
    use_nesterov_momentum = False
    input_width = 227
    input_height = 227
    batch_crop_mirror = False
    rand_crop = True
    monitor_grad = False
    bias_lr_mult = 2.0             # biases train with 2x lr in the reference's optimizer (lib/opt.py:181-268)
    optimizer = "msgd"             # update rule of the arena: 'msgd' (momentum SGD, lib/opt.py) or 'adam'; config['optimizer'] overrides
    graph_safe = True              # False: the step draws host-side randomness / has host control flow → never auto-capture
    name = "Model"

    def __init__(self, config):
        self.config = config
        self.verbose = config.get("verbose", False)
        opt = config.get("optimizer", self.optimizer)
        opt = "msgd" if opt == "sgd" else opt
        if opt not in ("msgd", "adam"):
            raise ValueError("optimizer must be 'msgd' or 'adam', got %r" % (opt,))
        self.optimizer = opt
        self.rank = config.get("rank", 0)
        self.size = config.get("size", 1)
        self.no_paraload = config.get("no_paraload", False)
        self.device = pick_device(config)
        self.cuda = self.device.type == "cuda"
        # compute precision of the native path: 'bf16' (bf16 operands, fp32 accumulate / master weights) or 'tf32' (fp32 storage
        # end to end, tcgen05 kind::tf32 — the reference's precision class); see ops/precision.py
        from ..ops import precision
        if config.get("dtype"):
            precision.set_precision(config["dtype"])
        self.precision = precision.precision()
        self.act_dtype = precision.act_dtype() if self.cuda else torch.float32
        # "auto" (default on CUDA): capture the whole step into a CUDA graph, fall back to eager launches if the model's
        # step cannot be captured (host-side control flow, library calls that synchronise, …)
        cg = config.get("cuda_graph", "auto")
        self._graph_auto = (cg == "auto")
        if self._graph_auto and not getattr(self, "graph_safe", True):
            cg = False            # e.g. in-graph random crops drawn from a host RNG every step: a replay would freeze them
        self.use_graph = bool(cg) and self.cuda
        self.epoch = 0
        self.step_idx = 0
        self.mu = self.momentum
        self.eta = self.weight_decay
        self.base_lr = np.float32(self.learning_rate)
        self.current_t = self.subb_t = 0
        self.current_v = self.subb_v = 0
        self.last_one_t = self.last_one_v = False
        self.compiled_train_fn_list = []
        self.train_iter_fn = None
        self.val_iter_fn = None
        self._graph = None
        self._graph_out = None
        self._gstream = None
        self._warm = 0
        self._tail = None
        self.exchanger = None          # set by the BSP worker for fused / overlapped exchange
        self.h2d_bytes_last = 0

    # ------------------------------------------------------------------ construction helpers
    def setup_data_parallel(self, data):
        """The 'mini batching and other data parallel common routine' block of every
        reference model (``alex_net.py:73-80``)."""
        self.data = data
        data.batch_data(self.file_batch_size)
        data.extend_data(rank=self.rank, size=self.size)
        data.shuffle_data(mode="train", common_seed=1234)
        data.shuffle_data(mode="val")
        data.shard_data(mode="train", rank=self.rank, size=self.size)
        data.shard_data(mode="val", rank=self.rank, size=self.size)
        self.n_subb = max(1, self.file_batch_size // self.batch_size)

    def finalize(self, params, weight_types, input_shape):
        """Bind parameters into the flat arena and allocate the shared input buffers."""
        self.params, self.weight_types = list(params), list(weight_types)
        count_params(self.params, verbose=False)
        allocator = self.config.get("arena_allocator")
        self.arena = FlatArena(self.params, self.weight_types, self.device, weight_decay=self.eta, bias_lr_mult=self.bias_lr_mult,
                               with_recv=allocator is not None, allocator=allocator,
                               shadow=False if self.precision == "tf32" else self.config.get("_arena_shadow"), optimizer=self.optimizer)
        self.shared_lr = SharedScalar(self.arena.hyper, 0, self.base_lr)
        self.sgd = FlatSGD(self.arena, self.mu, self.use_nesterov_momentum, self.use_momentum)
        self.adam = FlatAdam(self.arena) if self.optimizer == "adam" else None
        B = self.batch_size
        fb = self.file_batch_size
        self.input_shape = tuple(input_shape)           # (B, H, W, C)
        self.shared_x = torch.zeros((fb,) + self.input_shape[1:], dtype=self.act_dtype, device=self.device)
        self.shared_y = torch.zeros((fb,), dtype=torch.int64, device=self.device)
        self.x_in = torch.zeros((B,) + self.input_shape[1:], dtype=self.act_dtype, device=self.device)
        self.y_in = torch.zeros((B,), dtype=torch.int64, device=self.device)
        # label staging: a small ring of pinned buffers, each guarded by the event of its last H2D copy — the host runs
        # ahead of the device (always under CUDA graphs, and whenever a step is GPU-bound), so a single buffer would be
        # overwritten with the NEXT batch's labels before the copy of the current ones has executed
        self._y_ring = [torch.zeros((fb,), dtype=torch.int64, pin_memory=self.cuda) for _ in range(4 if self.cuda else 1)]
        self._y_ev = [None] * len(self._y_ring)
        self._y_k = 0
        self.vels, self.vels2 = [], []
        if self.verbose:
            print("%s: %d tensors, %.3f M params, arena %.1f MiB on %s"
                  % (self.name, len(self.params), self.arena.n_real / 1e6,
                     self.arena.nbytes / 2 ** 20, self.device))

    # ------------------------------------------------------------------ to be provided by the model
    def build_model(self):
        raise NotImplementedError

    def forward(self, x):
        """Return logits-layer output; must leave ``self.output_layer`` evaluated."""
        raise NotImplementedError

    def loss(self, x, y):
        self.forward(x)
        sm = self.output_layer
        return sm.negative_log_likelihood(y), sm.errors(y), sm.errors_top_x(y)

    # ------------------------------------------------------------------ step functions
    def _fwd_bwd_eager(self):
        cost, err, err5 = self.loss(self.x_in, self.y_in)
        self._dbg_capture("forward")
        cost.backward()
        return cost.detach(), err.detach()

    def forward_backward(self, subb_ind=0):
        """Forward + backward on sub-batch ``subb_ind`` of the shared input buffer;
        gradients land in the arena's G region.  Returns device scalars (cost, error)."""
        B = self.batch_size
        if self.n_subb == 1 and self.shared_x.shape[0] == B:
            self.x_in.copy_(self.shared_x, non_blocking=True)
            self.y_in.copy_(self.shared_y, non_blocking=True)
        else:
            self.x_in.copy_(self.shared_x[subb_ind * B:(subb_ind + 1) * B], non_blocking=True)
            self.y_in.copy_(self.shared_y[subb_ind * B:(subb_ind + 1) * B], non_blocking=True)
        if not self.use_graph:
            return self._step_body()
        if self._graph is None:
            if self._gstream is None:
                self._gstream = torch.cuda.Stream(device=self.device)
            if self._warm < 2:
                # Eager warm-up ON THE CAPTURE STREAM: autograd caches each leaf's AccumulateGrad node together
                # with the stream that was current when it was first built; if that were the default stream the
                # engine would make the capturing stream wait on uncaptured work at the end of backward
                # (cudaErrorStreamCaptureIsolation).
                self._warm += 1
                cur = torch.cuda.current_stream(self.device)
                self._gstream.wait_stream(cur)
                with torch.cuda.stream(self._gstream):
                    out = self._step_body()
                cur.wait_stream(self._gstream)
                return out
            ok, why = True, ""
            try:
                self._capture()
            except Exception as e:  # noqa: BLE001
                if not self._graph_auto:
                    raise
                ok, why = False, "%s: %s" % (type(e).__name__, str(e)[:200])
            ex = self.exchanger
            if ex is not None and getattr(ex, "fused", False) and getattr(ex, "size", 1) > 1:
                # the fused exchange pairs device-side barriers by launch order: either every rank replays the graph or
                # every rank runs eager — agree on it (a capture that failed on one rank only would desynchronise them)
                ok = all(ex.comm.allgather(bool(ok)))
            if not ok:
                print("[%s] CUDA-graph capture of the training step failed (%s) — running eager"
                      % (getattr(self, "name", type(self).__name__), why or "on another rank"))
                self.use_graph = False
                self._graph = None
                if ex is not None and hasattr(ex, "_reset_pending") and getattr(ex, "fused", False):
                    ex._reset_pending()          # a half-captured step consumed some grad-ready callbacks
                torch.cuda.synchronize()
                return self._step_body()
        self._graph.replay()
        return self._graph_out

    def _step_body(self):
        out = self._fwd_bwd_eager()
        self._dbg_capture("forward+backward")
        if self._tail is not None:
            with torch.no_grad():
                self._tail()
            self._dbg_capture("step tail")
        self._after_step()
        return out

    def _dbg_capture(self, where):
        """TMPI_DEBUG_CAPTURE=1: name the stage that invalidated an ongoing CUDA-graph capture."""
        import os
        if not self.cuda or os.environ.get("TMPI_DEBUG_CAPTURE") != "1":
            return
        from ..ops import native
        err, status = native.require().capture_status(torch.cuda.current_stream(self.device).cuda_stream)
        if err != 0 or status == 2:
            raise RuntimeError("CUDA graph capture invalidated during %s (err %d status %d)" % (where, err, status))

    def _after_step(self):
        if self.cuda:
            from ..ops import cuda_impl
            cuda_impl.advance_step(self.device)
        else:
            ops.advance_rng_step()

    def _capture(self):
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        s = self._gstream
        s.wait_stream(torch.cuda.current_stream())
        inner = None
        try:
            with torch.cuda.stream(s):
                with torch.cuda.graph(g, stream=s, capture_error_mode="thread_local"):
                    try:
                        out = self._step_body()
                    except BaseException as e:       # capture_end would mask it with "invalidated"
                        inner = e
                        raise
        except Exception:
            if inner is not None:
                raise inner
            raise
        torch.cuda.current_stream().wait_stream(s)
        self._graph, self._graph_out = g, out

    def set_step_tail(self, fn):
        """Register work that runs right after backward as part of the step — and
        therefore *inside* the captured CUDA graph: the local fused SGD (k = 1) or the
        fused allreduce+SGD exchange kernels (k > 1)."""
        self._tail = fn
        self._graph = None
        self._warm = 0

    def compile_val(self):
        def val_fn(subb_ind=0):
            B = self.batch_size
            x = self.shared_x[subb_ind * B:(subb_ind + 1) * B]
            y = self.shared_y[subb_ind * B:(subb_ind + 1) * B]
            with torch.no_grad():
                c, e, e5 = self.loss(x, y)
            return c, e, e5
        self.val_fn = val_fn

    def compile_inference(self):
        def inf_fn(x):
            with torch.no_grad():
                Dropout.SetDropoutOff(); Crop.SetRandCropOff(); BatchNormal.SetTrainOff()
                out = torch.softmax(self.forward(x).float(), dim=1)
                Dropout.SetDropoutOn(); Crop.SetRandCropOn(); BatchNormal.SetTrainOn()
            return out
        self.inf_fn = inf_fn

    def compile_train(self, *args):
        self.compiled_train_fn_list.extend(args)

    def compile_iter_fns(self, sync_type="avg", aggregate="momentum", fused_tail=None):
        """``sync_type='cdd'``: split step (get_vel / exchange / descent_vel);
        ``'avg'``: self-contained local update (k = 1), the exchanger then averages
        weights.  Fixes SURVEY §2.9 #5/#7: every model accepts ``sync_type`` and 'avg'
        really updates."""
        start = time.time()
        self.sync_type = sync_type
        k = self.size if sync_type == "cdd" else 1
        if k > 1 and fused_tail is None:
            _ = self.arena.R                      # allocate the receive region
        pre_model_iter_fn(self, k, aggregate=aggregate, fused_tail=fused_tail)
        if self.verbose:
            print("Compile time: %.3f s" % (time.time() - start))

    # ------------------------------------------------------------------ data movement
    def _labels_to_device(self, labels):
        n = len(labels)
        k = self._y_k
        self._y_k = (k + 1) % len(self._y_ring)
        if self._y_ev[k] is not None:
            self._y_ev[k].synchronize()
        buf = self._y_ring[k]
        buf[:n] = torch.as_tensor(np.asarray(labels, dtype=np.int64))
        self.shared_y[:n].copy_(buf[:n], non_blocking=True)
        if self.cuda:
            if self._y_ev[k] is None:
                self._y_ev[k] = torch.cuda.Event()
            self._y_ev[k].record(torch.cuda.current_stream(self.device))
        return n * 8

    def _load_file_batch(self, mode, idx, img, labels, n_batches):
        """Loader handshake (ref ``alex_net.py:394-448``): request the next file,
        wait for the current one, put labels on the device."""
        loader = getattr(self.data, "loader", None)
        last = idx == n_batches - 1
        nbytes = 0
        if loader is not None:
            if idx == 0:
                loader.set_mode(mode)
                loader.request(img[idx], mode)
            loader.request(img[idx + 1] if not last else img[idx], mode)
            b = loader.get()
            self.shared_x = b.x
            nbytes += b.h2d_bytes
        else:
            x = self.data.load_batch(img[idx], mode, self)
            self.shared_x[:x.shape[0]].copy_(x.to(self.act_dtype), non_blocking=True)
            nbytes += x.numel() * x.element_size()
        nbytes += self._labels_to_device(labels[idx])
        self.h2d_bytes_last = nbytes
        return last

    # ------------------------------------------------------------------ the contract
    def reset_iter(self, mode):
        if mode == "train":
            self.current_t = self.subb_t = 0
            self.last_one_t = False
        else:
            self.current_v = self.subb_v = 0
            self.last_one_v = False
        loader = getattr(self.data, "loader", None)
        if loader is not None:
            loader.drain()       # the one look-ahead request issued for the last file

    def train_iter(self, count, recorder):
        if self.current_t == 0 and self.subb_t == 0:
            self.data.shuffle_data(mode="train", common_seed=self.epoch)
            self.data.shard_data(mode="train", rank=self.rank, size=self.size)
        img, labels = self.data.train_img_shard, self.data.train_labels_shard
        if self.subb_t == 0:
            recorder.start()
            with nvtx.range("load"):
                self.last_one_t = self._load_file_batch("train", self.current_t, img, labels,
                                                        self.data.n_batch_train)
            recorder.end("wait")
        recorder.start()
        with nvtx.range("train_iter_fn"):
            cost, error = self.train_iter_fn(self.subb_t)
        recorder.train_error(count, cost, error)
        recorder.end("calc")
        if self.monitor_grad and self.verbose:
            print(self.grad_norms())
        if (self.subb_t + 1) // self.n_subb == 1:
            self.current_t = 0 if self.last_one_t else self.current_t + 1
            self.subb_t = 0
        else:
            self.subb_t += 1
        self.step_idx += 1

    def val_iter(self, count, recorder):
        if self.current_v == 0 and self.subb_v == 0:
            self.data.shuffle_data(mode="val")
            self.data.shard_data(mode="val", rank=self.rank, size=self.size)
        img, labels = self.data.val_img_shard, self.data.val_labels_shard
        if self.subb_v == 0:
            self.last_one_v = self._load_file_batch("val", self.current_v, img, labels,
                                                    self.data.n_batch_val)
        Dropout.SetDropoutOff(); Crop.SetRandCropOff(); BatchNormal.SetTrainOff()
        cost, error, error_top5 = self.val_iter_fn(self.subb_v)
        Dropout.SetDropoutOn(); Crop.SetRandCropOn(); BatchNormal.SetTrainOn()
        recorder.val_error(count, cost, error, error_top5)
        if (self.subb_v + 1) // self.n_subb == 1:
            self.current_v = 0 if self.last_one_v else self.current_v + 1
            self.subb_v = 0
        else:
            self.subb_v += 1

    def adjust_hyperp(self, epoch):
        """Once per epoch (ref ``alex_net.py:569-579``, ``googlenet.py:925-945``)."""
        if self.lr_policy == "step":
            if epoch in self.lr_step:
                self.shared_lr.set_value(np.float32(self.shared_lr.get_value() * self.lr_gamma))
        elif self.lr_policy == "poly":
            power = getattr(self, "lr_power", 0.5)
            self.shared_lr.set_value(np.float32(self.base_lr * (1.0 - float(epoch + 1) / self.n_epochs) ** power))
        elif self.lr_policy == "auto":
            pass

    def scale_lr(self, size):
        self.shared_lr.set_value(np.float32(self.shared_lr.get_value() * size))

    def grad_norms(self):
        """L2 grad-norm monitor (ref ``alex_net.py:311-320``): (sum, max) of log10 norms."""
        norms = torch.stack([g.float().norm() for g in self.arena.views("G")]).clamp_min(1e-30).log10()
        return [float(norms.sum()), float(norms.max())]

    # ------------------------------------------------------------------ checkpoint extras (non-parameter state)
    def _bn_layers(self):
        return [l for l in (getattr(self, "layers", None) or []) if isinstance(l, BatchNormal)]

    def extra_state(self):
        """Batch-norm running statistics (not parameters, so not in the arena)."""
        return {"bn": [(l.running_mean.detach().cpu(), l.running_var.detach().cpu()) for l in self._bn_layers()]}

    def load_extra_state(self, sd):
        for l, (m, v) in zip(self._bn_layers(), sd.get("bn", [])):
            l.running_mean = m.to(self.device).clone()
            l.running_var = v.to(self.device).clone()

    def cleanup(self):
        if getattr(self.data, "para_load", False) and hasattr(self.data, "para_load_close"):
            self.data.para_load_close()
