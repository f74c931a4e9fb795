"""Exchangers: the glue between a rule's runtime and the communication backend
(ref ``theanompi/lib/exchanger.py``).

``BSP_Exchanger``    (``exchanger.py:45-134``)  per-iteration exchange; strategy selection
``EASGD_Exchanger``  (``:137-286``)             elastic push/pull against the center
``ASGD_Exchanger``   (``:289-392``)             delta-accumulate variant (dead in the reference)
``GOSGD_Exchanger``  (``:412-617``)             gossip push-sum merge with a random peer

B200-native hot paths (no NCCL / MPI call on them):

* BSP ``fused*`` strategies: ONE kernel family reads all peers' gradients over NVLink,
  averages, applies the model's update rule (weight-decay + momentum + lr, or Adam),
  refreshes the bf16 compute shadow and
  (two-shot / NVLS) pushes the updated slice to the peers; launched per bucket on a side
  stream from the backward's grad-ready callbacks so it overlaps backward; part of the
  captured CUDA graph.
* EASGD: the worker's kernel computes ``d = α(w − c)`` against the center's memory mapped
  over NVLink and updates BOTH sides in one pass (the reference does two full-model
  broadcasts + an update sweep on each side).
* GOSGD: the sender snapshots its weights locally and keeps training; the receiver's
  kernel pulls the snapshot over NVLink and blends ``(α·w + α_s·b)/(α+α_s)`` in one pass.
"""
from __future__ import annotations

import os

import numpy as np
import torch
import torch.distributed as dist

from . import exchanger_strategy as ES
from ..utils import nvtx

FUSED = {"fused": ("auto", False), "fused16": ("auto", True), "oneshot": ("oneshot", False),
         "oneshot16": ("oneshot", True), "twoshot": ("twoshot", False), "twoshot16": ("twoshot", True),
         "nvls": ("nvls", False), "nvls16": ("nvls", True),
         # experimental (opt-in): reduce-scatter of the big FC gradients fused into the wgrad GEMM epilogue — each rank's
         # tcgen05 GEMM red.adds its dW tiles straight into the owner rank's G over NVLink, the exchange kernel only updates
         # its slice, all-gathers W / H and clears G
         "fused_rs": ("auto", False)}


# --------------------------------------------------------------------------- p2p helpers (ref :10-33)
def do_sendrecv(comm, glist, wlist, dest, group=None):
    """Exchange the tensors of ``glist`` with ``dest`` into ``wlist`` (device buffers)."""
    for g, w in zip(glist, wlist):
        ops = [dist.P2POp(dist.isend, g.contiguous(), dest, group=group), dist.P2POp(dist.irecv, w, dest, group=group)]
        for r in dist.batch_isend_irecv(ops):
            r.wait()


def do_send(comm, glist, dest, group=None):
    for g in glist:
        dist.send(g.contiguous(), dest, group=group)


def do_recv(comm, wlist, src, group=None):
    for w in wlist:
        dist.recv(w, src, group=group)


def remove_BN_params(param_list):
    """Drop params named gamma/beta from the exchanged list (ref ``:35-43``)."""
    return [p for p in param_list if getattr(p, "pname", None) not in ("gamma", "beta")]


# =========================================================================== BSP
class BSP_Exchanger(object):
    def __init__(self, comm, gpucomm, exch_strategy, sync_type, ctx, model, nccl_group=None,
                 bucket_bytes=None, overlap=True, comm_blocks=None):
        self.comm, self.gpucomm = comm, gpucomm
        self.size = comm.size
        self.exch_strategy, self.sync_type, self.ctx, self.model = exch_strategy, sync_type, ctx, model
        self.arena = getattr(model, "arena", None)
        self.fused = exch_strategy in FUSED and self.size > 1
        self.exch = None
        self.overlap = overlap
        self.comm_blocks = comm_blocks
        self.bucket_bytes = bucket_bytes
        self.nccl_group = nccl_group
        if self.size == 1:
            return
        if self.fused:
            if sync_type != "cdd":
                raise ValueError("fused strategies implement the cdd (gradient) exchange")
            self.adam = getattr(model, "optimizer", "msgd") == "adam"
            if self.adam and exch_strategy == "fused_rs":
                raise ValueError("fused_rs (gradients reduce-scattered by the GEMM epilogue) supports momentum SGD only, not Adam; "
                                 "use fused or fused16")
            if gpucomm is None:
                raise RuntimeError("strategy %s needs the symmetric peer arena (GPUs of one node)" % exch_strategy)
            self.algo, self.wire16 = FUSED[exch_strategy]
            # owner-keeps-master (default when the model computes from bf16 shadows): for WEIGHT tensors the fused kernel
            # ships only the bf16 compute shadow of an updated slice to the peers — a third of the all-gather bytes; their
            # fp32 master copies on non-owners go stale until sync_master() (called before checkpoints / by finalize).
            # Biases — which the forward kernels read in fp32 — always travel as masters.  TMPI_PUSH_MASTER=1 restores the
            # full push.
            self.push_master = (os.environ.get("TMPI_PUSH_MASTER", "0") == "1") or self.arena.H is None
            self._master_stale = False
            self._setup_buckets()
            return
        if sync_type == "cdd":
            src, dst, avg = model.vels, model.vels2, False
        elif sync_type == "avg":
            src = dst = remove_BN_params(model.params)
            avg = True
        else:
            raise ValueError("sync_type must be cdd or avg")
        s = exch_strategy
        if s == "ar":
            self.exch = ES.Exch_allreduce(comm, avg=avg)
        elif s == "nccl32":
            self.exch = ES.Exch_nccl32(comm, nccl_group, avg=avg)
        elif s == "nccl16":
            self.exch = ES.Exch_nccl16(comm, nccl_group, avg=avg)
        elif s == "asa32":
            self.exch = ES.Exch_asa32(comm, avg=avg, group=nccl_group)
        elif s == "asa16":
            self.exch = ES.Exch_asa16(comm, avg=avg, group=nccl_group)
        elif s == "copper":
            self.exch = ES.Exch_copper(comm, avg=avg, group=nccl_group)
        elif s == "copper16":
            self.exch = ES.Exch_copper16(comm, avg=avg, group=nccl_group)
        elif s == "swap":
            self.exch = ES.Exch_swap(comm, group=nccl_group)
            src = dst = remove_BN_params(model.params)       # fixes the undefined self.param_list (SURVEY §2.9 #4)
        elif s == "p2p32":
            if sync_type == "cdd":
                self.exch = ES.Exch_p2p32(gpucomm, self.arena, model._send_region, "R", avg=False)
            else:
                self.exch = ES.Exch_p2p32(gpucomm, self.arena, "W", "W", avg=True)
        else:
            raise ValueError("unknown exch_strategy %r" % s)
        self.exch.prepare(ctx, src, dst)

    # ------------------------------------------------------------------ fused path
    def _rs_params(self):
        """Indices of the parameters whose gradient is produced by one fp32 GEMM straight into ``gbuf`` (native FC / Softmax
        weights) and is big enough to be worth a bucket of its own."""
        out = set()
        for i, p in enumerate(self.arena.params):
            if getattr(p, "rs_ok", False) and p.dim() == 2 and p.shape[0] % 8 == 0 and p.shape[1] % 8 == 0 and p.numel() >= (1 << 20):
                out.add(i)
        return out

    def _setup_buckets(self):
        a = self.arena
        self.rs = self.exch_strategy == "fused_rs"
        bb = self.bucket_bytes or (a.numel * 4 if not self.overlap else 32 << 20)
        if self.rs:
            solo = self._rs_params()
            self.buckets = a.make_buckets(bb if self.overlap else a.numel * 4, solo=solo)
            ranges = []
            for b in self.buckets:
                b["rs"] = len(b["params"]) == 1 and b["params"][0] in solo
                if b["rs"]:
                    ranges.append((b["lo"], b["hi"]))
            # G must be clear everywhere before the first producer adds into a peer, and stays clear afterwards (the exchange
            # kernel zeroes what it consumed)
            a.G.zero_()
            torch.cuda.synchronize(a.device)
            self.comm.Barrier()
            self.gpucomm.configure_gemm_rs(a, ranges)
            self.gpucomm.barrier()
            torch.cuda.synchronize(a.device)
            self.comm.Barrier()
        else:
            tail = int(os.environ.get("TMPI_TAIL_BUCKET_BYTES", str(4 << 20)))
            self.buckets = a.make_buckets(bb, tail_bytes=tail) if self.overlap else [dict(lo=0, hi=a.numel, params=list(range(len(a.params))))]
        self._pending = [0] * len(self.buckets)
        self._bucket_of = {}
        for bi, b in enumerate(self.buckets):
            for pi in b["params"]:
                self._bucket_of[pi] = bi
        self._index_of = {id(p): i for i, p in enumerate(a.params)}
        self.side = torch.cuda.Stream(device=a.device) if self.overlap else None
        self._launched = 0
        if self.overlap:
            for p in a.params:
                p.on_ready = self._on_ready
            self._reset_pending()

    def _reset_pending(self):
        for bi, b in enumerate(self.buckets):
            self._pending[bi] = len(b["params"])
        self._launched = 0

    def _launch_bucket(self, bi):
        b, m = self.buckets[bi], self.model
        mu = m.mu if m.use_momentum else 0.0
        blocks = self.comm_blocks
        if blocks is None and self.overlap:
            big = int(os.environ.get("TMPI_OVERLAP_BLOCKS", "64"))     # measured at 2 ranks: 16 → 4.5 ms, 32 → 3.1, 64 → 2.17, 148 → 2.28
            blocks = big if (b["hi"] - b["lo"]) * 4 > (8 << 20) else min(8, big)
        if self.adam:
            # Adam: two-shot buckets update the moments on the owner of a slice only → sync_master() pushes them too
            ad = m.adam
            self.gpucomm.fused_allreduce_adam(self.arena, b["lo"], b["hi"], ad.b1, ad.b2, ad.eps, algo=self.algo, wire16=self.wire16,
                                              max_blocks=blocks, push_master=self.push_master)
            self._master_stale = True
            return
        self.gpucomm.fused_allreduce_sgd(self.arena, b["lo"], b["hi"], mu, m.use_nesterov_momentum,
                                         algo=self.algo, wire16=self.wire16, max_blocks=blocks, pre_reduced=b.get("rs", False),
                                         push_master=self.push_master)
        if not self.push_master:
            self._master_stale = True

    def sync_master(self):
        """Collective: make every rank's fp32 master weights (owner-keeps-master mode) and, for Adam, both moments current
        again.  Buckets that ran the one-shot algorithm are already identical everywhere; the two-shot ones push their owner
        slices."""
        if not getattr(self, "fused", False) or not self._master_stale:
            return
        regions = ([] if self.push_master else ["W"]) + (["U", "V"] if self.adam else [])
        if not regions:
            return
        for b in self.buckets:
            nbytes = (b["hi"] - b["lo"]) * (2 if self.wire16 else 4)
            if self.gpucomm.pick_algo(nbytes, self.algo) != 0 or b.get("rs", False):
                for r in regions:
                    self.gpucomm.push_region_slices(self.arena, r, b["lo"], b["hi"])
        torch.cuda.synchronize(self.arena.device)
        self.comm.Barrier()
        self._master_stale = False

    def _on_ready(self, p):
        """Called by a backward kernel wrapper right after it enqueued the gradient of ``p``."""
        bi = self._bucket_of[self._index_of[id(p)]]
        self._pending[bi] -= 1
        # buckets must start in the SAME order on every rank (device-side barriers pair up by launch order)
        while self._launched < len(self.buckets) and self._pending[self._launched] == 0:
            cur = torch.cuda.current_stream()
            self.side.wait_stream(cur)
            with torch.cuda.stream(self.side):
                self._launch_bucket(self._launched)
            self._launched += 1

    def fused_step(self):
        """The model's *step tail*: everything left of the exchange + update, then join."""
        if self.overlap:
            # parameters that did not go through an on_ready callback (e.g. unused) flush here
            cur = torch.cuda.current_stream()
            while self._launched < len(self.buckets):
                self.side.wait_stream(cur)
                with torch.cuda.stream(self.side):
                    self._launch_bucket(self._launched)
                self._launched += 1
            cur.wait_stream(self.side)
            self._reset_pending()
        else:
            for bi in range(len(self.buckets)):                   # one bucket, or solo reduce-scatter buckets + the rest
                self._launch_bucket(bi)
        if self.adam:
            # every bucket of this step read the same t; the next step's first bucket waits on this stream
            self.gpucomm.adam_advance(self.arena)

    # ------------------------------------------------------------------ the per-iteration call
    def exchange(self, recorder):
        """Barrier timed as *sync*, collective as *comm* (ref ``:120-134``); then the post
        update runs immediately (SURVEY §2.9 #8).  For fused strategies both already
        happened inside the step (device-side barrier + fused kernel): nothing to launch."""
        if self.size == 1:
            return
        if self.fused:
            return
        recorder.start()
        self.comm.Barrier()
        recorder.end("sync")
        recorder.start()
        with torch.no_grad(), nvtx.range("exchange:" + self.exch_strategy):
            self.exch.exchange()
        if self.sync_type == "cdd":
            self.model.descent_vel()
        elif self.arena is not None and self.exch_strategy != "p2p32":
            self.arena.refresh_shadow()
        recorder.end("comm")


# =========================================================================== EASGD
class EASGD_Exchanger(object):
    """Elastic averaging against the center.

    ``etype='server'`` owns the center (its model's arena W); ``etype='worker'`` owns a
    replica.  GPU path: worker-side fused kernel on the peer-mapped center.  CPU path:
    the two sides swap flat copies (gloo) and apply the reference's update functions
    (``exchanger.py:188-211``): server ``g += α(w−g)``, worker ``w −= α(w−g)``."""

    def __init__(self, alpha, param_list, etype, comm=None, gpucomm=None, arena=None, server_rank=0, group=None):
        self.alpha, self.etype = alpha, etype
        self.param_list = param_list
        self.comm, self.gpucomm, self.arena, self.group = comm, gpucomm, arena, group
        self.server_rank = server_rank
        self.peer = None                       # server: rank of the worker being served
        self.device = arena.W.device if arena is not None else param_list[0].device
        self.use_p2p = gpucomm is not None and self.device.type == "cuda"
        # TMPI_EASGD_LOCKFREE=1: no ticket lock — the center is updated with vector red.add over NVLink (commutative: no
        # update can be lost) and all workers exchange concurrently
        self.lockfree = os.environ.get("TMPI_EASGD_LOCKFREE", "0") == "1"
        self.max_blocks = int(os.environ.get("TMPI_EASGD_BLOCKS", "0")) or None
        self.n_exchanges = 0
        if not self.use_p2p:
            n = arena.numel if arena is not None else sum(p.numel() for p in param_list)
            self.mirror = torch.zeros(n, dtype=torch.float32, device=self.device)

    def _flat(self):
        if self.arena is not None:
            return self.arena.W
        return torch.cat([p.detach().reshape(-1) for p in self.param_list])

    def _unflat(self, flat):
        if self.arena is not None:
            if flat.data_ptr() != self.arena.W.data_ptr():
                self.arena.W.copy_(flat)
            self.arena.refresh_shadow()
            return
        off = 0
        with torch.no_grad():
            for p in self.param_list:
                p.copy_(flat[off:off + p.numel()].view_as(p)); off += p.numel()

    # ---- GPU data plane: everything below is enqueued on the worker's stream and returns immediately
    def _lock_state(self):
        if getattr(self, "_lstate", None) is None:
            self._lstate = torch.zeros(4, dtype=torch.int32, device=self.device)
        return self._lstate

    def _p2p_section(self, body):
        """Run ``body`` (kernel launches touching the center) under the device-side ticket lock of the center rank."""
        gc = self.gpucomm
        if self.lockfree:
            body()
            return
        st = self._lock_state()
        gc.ticket_acquire(self.server_rank, st)
        body()
        gc.ticket_release(self.server_rank, st)

    def exchange(self):
        if self.use_p2p:
            if self.etype == "worker":
                from ..ops import native
                a, gc = self.arena, self.gpucomm
                center = gc.peer_region(self.server_rank, a.layout["W"], a.numel)
                self._p2p_section(lambda: native.require().easgd_elastic(
                    a.W.data_ptr(), a.H.data_ptr() if a.H is not None else 0, center.data_ptr(), float(self.alpha), a.numel,
                    gc._blocks(self.max_blocks), gc._stream(), int(self.lockfree)))
                self.n_exchanges += 1
            return
        other = self.peer if self.etype == "server" else self.server_rank
        mine = self._flat().contiguous()
        ops = [dist.P2POp(dist.isend, mine, other, group=self.group), dist.P2POp(dist.irecv, self.mirror, other, group=self.group)]
        for r in dist.batch_isend_irecv(ops):
            r.wait()
        with torch.no_grad():
            if self.etype == "server":
                new = mine + self.alpha * (self.mirror - mine)          # g += α(w − g)
            else:
                new = mine - self.alpha * (mine - self.mirror)          # w −= α(w − g)
            self._unflat(new)

    def copy_to_local(self):
        """Worker ← center (before/after validation and at stop, ref ``:264-286``)."""
        if self.use_p2p:
            if self.etype == "worker":
                from ..ops import native
                a, gc = self.arena, self.gpucomm
                center = gc.peer_region(self.server_rank, a.layout["W"], a.numel)
                self._p2p_section(lambda: native.require().copy_flat(
                    a.W.data_ptr(), a.H.data_ptr() if a.H is not None else 0, center.data_ptr(), a.numel,
                    gc._blocks(self.max_blocks), gc._stream()))
            return
        if self.etype == "server":
            dist.send(self._flat().contiguous(), self.peer, group=self.group)
        else:
            dist.recv(self.mirror, self.server_rank, group=self.group)
            self._unflat(self.mirror.clone())


# =========================================================================== ASGD (delta push)
class ASGD_Exchanger(object):
    """Server ``g += Δ``; worker ``w = g_new; Δ = 0`` where Δ = w − w_at_last_sync
    (ref ``exchanger.py:289-392``; no reference rule uses it — kept for the ``ASGD`` stub)."""

    def __init__(self, param_list, etype, comm=None, arena=None, server_rank=0, group=None):
        self.etype, self.comm, self.arena, self.server_rank, self.group = etype, comm, arena, server_rank, group
        self.param_list = param_list
        self.peer = None
        n = arena.numel if arena is not None else sum(p.numel() for p in param_list)
        dev = arena.W.device if arena is not None else param_list[0].device
        self.buf = torch.zeros(n, dtype=torch.float32, device=dev)
        self.last = self._flat().clone()

    _flat = EASGD_Exchanger._flat
    _unflat = EASGD_Exchanger._unflat

    def exchange(self):
        if self.etype == "server":
            dist.recv(self.buf, self.peer, group=self.group)             # Δ from the worker
            new = self._flat() + self.buf
            self._unflat(new)
            dist.send(self._flat().contiguous(), self.peer, group=self.group)
        else:
            delta = (self._flat() - self.last).contiguous()
            dist.send(delta, self.server_rank, group=self.group)
            dist.recv(self.buf, self.server_rank, group=self.group)
            self._unflat(self.buf.clone())
            self.last = self._flat().clone()

    def copy_to_local(self):
        """Worker ← center (before / after validation and at stop): the server sends its flat weights, the worker adopts
        them and restarts its delta from there."""
        if self.etype == "server":
            dist.send(self._flat().contiguous(), self.peer, group=self.group)
        else:
            dist.recv(self.buf, self.server_rank, group=self.group)
            self._unflat(self.buf.clone())
            self.last = self._flat().clone()


# =========================================================================== GOSGD
class GOSGD_Exchanger(object):
    """Gossip push-sum exchange (ref ``lib/exchanger.py:412-617``).

    GPU data plane = a device-side protocol (``csrc/comm_kernels.cu``, ``gosgd_*``): the sender snapshots W into its R
    region, halves its push-sum weight (a device scalar) and posts ``{seq, α}`` into the receiver's inbox slot in the
    receiver's signal pad; every iteration the receiver runs ``poll → pull-merge → ack`` (three launches, no-ops when nothing
    is pending) that blends the sender's snapshot over NVLink and acknowledges on the sender's pad.  No host message, no
    ``stream.synchronize()`` — a push that finds the previous snapshot still un-pulled is skipped (counted) instead of
    blocking, so two ranks pushing to each other cannot deadlock.  CPU / gloo: host mailbox + isend of the snapshot."""
    TAG_REQ, TAG_ACK = 700, 703

    def __init__(self, comm, gpucomm, model, p=0.01, seed=None, group=None):
        self.comm, self.gpucomm, self.model, self.p = comm, gpucomm, model, p
        self.rank, self.size = comm.rank, comm.size
        self.arena = model.arena
        self._alpha = 1.0 / self.size                             # push-sum weight (ref :430)
        self.rs = np.random.RandomState(seed if seed is not None else (1000 + 7919 * self.rank))
        self.group = group
        self.device = self.arena.W.device
        self.use_p2p = gpucomm is not None and self.device.type == "cuda"
        self._unacked = 0
        self._pending_sends = []
        self.max_blocks = int(os.environ.get("TMPI_GOSGD_BLOCKS", "0")) or None
        if not self.use_p2p:
            self.b = torch.zeros(self.arena.numel, dtype=torch.float32, device=self.device)
            self.snap = torch.zeros_like(self.b)
        else:
            if "R" not in self.arena.layout:
                _ = self.arena.R
            self.state = torch.zeros(64, dtype=torch.int32, device=self.device)
            self.state[:1].view(torch.float32).fill_(self._alpha)
            self._count_tick = 0
        self.n_merged = 0
        self.n_pushed = 0

    # ---- push-sum weight (device scalar on the GPU path)
    @property
    def alpha(self):
        if self.use_p2p:
            return float(self.state[:1].view(torch.float32).item())
        return self._alpha

    @alpha.setter
    def alpha(self, v):
        if self.use_p2p:
            self.state[:1].view(torch.float32).fill_(float(v))
        else:
            self._alpha = float(v)

    def device_counters(self):
        """(pushes done, pushes skipped, merges done) as counted by the device protocol (synchronises)."""
        st = self.state.cpu()
        return int(st[4]), int(st[5]), int(st[6])

    # ---- Bernoulli draw + uniform peer (ref :586-617)
    def draw(self):
        return self.rs.binomial(1, self.p) == 1

    def choose(self):
        if self.size < 2:
            return None
        d = self.rs.randint(0, self.size - 1)
        return d if d < self.rank else d + 1

    def _share_counts(self, count_arr):
        """Progress counters used for the epoch arithmetic travel through the store (best effort, every 16 calls): the device
        protocol carries weights only.  Element-wise max, as for the host messages (SURVEY §2.9 #14)."""
        if count_arr is None:
            return
        self._count_tick += 1
        if self._count_tick % 16:
            return
        st, pre = self.comm.store, self.comm.prefix
        st.set("%s/gosgd_count/%d" % (pre, self.rank), str(float(count_arr[self.rank])))
        for r in range(self.size):
            if r == self.rank:
                continue
            key = "%s/gosgd_count/%d" % (pre, r)
            try:
                if st.check([key]):
                    count_arr[r] = max(count_arr[r], float(st.get(key)))
            except Exception:  # noqa: BLE001
                pass

    # ---- receiver side
    def process_messages(self, count_arr=None):
        """Drain inbound pushes: pull the sender's snapshot, blend, add its weight
        (ref ``:484-535``).  ``count_arr`` is merged element-wise (max) instead of being
        overwritten by the sender's view (SURVEY §2.9 #14)."""
        if self.use_p2p:
            a, gc = self.arena, self.gpucomm
            gc.pa.gosgd_poll_merge(self.state.data_ptr(), int(a.layout["W"]), int(a.layout["H"]) if a.H is not None else -1,
                                   int(a.layout["R"]), int(a.numel), gc._blocks(self.max_blocks), gc._stream())
            self._share_counts(count_arr)
            return 0
        while self.comm.iprobe(tag=self.TAG_ACK):
            self.comm.recv(tag=self.TAG_ACK)
            self._unacked -= 1
        merged = 0
        while self.comm.iprobe(tag=self.TAG_REQ):
            msg = self.comm.recv(tag=self.TAG_REQ)
            src, a_src = msg["src"], float(msg["alpha"])
            if count_arr is not None and msg.get("count") is not None:
                np.maximum(count_arr, np.asarray(msg["count"]), out=count_arr)
            self._merge_params_from(src, a_src)
            self._alpha += a_src
            self.comm.send(self.rank, src, tag=self.TAG_ACK)
            merged += 1
        self.n_merged += merged
        return merged

    def _merge_params_from(self, src, a_src):
        a = self.arena
        dist.recv(self.b, src, group=self.group)
        from ..ops import reference as ref
        with torch.no_grad():
            ref.gosgd_merge(a.W, self.b, self._alpha, a_src)
        a.refresh_shadow()

    # ---- sender side
    def push_message(self, dest, count_arr=None):
        """Snapshot my weights, halve my push-sum weight, notify ``dest`` and keep training
        (ref ``:538-584`` blocks inside ncclBcast until the receiver joins)."""
        a = self.arena
        if self.use_p2p:
            gc = self.gpucomm
            gc.pa.gosgd_push(self.state.data_ptr(), int(dest), int(a.layout["W"]), int(a.layout["R"]), int(a.numel),
                             gc._blocks(self.max_blocks), gc._stream())
            self.n_pushed += 1
            return
        while self._unacked > 0:                                   # my snapshot buffer is still being pulled
            self.process_messages(count_arr)
        self.snap.copy_(a.W)
        self._alpha *= 0.5
        self.comm.send({"src": self.rank, "alpha": self._alpha,
                        "count": None if count_arr is None else np.asarray(count_arr).tolist()}, dest, tag=self.TAG_REQ)
        self._unacked += 1
        self._pending_sends = [w for w in self._pending_sends if not w.is_completed()]
        self._pending_sends.append(dist.isend(self.snap, dest, group=self.group))
        self.n_pushed += 1

    def _outstanding(self):
        """GPU path: is my last snapshot still waiting to be pulled?  (synchronises)"""
        st = self.state.cpu()
        last = int(st[2])
        if last == 0:
            return False
        acked = int(self.gpucomm.proto_words(self.gpucomm.rank)[96 + last - 1].item())
        return (acked & 0xFFFFFFFF) != (int(st[3]) & 0xFFFFFFFF)

    def finish(self, count_arr=None):
        """Clean shutdown without deadlock: (1) keep serving inbound pushes until all of mine
        are acknowledged, (2) announce completion, (3) keep serving until every rank has
        announced — at that point no push can be in flight any more."""
        import time
        busy = self._outstanding if self.use_p2p else (lambda: self._unacked > 0)
        while busy():
            self.process_messages(count_arr)
            time.sleep(0.0005)
        key = "%s/gosgd_done" % self.comm.prefix
        self.comm.store.add(key, 1)
        while int(self.comm.store.add(key, 0)) < self.size:
            self.process_messages(count_arr)
            time.sleep(0.0005)
        self.process_messages(count_arr)
        if self.use_p2p:
            self.process_messages(count_arr)
            torch.cuda.synchronize(self.device)
            pushed, skipped, merged = self.device_counters()
            self.n_pushed, self.n_skipped, self.n_merged = pushed, skipped, merged
        for w in self._pending_sends:
            w.wait()
