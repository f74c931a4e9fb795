"""Symmetric peer memory: Python face of ``csrc/peer_arena.cpp`` + ``csrc/comm_kernels.cu``.

Every rank of a node allocates an identically laid-out arena (see
:class:`theanompi_b200.parallel.arena.FlatArena`) from CUDA VMM memory, exchanges the
shareable handles with its peers and maps all of them — plus, when the fabric supports
it, one NVLS multicast mapping over all arenas.  The fused exchange kernels then read
and write peers' gradients / weights directly over NVLink 5 / NVSwitch.

This replaces the reference's data plane — NCCL-1 cliques created by shipping the
unique id over MPI (``theanompi/lib/base.py:22-150``), CUDA-aware MPI on raw device
pointers through the patched ``as_buffer`` (``test/test-train-mode/test-as-buffer``),
and the cudaIpc + ZeroMQ hand-off of the loader (``models/data/imagenet.py:302-311``).
"""
from __future__ import annotations

import os
import uuid

import torch

from ..ops import native

ALGO = {"oneshot": 0, "twoshot": 1, "nvls": 2}


class _CudaBuffer(object):
    """Expose a raw device pointer to torch through ``__cuda_array_interface__``."""

    def __init__(self, ptr, nbytes, owner):
        self.__cuda_array_interface__ = {"shape": (int(nbytes),), "typestr": "|u1", "data": (int(ptr), False), "version": 2}
        self._owner = owner


def tensor_from_ptr(ptr, nbytes, device, owner):
    return torch.as_tensor(_CudaBuffer(ptr, nbytes, owner), device=device)


class SymmetricComm(object):
    def __init__(self, comm, device, nbytes=None, local_ranks=None):
        self.comm = comm
        self.device = torch.device(device)
        self.L = native.require()
        self.local_ranks = list(local_ranks) if local_ranks is not None else list(range(comm.size))
        self.rank = self.local_ranks.index(comm.rank)
        self.size = len(self.local_ranks)
        if self.size != comm.size:
            raise RuntimeError("symmetric peer memory spans one node; use exch_strategy nccl32 across nodes")
        self.pa = None
        self.has_multicast = False
        self.multicast_error = None
        self.nbytes = 0
        self.max_blocks = int(os.environ.get("TMPI_COMM_BLOCKS", "0")) or None
        self._tensors = {}
        if nbytes is not None:
            self.create(nbytes)

    # ------------------------------------------------------------------ allocation + handle exchange
    def create(self, nbytes):
        assert self.pa is None, "symmetric arena already created"
        L, comm = self.L, self.comm
        job = comm.bcast(uuid.uuid4().hex[:12] if comm.rank == 0 else None, root=0)
        sizes = comm.allgather(int(nbytes))
        if len(set(sizes)) != 1:
            raise RuntimeError("symmetric arena: ranks disagree on the size: %s" % sizes)
        force_ipc = os.environ.get("TMPI_ARENA", "vmm") == "ipc"
        self.pa = L.PeerArena(self.rank, self.size, self.device.index, int(nbytes), job, force_ipc)
        modes = comm.allgather(self.pa.mode())
        if len(set(modes)) != 1:                      # mixed outcome: everybody falls back to cudaIpc
            self.pa = None
            self.pa = L.PeerArena(self.rank, self.size, self.device.index, int(nbytes), job + "i", True)
        self.mode = self.pa.mode()
        self.nbytes = int(self.pa.arena_bytes())
        comm.Barrier()
        if self.size > 1:
            if self.mode == "vmm":
                for p in range(self.size):
                    if p != self.rank:
                        self.pa.send_handles_to(p)
                self.pa.recv_handles()
            else:
                blobs = comm.allgather(bytes(self.pa.ipc_handles()))
                for p, blob in enumerate(blobs):
                    if p != self.rank:
                        self.pa.ipc_open(p, blob)
            comm.Barrier()
            self._try_multicast()
        self.barrier()
        torch.cuda.synchronize(self.device)
        comm.Barrier()
        return self

    def _try_multicast(self):
        want = os.environ.get("TMPI_NVLS", "1") != "0" and self.mode == "vmm"
        ok = bool(want and self.pa.multicast_supported())
        if not all(self.comm.allgather(ok)):
            return
        err = None
        try:
            if self.rank == 0:
                self.pa.mc_create_and_send()
        except Exception as e:  # noqa: BLE001
            err = repr(e)
        errs = self.comm.allgather(err)
        if any(errs):
            self.multicast_error = "create: %s" % [e for e in errs if e]
            if self.comm.rank == 0:
                print("[symmetric] NVLS multicast unavailable (%s)" % self.multicast_error)
            return
        steps = [self.pa.mc_recv, self.pa.mc_add_device, self.pa.mc_bind_and_map]
        for fn in steps:
            err = None
            try:
                fn()
            except Exception as e:  # noqa: BLE001
                err = repr(e)
            errs = self.comm.allgather(err)
            if any(errs):
                self.multicast_error = "%s: %s" % (fn.__name__, [e for e in errs if e])
                if self.comm.rank == 0:
                    print("[symmetric] NVLS multicast unavailable (%s)" % self.multicast_error)
                return
        self.has_multicast = True

    # ------------------------------------------------------------------ tensors over (peer) memory
    def alloc(self, nbytes):
        """Arena allocator handed to :class:`FlatArena` (must be called once, by all ranks)."""
        if self.pa is None:
            self.create(nbytes)
        assert nbytes <= self.nbytes
        return self.local_bytes()[:nbytes]

    def local_bytes(self):
        return self.peer_bytes(self.rank)

    def peer_bytes(self, p):
        if p not in self._tensors:
            self._tensors[p] = tensor_from_ptr(self.pa.arena_ptr(p), self.nbytes, self.device, self.pa)
        return self._tensors[p]

    def peer_region(self, p, byte_off, numel, dtype=torch.float32):
        nb = numel * torch.empty((), dtype=dtype).element_size()
        return self.peer_bytes(p)[byte_off:byte_off + nb].view(dtype)

    def proto_words(self, p):
        """int32 view of rank ``p``'s protocol words (tail of its signal pad): EASGD ticket lock, GOSGD inbox / acks —
        layout in ``csrc/comm_kernels.cu``."""
        key = ("proto", p)
        if key not in self._tensors:
            off = int(self.pa.proto_words_offset())
            self._tensors[key] = tensor_from_ptr(self.pa.sig_ptr(p) + off, 4096, self.device, self.pa).view(torch.int32)
        return self._tensors[key]

    # ------------------------------------------------------------------ device-side ticket lock (EASGD center)
    def ticket_acquire(self, owner, state):
        self.pa.ticket_acquire(int(owner), state.data_ptr(), self._stream())

    def ticket_release(self, owner, state):
        self.pa.ticket_release(int(owner), state.data_ptr(), self._stream())

    # ------------------------------------------------------------------ kernels
    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    def _blocks(self, max_blocks):
        if max_blocks:
            return int(max_blocks)
        if self.max_blocks:
            return self.max_blocks
        return 2 * torch.cuda.get_device_properties(self.device).multi_processor_count

    def barrier(self):
        """Device-side flag barrier across the node's ranks (one tiny kernel)."""
        self.pa.device_barrier(self._stream())

    def pick_algo(self, nbytes, algo="auto"):
        """Size-based one-shot / two-shot / NVLS switch (SURVEY §5.8): one-shot moves
        (N−1)× the bytes but has a single barrier pair and no push phase — best for the
        small buckets; two-shot (or NVLS when a multicast mapping exists) is
        bandwidth-optimal for the big ones."""
        if algo != "auto":
            if algo == "nvls" and not self.has_multicast:
                return ALGO["twoshot"]
            return ALGO[algo]
        # measured crossovers (profiles/allreduce_sweep.md): 8 ranks — two-shot/NVLS wins from 16 KiB up;
        # 2 ranks — one-shot is on par up to a few MiB (a single barrier pair, no push phase)
        default = 2 << 20 if self.size == 2 else (64 << 10 if self.size <= 4 else 8 << 10)
        thresh = int(os.environ.get("TMPI_ONESHOT_BYTES", str(default)))
        if nbytes <= thresh:
            return ALGO["oneshot"]
        return ALGO["nvls"] if self.has_multicast else ALGO["twoshot"]

    def fused_allreduce_sgd(self, arena, lo, hi, mu, nesterov, inv_k=None, algo="auto", wire16=False, max_blocks=None,
                            pre_reduced=False, push_master=True):
        """``pre_reduced``: the range's gradients were already reduce-scattered into their owner's G by the wgrad GEMM
        epilogues (``configure_gemm_rs`` / ``gemm_rs_add_range``) — the kernel skips the gather, updates its slice, pushes
        W / H and clears G."""
        from ..ops.cuda_impl import _table
        lrm, wd, ex = _table(arena)
        h_off = arena.layout["H"] if arena.H is not None else -1
        a = self.pick_algo((hi - lo) * (2 if wire16 else 4), algo)
        if pre_reduced and a == ALGO["oneshot"]:
            a = ALGO["nvls"] if self.has_multicast else ALGO["twoshot"]
        self.pa.fused_allreduce_sgd(arena.layout["W"], arena.layout["G"], arena.layout["U"], h_off, arena.layout["R"],
                                    arena.block_group.data_ptr(), lrm, wd, ex, arena.hyper.data_ptr(), float(mu),
                                    int(bool(nesterov)), float(inv_k if inv_k is not None else 1.0 / self.size),
                                    int(lo), int(hi), int(bool(wire16)), a, self._blocks(max_blocks), self._stream(),
                                    int(bool(pre_reduced)), int(bool(push_master)))
        return a

    def fused_allreduce_adam(self, arena, lo, hi, b1, b2, eps, inv_k=None, algo="auto", wire16=False, max_blocks=None,
                             push_master=True):
        """Average the ranks' gradients of ``[lo, hi)`` and take one Adam step (moments in the arena's U and V regions, step
        counter ``arena.adam_t``, which this call reads but does not advance: the caller advances it once per optimizer step
        with :meth:`adam_advance`).  Same algorithms, wire formats and owner-keeps-master mode as :meth:`fused_allreduce_sgd`;
        two-shot updates the moments on the owner of a slice only (:meth:`push_region_slices` re-synchronises them)."""
        from ..ops.cuda_impl import _table
        if "V" not in arena.layout:
            raise ValueError("fused Adam needs an arena built with optimizer='adam' (V region in the symmetric allocation)")
        lrm, wd, ex = _table(arena)
        h_off = arena.layout["H"] if arena.H is not None else -1
        a = self.pick_algo((hi - lo) * (2 if wire16 else 4), algo)
        self.pa.fused_allreduce_adam(arena.layout["W"], arena.layout["G"], arena.layout["U"], arena.layout["V"], h_off,
                                     arena.layout["R"], arena.block_group.data_ptr(), lrm, wd, ex, arena.hyper.data_ptr(),
                                     arena.adam_t.data_ptr(), float(b1), float(b2), float(eps),
                                     float(inv_k if inv_k is not None else 1.0 / self.size), int(lo), int(hi), int(bool(wire16)), a,
                                     self._blocks(max_blocks), self._stream(), int(bool(push_master)))
        return a

    def adam_advance(self, arena):
        """``arena.adam_t += 1`` on the current stream (one tiny kernel; graph-capturable)."""
        self.L.adam_advance(arena.adam_t.data_ptr(), self._stream())

    def push_region_slices(self, arena, region, lo, hi, max_blocks=None):
        """All ranks: push the slice of fp32 region ``region`` ('W', 'U', 'V') each rank owns in the two-shot partition of
        ``[lo, hi)`` to the peers."""
        from ..ops.cuda_impl import _table
        lrm, wd, ex = _table(arena)
        self.pa.push_region_slices(arena.layout[region], arena.block_group.data_ptr(), lrm, wd, ex, int(lo), int(hi),
                                   self._blocks(max_blocks), self._stream())

    def push_master_slices(self, arena, lo, hi, max_blocks=None):
        """All ranks: push the fp32 master weights of the slice each rank owns in the two-shot partition of ``[lo, hi)`` to the
        peers (re-synchronises ``W`` after fused steps that ran with ``push_master=False``)."""
        self.push_region_slices(arena, "W", lo, hi, max_blocks)

    def configure_gemm_rs(self, arena, ranges):
        """Arm the reduce-scatter epilogue of the GEMM for the given single-tensor buckets ``[(lo, hi), …]`` (element ranges
        of the arena): fp32 GEMM outputs written into those parts of ``arena.G`` are red.add-ed into the owner rank's G."""
        self.pa.configure_gemm_rs(int(arena.layout["G"]))
        g0 = arena.G.data_ptr()
        for lo, hi in ranges:
            nb = (hi - lo) // self.L.ARENA_BLOCK
            per = (nb + self.size - 1) // self.size
            self.L.gemm_rs_add_range(g0 + lo * 4, g0 + hi * 4, lo // self.L.ARENA_BLOCK, per)

    def allreduce(self, arena, src, dst, scale, lo=0, hi=None, algo="auto", refresh_shadow=False, skip_local=True,
                  max_blocks=None):
        from ..ops.cuda_impl import _table
        lrm, wd, ex = _table(arena)
        hi = arena.numel if hi is None else hi
        a = self.pick_algo((hi - lo) * 4, algo)
        if src == dst and a == ALGO["oneshot"]:
            a = ALGO["nvls"] if self.has_multicast else ALGO["twoshot"]
        h_off = arena.layout["H"] if (refresh_shadow and arena.H is not None) else -1
        self.pa.allreduce_flat(arena.layout[src], arena.layout[dst], h_off, arena.block_group.data_ptr(), lrm, wd, ex,
                               float(scale), int(lo), int(hi), int(bool(skip_local)), a, self._blocks(max_blocks), self._stream())
        return a
