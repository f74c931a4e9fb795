"""Flat parameter arena.

The reference keeps every parameter, momentum buffer (``vels``) and receive
buffer (``vels2``) as a separate GPU shared variable and therefore issues one
NCCL call and several elementwise kernels **per tensor** per iteration
(``theanompi/lib/exchanger_strategy.py:121-127``, ``theanompi/lib/opt.py:181-268``:
AlexNet 22 tensors, GoogLeNet 128).  Here all of them live in a handful of
contiguous fp32 regions of ONE allocation:

    W  master weights        (``model.params`` are *views* into it)
    G  gradients / send buf  (``model.vels`` views; backward kernels write here)
    U  momentum
    R  receive buffer        (``model.vels2`` views; only classic strategies use it)
    H  bf16 compute shadow of W (GPU only; written by the fused update kernel)
    V  Adam second moment    (``optimizer='adam'`` only; U then holds the first moment)

so that optimizer + collective become one or a few launches over a flat range,
and — when the allocation comes from the peer-mapped symmetric allocator
(:mod:`theanompi_b200.parallel.symmetric`) — peers can read/write the regions
directly over NVLink from inside a kernel.

Every tensor starts on a ``BLOCK``-element boundary; a one-byte-per-block
*group table* tells the flat kernels which hyper-parameter group a block
belongs to (lr multiplier, weight decay, exchanged-or-local), replacing the
reference's per-tensor Python branching on ``weight_type`` / BN names.
"""
from __future__ import annotations

import math

import numpy as np
import torch

BLOCK = 1024           # elements per block (4 KiB fp32): alignment + group granularity
MAX_GROUPS = 8

# group ids
G_W, G_B, G_BN_GAMMA, G_BN_BETA = 0, 1, 2, 3


def default_group(name, weight_type):
    """Reference rules: 'W' → lr·1 + weight decay; 'b' → lr·2, no decay
    (``opt.py:229-236``); params *named* gamma/beta are never exchanged
    (``exchanger.py:35-43``) and never decayed (``opt.py:211-216``)."""
    if name == "gamma":
        return G_BN_GAMMA
    if name == "beta":
        return G_BN_BETA
    return G_W if weight_type == "W" else G_B


class FlatArena(object):
    def __init__(self, params, weight_types=None, device=None, weight_decay=0.0,
                 shadow=None, with_recv=False, allocator=None, bias_lr_mult=2.0,
                 exchange_bn=False, optimizer="msgd"):
        self.params = list(params)
        n = len(self.params)
        if weight_types is None:
            weight_types = ["W" if p.dim() > 1 else "b" for p in self.params]
        self.weight_types = list(weight_types)
        self.device = torch.device(device) if device is not None else self.params[0].device
        self.sizes = [int(p.numel()) for p in self.params]
        self.offsets = []
        off = 0
        for s in self.sizes:
            self.offsets.append(off)
            off += int(math.ceil(s / BLOCK)) * BLOCK
        self.numel = off                      # padded element count (multiple of BLOCK)
        self.n_blocks = off // BLOCK
        self.n_real = sum(self.sizes)
        self.use_shadow = (self.device.type == "cuda") if shadow is None else bool(shadow)
        self.allocator = allocator
        self.optimizer = optimizer

        # ---- group table
        self.group_of = [default_group(getattr(p, "pname", None), wt)
                         for p, wt in zip(self.params, self.weight_types)]
        lr_mult = np.ones(MAX_GROUPS, dtype=np.float32)
        wd = np.zeros(MAX_GROUPS, dtype=np.float32)
        exch = np.ones(MAX_GROUPS, dtype=np.int32)
        lr_mult[G_B] = bias_lr_mult
        lr_mult[G_BN_BETA] = bias_lr_mult
        wd[G_W] = weight_decay
        if not exchange_bn:
            exch[G_BN_GAMMA] = 0
            exch[G_BN_BETA] = 0
        self.group_lr_mult_np, self.group_wd_np, self.group_exch_np = lr_mult, wd, exch
        bg = np.zeros(self.n_blocks, dtype=np.uint8)
        for o, s, g in zip(self.offsets, self.sizes, self.group_of):
            bg[o // BLOCK:(o + int(math.ceil(s / BLOCK)) * BLOCK) // BLOCK] = g
        self.block_group_np = bg

        # ---- storage: one allocation, carved into regions (256 B aligned)
        self._regions = {}
        want = ["W", "G", "U"] + (["R"] if with_recv else [])
        nbytes = 0
        layout = {}
        for r in want:
            layout[r] = nbytes
            nbytes += self.numel * 4
        if self.use_shadow:
            layout["H"] = nbytes
            nbytes += self.numel * 2
        if optimizer == "adam":                 # after H: SGD arenas keep their layout
            layout["V"] = nbytes
            nbytes += self.numel * 4
        self.nbytes = nbytes
        self.layout = layout
        if allocator is not None:
            self.raw = allocator(nbytes)
        else:
            self.raw = torch.zeros(nbytes, dtype=torch.uint8, device=self.device)
        assert self.raw.numel() >= nbytes
        for r in want:
            self._regions[r] = self.raw[layout[r]:layout[r] + self.numel * 4].view(torch.float32)
            self._regions[r].zero_()
        if self.use_shadow:
            self._regions["H"] = self.raw[layout["H"]:layout["H"] + self.numel * 2].view(torch.bfloat16)
            self._regions["H"].zero_()
        if "V" in layout:
            self._regions["V"] = self.raw[layout["V"]:layout["V"] + self.numel * 4].view(torch.float32)
            self._regions["V"].zero_()

        dev = self.device
        self.block_group = torch.from_numpy(bg).to(dev)
        self.group_lr_mult = torch.from_numpy(lr_mult).to(dev)
        self.group_wd = torch.from_numpy(wd).to(dev)
        self.group_exch = torch.from_numpy(exch).to(dev)
        # hyper-parameters live on the device so CUDA graphs never need re-capture:
        # [lr, mu, inv_k, nesterov_flag]
        self.hyper = torch.zeros(8, dtype=torch.float32, device=dev)
        # Adam bias-correction counter: optimizer steps taken so far (device memory, advanced once per step inside the graph)
        self.adam_t = torch.zeros(1, dtype=torch.int64, device=dev) if optimizer == "adam" else None
        self._bind()

    # ------------------------------------------------------------------ regions
    @property
    def W(self):
        return self._regions["W"]

    @property
    def G(self):
        return self._regions["G"]

    @property
    def U(self):
        return self._regions["U"]

    @property
    def H(self):
        return self._regions.get("H")

    @property
    def V(self):
        return self._regions.get("V")

    def ensure_adam_state(self):
        """V region + step counter of an arena built for another optimizer (a plain local buffer outside the allocation, like
        a late ``R``): enough for the local :class:`FlatAdam` step, not for the fused exchange."""
        if "V" not in self._regions:
            self._regions["V"] = torch.zeros(self.numel, dtype=torch.float32, device=self.device)
        if self.adam_t is None:
            self.adam_t = torch.zeros(1, dtype=torch.int64, device=self.device)

    @property
    def R(self):
        if "R" not in self._regions:
            self._regions["R"] = torch.zeros(self.numel, dtype=torch.float32, device=self.device)
        return self._regions["R"]

    def region_offset_bytes(self, name):
        return self.layout[name]

    # ------------------------------------------------------------------ binding
    def _bind(self):
        with torch.no_grad():
            for p, o, s in zip(self.params, self.offsets, self.sizes):
                view = self.W[o:o + s].view(p.shape)
                view.copy_(p.detach().to(self.device, torch.float32))
                p.data = view
                p.gbuf = self.G[o:o + s].view(p.shape)
                p.arena = self
                p.arena_off = o
                if self.use_shadow:
                    p.shadow = self.H[o:o + s].view(p.shape)
                    p.shadow.copy_(view)
                else:
                    p.shadow = None

    def views(self, region):
        """Per-parameter views of a region, in ``params`` order (``model.vels`` …)."""
        buf = getattr(self, region)
        return [buf[o:o + s].view(p.shape) for p, o, s in zip(self.params, self.offsets, self.sizes)]

    def exchanged_mask(self):
        """Per-parameter booleans: does the BSP exchanger touch this tensor?"""
        return [bool(self.group_exch_np[g]) for g in self.group_of]

    def refresh_shadow(self):
        if self.use_shadow:
            self.H.copy_(self.W)

    def zero_grad(self):
        self.G.zero_()

    def set_weight_decay(self, wd):
        self.group_wd_np[G_W] = wd
        self.group_wd = torch.from_numpy(self.group_wd_np).to(self.device)

    # ------------------------------------------------------------------ per-element expansions (reference path)
    def lr_mult_vector(self):
        if not hasattr(self, "_lr_vec"):
            self._lr_vec = self.group_lr_mult[self.block_group.long()].repeat_interleave(BLOCK)
        return self._lr_vec

    def wd_vector(self):
        return self.group_wd[self.block_group.long()].repeat_interleave(BLOCK)

    def exch_vector(self):
        if not hasattr(self, "_ex_vec"):
            self._ex_vec = self.group_exch[self.block_group.long()].repeat_interleave(BLOCK).bool()
        return self._ex_vec

    # ------------------------------------------------------------------ buckets (reverse layer order for overlap)
    def make_buckets(self, bucket_bytes, solo=(), tail_bytes=0):
        """Split the arena into contiguous block ranges.  Bucket 0 holds the LAST
        parameters (their gradients are ready first in backward).  Parameters listed in
        ``solo`` always get a bucket of their own."""
        target = max(BLOCK, int(bucket_bytes) // 4)
        buckets = []
        hi = self.numel
        i = len(self.params) - 1
        while i >= 0:
            lo = self.offsets[i]
            members = [i]
            while i not in solo and i - 1 >= 0 and (i - 1) not in solo and hi - self.offsets[i - 1] <= target:
                i -= 1
                lo = self.offsets[i]
                members.append(i)
            buckets.append({"lo": lo, "hi": hi, "params": members[::-1]})
            hi = lo
            i -= 1
        # The LAST bucket (the first layers) becomes ready only when backward ends: whatever it exchanges is exposed.  Split it so
        # that only a small tail (<= tail_bytes) waits for the very last gradients; the rest starts as soon as its own layers
        # are done.
        if tail_bytes and buckets and len(buckets[-1]["params"]) > 1 and not (set(buckets[-1]["params"]) & set(solo)):
            b = buckets[-1]
            tail_target = max(BLOCK, int(tail_bytes) // 4)
            if b["hi"] - b["lo"] > 2 * tail_target:
                ps = b["params"]
                k = 1
                while k < len(ps) - 1 and self.offsets[ps[k + 1]] - b["lo"] <= tail_target:
                    k += 1
                cut = self.offsets[ps[k]]
                if b["lo"] < cut < b["hi"]:
                    buckets[-1] = {"lo": cut, "hi": b["hi"], "params": ps[k:]}
                    buckets.append({"lo": b["lo"], "hi": cut, "params": ps[:k]})
        return buckets

    # ------------------------------------------------------------------ checkpoint
    def state_dict(self):
        sd = {"W": self.W.detach().cpu().clone(), "U": self.U.detach().cpu().clone(),
              "offsets": list(self.offsets), "sizes": list(self.sizes)}
        if self.V is not None:
            sd["V"] = self.V.detach().cpu().clone()
            sd["t"] = int(self.adam_t)
        return sd

    def load_state_dict(self, sd):
        assert list(sd["sizes"]) == list(self.sizes), "arena layout mismatch"
        with torch.no_grad():
            self.W.copy_(sd["W"].to(self.device))
            self.U.copy_(sd["U"].to(self.device))
            if self.V is not None and "V" in sd:
                self.V.copy_(sd["V"].to(self.device))
                self.adam_t.fill_(int(sd["t"]))
        self.refresh_shadow()
