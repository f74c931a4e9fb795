#!/usr/bin/env python
"""Benchmarks of the BASELINE.json configs: seconds per 5120 images (the reference's Recorder print period).

    python bench.py --gpus N --steps K --warmup W                                   # AlexNet-128b BSP (flagship), N = 1
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W [--model M] [--rule R] [--dtype D]

    --model  alexnet | googlenet | vgg16 | resnet50 | wrn       (batch per GPU as published: 128 / 32 / 32 / 64 / 128)
    --rule   bsp | easgd | gosgd       (easgd: rank 0 holds the center, N-1 workers, tau = --tau; gosgd: N gossiping workers)
    --dtype  bf16 | tf32               (bf16: bf16 operands, fp32 accumulate, fp32 master weights;
                                        tf32: fp32 storage end to end, tcgen05 kind::tf32 — the reference's precision class)
    --impl   ours | reference | torch_best | nccl_baseline

One rank per GPU.  Two timed regions per run, both bracketed by barrier + synchronize and timed with CUDA events, max over
ranks; each region is repeated ``--repeats`` times (K steps each) and the MEDIAN is reported together with min / max:

* ``value``  — K training steps (forward + backward + gradient exchange + optimizer update) on a device-resident batch:
  the reference's "train + comm" metric (file-wait excluded, ``speedup-n_workers.ipynb:53-55``).
* ``e2e``    — the same K steps through the public API (``model.train_iter`` + ``exchanger.exchange``): every step the
  loader copies a fresh uint8 batch from pinned host memory (H2D) and the host reads the step's loss back (D2H).

The device-resident batch of the ``value`` region is drawn from a fixed seed, so runs with the same arguments see the same
inputs; ``--dump-outputs DIR`` writes what the last step of that region returned, and the weights it left, as ``DIR/*.npy``
so that two builds can be compared output for output.

``--impl reference`` runs the unmodified reference from ``baseline/_ref`` if it can run (it cannot in this image: Theano /
pygpu / mpi4py / mpirun are not installable offline).  ``--impl torch_best`` is the strongest same-semantics LIBRARY build
(cuDNN / cuBLAS channels-last, CUDA-graph-captured step, fused foreach momentum-SGD, one flat-bucket ncclAllReduce);
``--impl nccl_baseline`` is the reference-*semantics* one (per-tensor ncclAllReduce + per-tensor updates, eager).
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# BASELINE.md: published seconds per 5120 images (train + comm), K80
K80_PUBLISHED = {
    "alexnet": {1: 20.50, 2: 10.35 + 0.78, 4: 5.13 + 0.54, 8: 2.63 + 0.61},
    "googlenet": {1: 63.89, 2: 31.40 + 1.00, 4: 15.51 + 0.71, 8: 7.69 + 0.80},
    "vgg16": {1: 343.37, 2: 169.12 + 7.14, 4: 86.97 + 4.80, 8: 43.29 + 5.41},
    "resnet50": {1: 163.15, 2: 80.09 + 0.81, 4: 40.25 + 0.56, 8: 20.12 + 0.57},
}
MODELS = {
    "alexnet": ("theanompi_b200.models.alex_net", "AlexNet", dict(batch_size=128, file_batch_size=128), "3x227x227"),
    "googlenet": ("theanompi_b200.models.googlenet", "GoogLeNet", dict(batch_size=32, file_batch_size=128), "3x224x224"),
    "vgg16": ("theanompi_b200.models.lasagne_model_zoo.vgg16", "VGG16", dict(batch_size=32, file_batch_size=128), "3x224x224"),
    "resnet50": ("theanompi_b200.models.lasagne_model_zoo.resnet50", "ResNet50", dict(batch_size=64, file_batch_size=64), "3x224x224"),
    "wrn": ("theanompi_b200.models.keras_model_zoo.wresnet", "Wide_ResNet", dict(batch_size=128, file_batch_size=128), "3x32x32"),
}
INPUT_SEED = 1234          # the device-resident batch of the timed region: the same pixels and labels on every run
DUMP_WEIGHTS = 1 << 22     # --dump-outputs: weights sampled beyond this many values (16 MiB of float32)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "torch_best", "nccl_baseline"])
    ap.add_argument("--model", default="alexnet", choices=sorted(MODELS))
    ap.add_argument("--rule", default="bsp", choices=["bsp", "easgd", "gosgd"])
    ap.add_argument("--dtype", default=os.environ.get("TMPI_DTYPE", "bf16"), choices=["bf16", "tf32"])
    ap.add_argument("--strategy", default=os.environ.get("TMPI_BENCH_STRATEGY", "fused"))
    ap.add_argument("--tau", type=int, default=4, help="EASGD: local steps per elastic exchange")
    ap.add_argument("--gosgd-p", type=float, default=0.1, help="GOSGD: push probability per step (reference default 0.01)")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-overlap", action="store_true")
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: the published one for the model)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last step of the device-timed region returned (cost.npy, error.npy) "
                         "and the weights it left (weights.npy: all of them, or a fixed seeded sample of %d) as float32 .npy files "
                         "(BSP rule, --impl ours)" % DUMP_WEIGHTS)
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.rule != "bsp"):
        ap.error("--dump-outputs needs --impl ours --rule bsp")
    return args


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def reference_arm(args):
    """Run the UNMODIFIED reference from baseline/_ref through its own public API."""
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    why = None
    if not os.path.isdir(os.path.join(ref_dir, "theanompi")):
        why = "baseline/_ref not installed"
    else:
        sys.path.insert(0, ref_dir)
        import shutil
        missing = []
        for mod in ("theano", "pygpu", "mpi4py", "hickle"):
            try:
                __import__(mod)
            except Exception:
                missing.append(mod)
        if shutil.which("mpirun") is None:
            missing.append("mpirun")
        if missing:
            why = ("reference installs (pure python) but cannot run: missing %s — Theano 0.9/libgpuarray/mpi4py/OpenMPI "
                   "are not in the offline wheelhouse and the code is Python-2 era" % ",".join(missing))
    if why is None:
        why = "reference import unexpectedly succeeded but no runnable stock path is wired"
    if int(os.environ.get("RANK", "0")) == 0:
        print(json.dumps({"impl": "reference", "unavailable": why}))
    return 0


# ---------------------------------------------------------------------------------------------------------------- helpers
class Timer(object):
    """R repeats of a K-step region, each bracketed by barrier + synchronize, CUDA events on the launching stream."""

    def __init__(self, world, dev):
        import torch
        self.torch, self.world, self.dev = torch, world, dev

    def barrier(self):
        if self.world > 1:
            self.torch.distributed.barrier()
        self.torch.cuda.synchronize()

    def region(self, fn, K):
        torch = self.torch
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        e0.record()
        out = None
        for i in range(K):
            out = fn(i)
        e1.record()
        self.barrier()
        return e0.elapsed_time(e1), out

    def max_over_ranks(self, values, group_ranks=None):
        torch = self.torch
        t = torch.tensor(values, dtype=torch.float64, device=self.dev)
        if self.world > 1:
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        return [float(v) for v in t]


def stats(ms_list, K):
    per = sorted(m / K for m in ms_list)
    return {"median": statistics.median(per), "min": per[0], "max": per[-1], "n": len(per),
            "spread_pct": 100.0 * (per[-1] - per[0]) / statistics.median(per)}


def model_cfg(args, name, world_for_data):
    """Model config for the bench: published per-GPU batch, synthetic data (the iterators wrap around, so a small file list is
    enough — the loader still copies a full file batch from pinned memory every file)."""
    modfile, cls, cfg, inp = MODELS[name]
    cfg = dict(cfg)
    if args.batch:
        ratio = max(1, cfg["file_batch_size"] // cfg["batch_size"])
        cfg["batch_size"] = args.batch
        cfg["file_batch_size"] = args.batch * ratio
    if name == "wrn":
        cfg["data_kwargs"] = dict(synthetic=True, n_synthetic=cfg["batch_size"] * 20 * world_for_data)
    else:
        cfg["data_kwargs"] = dict(n_train_files=16 * world_for_data, n_val_files=world_for_data, synthetic=True)
    cfg["dtype"] = args.dtype
    cfg["verbose"] = False
    return modfile, cls, cfg, inp


def set_device_batch(model, torch, dev):
    """Device-resident batch for the kernel-timed region (seeded random pixels of the model's input shape, random labels)."""
    shp = tuple(model.shared_x.shape)
    g = torch.Generator(device=dev)
    g.manual_seed(INPUT_SEED)
    model.shared_x = torch.randn(shp, device=dev, generator=g).to(model.act_dtype)
    hi = int(getattr(model, "n_softmax_out", 0) or getattr(model.data, "n_class", 10))
    model.shared_y.copy_(torch.randint(0, hi, (shp[0],), device=dev, generator=g))


def step_outputs(model, out, torch):
    """Host copies of what a training step hands back: its (cost, error) and the model's weights after the update — all of
    them, or a fixed seeded sample of DUMP_WEIGHTS values taken in parameter order."""
    import numpy as np
    cost, error = out[:2]
    w = torch.cat([p.detach().reshape(-1).float() for p in model.params])
    if w.numel() > DUMP_WEIGHTS:
        idx = np.sort(np.random.default_rng(0).choice(w.numel(), DUMP_WEIGHTS, replace=False))
        w = w[torch.from_numpy(idx).to(w.device)]
    return {"cost": cost.detach().float().reshape(1).cpu().numpy(), "error": error.detach().float().reshape(1).cpu().numpy(),
            "weights": w.cpu().numpy()}


def dump_outputs(out_dir, arrays):
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def e2e_loop(model, rec, step_extra, K, Wm, torch, start_count):
    """K steps through the public API, each with the loader's H2D and an async D2H read of the step's loss (consumed by the
    host one step later, the way a training loop logs it)."""
    loss_host = torch.empty(K, dtype=torch.float32).pin_memory()
    loss_evs, losses = [], []

    def one(i):
        model.train_iter(start_count + i, rec)
        step_extra(i)
        loss_host[i:i + 1].copy_(rec.train_info["cost"][-1].detach().reshape(1).float(), non_blocking=True)
        ev = torch.cuda.Event(); ev.record(); loss_evs.append(ev)
        if i >= 1:
            loss_evs[i - 1].synchronize()
            losses.append(float(loss_host[i - 1]))
        if i == K - 1:
            loss_evs[-1].synchronize()
            losses.append(float(loss_host[K - 1]))
        return losses
    return one


def emit(args, world, K, Wm, dev_stats, e2e_stats, extra, model_name, inp, batch, n_train_gpus, launches, h2d, loss, clocks, rule,
         strategy):
    steps_per_5120 = 5120.0 / (batch * n_train_gpus)
    sec = dev_stats["median"] * steps_per_5120 / 1000.0
    sec_e2e = e2e_stats["median"] * steps_per_5120 / 1000.0
    base = K80_PUBLISHED.get(model_name, {}).get(world) if rule == "bsp" else None
    cls = MODELS[model_name][1]
    metric = "%s-%db %s seconds per 5120 images (train+comm, device-timed, max over ranks)" % (cls, batch, rule.upper())
    out = {
        "metric": metric, "value": sec, "unit": "s/5120img", "n_gpus": world, "steps": K, "warmup": Wm,
        "ms_per_step": dev_stats["median"], "higher_is_better": False, "scaling": "weak",
        "vs_baseline": (sec / base) if base else None, "dtype": args.dtype, "data": "synthetic", "impl": "ours",
        "images_per_s": batch * n_train_gpus / (dev_stats["median"] / 1000.0),
        "repeats": {"n": dev_stats["n"], "ms_per_step_min": dev_stats["min"], "ms_per_step_max": dev_stats["max"],
                    "spread_pct": dev_stats["spread_pct"], "reported": "median"},
        "config": {"model": cls, "global_batch": batch * n_train_gpus, "seq_len": None, "input": inp,
                   "parallelism": "dp%d" % n_train_gpus, "rule": rule.upper(), "exch_strategy": strategy,
                   "push_master": os.environ.get("TMPI_PUSH_MASTER", "0") == "1",
                   "cuda_graph": not args.no_graph, "overlap": not args.no_overlap,
                   "l2": "per-step working set (weights + grads + momentum + activations) >> 126 MB L2; no flush"},
        "clocks": clocks,
        "e2e": {"value": sec_e2e, "unit": "s/5120img", "ms_per_step": e2e_stats["median"], "ms_per_step_min": e2e_stats["min"],
                "ms_per_step_max": e2e_stats["max"], "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                "d2h_mode": "async copy of each step's loss to pinned memory, read by the host one step later"},
        "gpu_launches": int(launches * K), "native_launches_per_step": int(launches), "final_loss": loss,
    }
    out.update(extra or {})
    print(json.dumps(out))


# ---------------------------------------------------------------------------------------------------------------- BSP
def run_bsp(args, rank, world, local):
    import torch
    from theanompi_b200.ops import native
    from theanompi_b200.worker import BSP_Worker

    K, Wm, R = args.steps, max(3, args.warmup), max(1, args.repeats)
    strategy = args.strategy if world > 1 else "fused"
    worker = BSP_Worker("cuda%d" % local, "cdd", strategy)
    modfile, cls, cfg, inp = model_cfg(args, args.model, world)
    full = worker.model_config(cls, cuda_graph=not args.no_graph, overlap=not args.no_overlap, **cfg)
    model = getattr(importlib.import_module(modfile), cls)(full)
    worker.build(model, full)
    rec, exch = worker.recorder, worker.exchanger
    dev = torch.device("cuda", local)
    T = Timer(world, dev)
    batch = model.batch_size
    n_subb = model.n_subb

    set_device_batch(model, torch, dev)

    def dev_step(i=0):
        out = model.train_iter_fn(i % n_subb)
        exch.exchange(rec)
        return out

    native.reset_launch_count()
    dev_step(0)
    launches = native.launch_count()
    for i in range(Wm + 2):
        dev_step(i)
    T.barrier()
    sampler = ClockSampler(local)
    sampler.start()
    dev_ms = []
    for _ in range(R):
        ms, last = T.region(dev_step, K)
        dev_ms.append(ms)
    outputs = step_outputs(model, last, torch) if args.dump_outputs else None

    # ---------------- end-to-end region through the public API (loader H2D + loss D2H every step)
    model.reset_iter("train")
    cnt = 0
    for i in range(Wm):
        model.train_iter(cnt, rec); exch.exchange(rec); cnt += 1
        float(rec.train_info["cost"][-1])
    e2e_ms, losses = [], []
    for _ in range(R):
        one = e2e_loop(model, rec, lambda i: exch.exchange(rec), K, Wm, torch, cnt)
        ms, losses = T.region(one, K)
        cnt += K
        e2e_ms.append(ms)
        rec.clear_train_info()
    clocks = sampler.stop()
    h2d = int(model.h2d_bytes_last) // n_subb

    dev_ms = [list(x) for x in zip(*[T.max_over_ranks([m]) for m in dev_ms])][0]
    e2e_ms = [list(x) for x in zip(*[T.max_over_ranks([m]) for m in e2e_ms])][0]
    if rank == 0:
        emit(args, world, K, Wm, stats(dev_ms, K), stats(e2e_ms, K), None, args.model, inp, batch, world, launches, h2d,
             losses[-1] if losses else None, clocks, "bsp", strategy if world > 1 else "local fused SGD")
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
    model.cleanup()
    worker.finalize()
    return 0


# ---------------------------------------------------------------------------------------------------------------- EASGD
def run_easgd(args, rank, world, local):
    """Rank 0 holds the center (no compute); ranks 1..N-1 train and run the elastic exchange every tau steps."""
    import torch
    import torch.distributed as dist
    from theanompi_b200.ops import native
    if world < 2:
        print(json.dumps({"impl": "ours", "rule": "EASGD", "unavailable": "EASGD needs >= 2 GPUs (center + workers)"}))
        return 0
    K, Wm, R, tau = args.steps, max(3, args.warmup), max(1, args.repeats), max(1, args.tau)
    nw = world - 1
    modfile, cls, cfg, inp = model_cfg(args, args.model, nw)
    dev = torch.device("cuda", local)
    Model = getattr(importlib.import_module(modfile), cls)
    T = Timer(world, dev)
    if rank == 0:
        from theanompi_b200.easgd_server import EASGD_Server
        server = EASGD_Server("cuda%d" % local)
        full = dict(cfg)
        full.update(verbose=False, rank=0, size=1, no_paraload=True, device=str(server.ctx), mname=cls,
                    arena_allocator=server.arena_allocator())
        model = Model(full)
        server.build(model)
        c0 = model.arena.W.clone()
        for _ in range(4 * R + 5):                      # mirrors the workers' barriers below (1 + 2R + 4 + 2R)
            T.barrier()
        dist.all_reduce(torch.zeros(4, dtype=torch.float64, device=dev), op=dist.ReduceOp.MAX)
        for _ in range(2 * R):
            dist.all_reduce(torch.zeros(1, dtype=torch.float64, device=dev), op=dist.ReduceOp.MAX)
        served = int(server.gpucomm.proto_words(0)[2].item())
        drift = float((model.arena.W - c0).abs().max())
        gathered = [None] * world
        dist.all_gather_object(gathered, None)
        res = [g for g in gathered if g]
        w = res[0]
        extra = {"easgd": {"tau": tau, "workers": nw, "alpha": 0.5, "lock": "lock-free red.add" if os.environ.get("TMPI_EASGD_LOCKFREE") == "1"
                           else "device-side ticket lock", "center_exchanges_served": served, "center_moved": drift > 0,
                           "exchange_us_contended": w["xch_us"], "exchange_GBps_per_worker_contended": w["xch_gbps"],
                           "center_link_GBps_each_direction": w["xch_gbps"] * nw / 2.0,
                           "exchange_us_alone": w["xch_us_alone"], "exchange_GBps_alone": w["xch_gbps_alone"],
                           "bytes_per_exchange_over_nvlink": w["xch_bytes"]}}
        emit(args, world, K, Wm, w["dev"], w["e2e"], extra, args.model, inp, w["batch"], nw, w["launches"], w["h2d"], w["loss"],
             w["clocks"], "easgd", "elastic kernel over NVLink peer memory")
        server.finalize()
        return 0

    from theanompi_b200.easgd_worker import EASGD_Worker
    worker = EASGD_Worker("cuda%d" % local)
    full = dict(cfg)
    full.update(verbose=False, rank=rank - 1, size=nw, mname=cls, device=str(worker.ctx), arena_allocator=worker.arena_allocator(),
                cuda_graph=not args.no_graph)
    model = Model(full)
    worker.build(model, full)
    rec, exch = worker.recorder, worker.exchanger
    batch, n_subb = model.batch_size, model.n_subb
    set_device_batch(model, torch, dev)

    def dev_step(i=0):
        out = model.train_iter_fn(i % n_subb)
        if (i + 1) % tau == 0:
            exch.exchange()
        return out

    native.reset_launch_count()
    dev_step(0)
    launches = native.launch_count()
    for i in range(Wm + 2):
        dev_step(i)
    T.barrier()
    sampler = ClockSampler(local)
    sampler.start()
    dev_ms = []
    for _ in range(R):
        T.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(K):
            dev_step(i)
        e1.record()
        T.barrier()
        dev_ms.append(e0.elapsed_time(e1))
    # exchange alone: all workers hammer the center back to back (contended), then worker 1 alone
    E = 10
    xb = 2 * model.arena.numel * 4
    T.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(E):
        exch.exchange()
    e1.record()
    T.barrier()
    xch_ms = e0.elapsed_time(e1) / E
    T.barrier()
    xa = 0.0
    if rank == 1:
        e0.record()
        for _ in range(E):
            exch.exchange()
        e1.record()
        torch.cuda.synchronize()
        xa = e0.elapsed_time(e1) / E
    T.barrier()
    # e2e: public API incl. loader + loss read-back (the control plane's progress reports are host messages: not sent here,
    # the server of this bench does not run its request loop)
    model.reset_iter("train")
    cnt = 0
    for i in range(Wm):
        model.train_iter(cnt, rec); cnt += 1
        float(rec.train_info["cost"][-1])
    e2e_ms, losses = [], []
    for _ in range(R):
        one = e2e_loop(model, rec, lambda i: exch.exchange() if (i + 1) % tau == 0 else None, K, Wm, torch, cnt)
        T.barrier()
        e0.record()
        for i in range(K):
            losses = one(i)
        e1.record()
        T.barrier()
        cnt += K
        e2e_ms.append(e0.elapsed_time(e1))
        rec.clear_train_info()
    clocks = sampler.stop()
    t = torch.tensor([xch_ms, xa, 0, 0], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    xch_ms, xa = float(t[0]), float(t[1])
    red = []
    for m in dev_ms + e2e_ms:
        tt = torch.tensor([m], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        red.append(float(tt[0]))
    dev_ms, e2e_ms = red[:R], red[R:]
    payload = None
    if rank == 1:
        payload = dict(dev=stats(dev_ms, K), e2e=stats(e2e_ms, K), batch=batch, launches=launches, h2d=int(model.h2d_bytes_last) // n_subb,
                       loss=losses[-1] if losses else None, clocks=clocks, xch_us=xch_ms * 1000.0, xch_gbps=xb / (xch_ms / 1000.0) / 1e9,
                       xch_us_alone=xa * 1000.0, xch_gbps_alone=xb / (xa / 1000.0) / 1e9 if xa > 0 else None, xch_bytes=xb)
    gathered = [None] * world
    dist.all_gather_object(gathered, payload)
    model.cleanup()
    worker.finalize()
    return 0


# ---------------------------------------------------------------------------------------------------------------- GOSGD
def run_gosgd(args, rank, world, local):
    import torch
    import torch.distributed as dist
    from theanompi_b200.ops import native
    from theanompi_b200.gosgd_worker import GOSGD_Worker
    if world < 2:
        print(json.dumps({"impl": "ours", "rule": "GOSGD", "unavailable": "GOSGD needs >= 2 GPUs"}))
        return 0
    K, Wm, R = args.steps, max(3, args.warmup), max(1, args.repeats)
    modfile, cls, cfg, inp = model_cfg(args, args.model, world)
    worker = GOSGD_Worker("cuda%d" % local)
    full = dict(cfg)
    full.update(verbose=False, rank=rank, size=world, mname=cls, device=str(worker.ctx), arena_allocator=worker.arena_allocator(),
                gosgd_p=args.gosgd_p, cuda_graph=not args.no_graph)
    model = getattr(importlib.import_module(modfile), cls)(full)
    worker.build(model, full)
    rec, exch = worker.recorder, worker.exchanger
    dev = torch.device("cuda", local)
    T = Timer(world, dev)
    batch, n_subb = model.batch_size, model.n_subb
    set_device_batch(model, torch, dev)

    def gossip(i):
        exch.process_messages(None)
        if exch.draw():
            d = exch.choose()
            if d is not None:
                exch.push_message(d, None)

    def dev_step(i=0):
        out = model.train_iter_fn(i % n_subb)
        gossip(i)
        return out

    native.reset_launch_count()
    dev_step(0)
    launches = native.launch_count()
    for i in range(Wm + 2):
        dev_step(i)
    T.barrier()
    sampler = ClockSampler(local)
    sampler.start()
    dev_ms = [T.region(dev_step, K)[0] for _ in range(R)]
    torch.cuda.synchronize()
    pushed, skipped, merged = exch.device_counters()
    # merge alone: every rank pull-merges its right neighbour's snapshot E times (all links busy at once)
    E = 10
    a = model.arena
    nb = a.numel * 4
    src = worker.gpucomm.peer_region((rank + 1) % world, a.layout["R"], a.numel)
    L = native.require()
    T.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(E):
        L.gosgd_merge(a.W.data_ptr(), a.H.data_ptr() if a.H is not None else 0, src.data_ptr(), 0.5, 0.5, a.numel,
                      worker.gpucomm._blocks(None), worker.gpucomm._stream())
    e1.record()
    T.barrier()
    merge_ms = e0.elapsed_time(e1) / E

    model.reset_iter("train")
    cnt = 0
    for i in range(Wm):
        model.train_iter(cnt, rec); gossip(i); cnt += 1
        float(rec.train_info["cost"][-1])
    e2e_ms, losses = [], []
    for _ in range(R):
        one = e2e_loop(model, rec, gossip, K, Wm, torch, cnt)
        ms, losses = T.region(one, K)
        cnt += K
        e2e_ms.append(ms)
        rec.clear_train_info()
    clocks = sampler.stop()
    exch.finish(None)
    alphas = worker.comm.allgather(exch.alpha)
    counts = worker.comm.allgather((exch.n_pushed, getattr(exch, "n_skipped", 0), exch.n_merged))
    red = T.max_over_ranks(dev_ms + e2e_ms + [merge_ms])
    dev_ms, e2e_ms, merge_ms = red[:R], red[R:2 * R], red[-1]
    if rank == 0:
        tot_push = sum(c[0] for c in counts)
        dev_s = stats(dev_ms, K)
        extra = {"gosgd": {"p": args.gosgd_p, "workers": world, "pushes": tot_push, "pushes_skipped_busy": sum(c[1] for c in counts),
                           "merges": sum(c[2] for c in counts), "sum_push_sum_weights": sum(alphas),
                           "pushes_per_s": pushed * world / max(1e-9, (sum(dev_ms) / 1000.0)),
                           "merge_us": merge_ms * 1000.0, "merge_GBps_per_rank": nb / (merge_ms / 1000.0) / 1e9,
                           "bytes_per_merge_over_nvlink": nb, "protocol": "device-side inbox / ack words in the signal pads"}}
        emit(args, world, K, Wm, dev_s, stats(e2e_ms, K), extra, args.model, inp, batch, world, launches,
             int(model.h2d_bytes_last) // n_subb, losses[-1] if losses else None, clocks, "gosgd", "pull-merge kernel over NVLink peer memory")
    model.cleanup()
    worker.finalize()
    return 0


def main():
    args = parse()
    if args.impl == "reference":
        return reference_arm(args)

    import torch
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", str(rank)))
    if world != args.gpus and world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, world))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device")
    torch.cuda.set_device(local)
    os.environ["TMPI_DTYPE"] = args.dtype

    if args.impl in ("nccl_baseline", "torch_best"):
        from theanompi_b200 import baseline_torch
        K, Wm = args.steps, max(3, args.warmup)
        if not args.batch:
            args.batch = MODELS[args.model][2]["batch_size"]
        fn = baseline_torch.run_baseline if args.impl == "nccl_baseline" else baseline_torch.run_torch_best
        return fn(args, rank, world, local, K, Wm, ClockSampler, K80_PUBLISHED.get(args.model, {}))
    if args.rule == "easgd":
        return run_easgd(args, rank, world, local)
    if args.rule == "gosgd":
        return run_gosgd(args, rank, world, local)
    return run_bsp(args, rank, world, local)


if __name__ == "__main__":
    sys.exit(main())
