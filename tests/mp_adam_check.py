"""Multi-process GPU checks of the fused all-reduce + Adam exchange.  Launched by ``tests/test_gpu_adam_fused.py`` as

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        tests/mp_adam_check.py <case> [args]

cases
  kernels              every fused algorithm x wire16 x push_master through BSP_Exchanger, 3 steps over >= 2 buckets, against an
                       fp64 torch "average the all-gathered gradients, then Adam"; the step captured in a CUDA graph and replayed
                       5 times; checkpoint / resume; fused_rs rejected
  wrn <strategy> <n>   native Wide_ResNet, BSP cdd, n steps: prints the training-loss curve
"""
import json
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

LR, B1, B2, EPS, WD = 1e-2, 0.9, 0.999, 1e-8, 5e-4


class _AdamModel(object):
    """The part of the model contract the fused exchanger reads."""
    optimizer = "adam"
    mu, use_momentum, use_nesterov_momentum = 0.9, True, False

    def __init__(self, arena):
        from theanompi_b200.utils.opt import FlatAdam
        self.arena = arena
        self.adam = FlatAdam(arena, B1, B2, EPS)


def _ref_adam(w, m, v, g, lrm, wd, t):
    """fp64: ge = g + wd w; Adam step number t (1-based)."""
    ge = g + wd * w
    m.mul_(B1).add_(ge, alpha=1 - B1)
    v.mul_(B2).addcmul_(ge, ge, value=1 - B2)
    w.sub_(LR * lrm * (m / (1 - B1 ** t)) / ((v / (1 - B2 ** t)).sqrt() + EPS))


def case_kernels():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    from theanompi_b200.parallel.arena import FlatArena
    from theanompi_b200.parallel.exchanger import BSP_Exchanger
    from theanompi_b200.worker import BSP_Worker

    worker = BSP_Worker("cuda%d" % local, "cdd", "fused")
    dev, gc = worker.ctx, None
    alloc = worker.arena_allocator()
    gc = worker.gpucomm
    torch.manual_seed(1234)
    shapes = [(257, 300), (257,), (33,), (33,), (96, 11, 11, 3), (96,), (1023, 1029), (77,)]
    names = [None, None, "gamma", "beta", None, None, None, None]
    params = []
    for s, n in zip(shapes, names):
        p = torch.randn(s) * 0.1
        p.pname = n
        params.append(p)
    wtypes = ["W" if len(s) > 1 else "b" for s in shapes]
    arena = FlatArena(params, wtypes, dev, weight_decay=WD, allocator=alloc, with_recv=True, optimizer="adam")
    model = _AdamModel(arena)
    arena.hyper[0] = LR
    lrm, wdv, exv = arena.lr_mult_vector().double(), arena.wd_vector().double(), arena.exch_vector()
    real = torch.zeros(arena.numel, dtype=torch.bool, device=dev)
    for o, s in zip(arena.offsets, arena.sizes):
        real[o:o + s] = True
    results = dict(rank=rank, multicast=gc.has_multicast, numel=arena.numel)

    def reset():
        torch.manual_seed(7)
        w = torch.randn(arena.numel, device=dev) * 0.1
        dist.broadcast(w, 0)
        arena.W.copy_(w); arena.U.zero_(); arena.V.zero_(); arena.adam_t.zero_(); arena.refresh_shadow()
        torch.cuda.synchronize(); dist.barrier()
        return arena.W.double(), torch.zeros_like(arena.W, dtype=torch.float64), torch.zeros_like(arena.W, dtype=torch.float64)

    def grads(step):
        torch.manual_seed(1000 * step + rank)
        return torch.randn(arena.numel, device=dev)

    def ref_step(state, g, t, wire16):
        gl = [torch.empty_like(g) for _ in range(world)]
        dist.all_gather(gl, g)
        if wire16:
            gl = [x.to(torch.bfloat16).float() for x in gl]
        gavg = torch.stack([x.double() for x in gl]).sum(0) / world
        geff = torch.where(exv, gavg, g.double())             # BN groups: the rank's own gradient, no averaging
        _ref_adam(state[0], state[1], state[2], geff, lrm, wdv, t)

    def check(tag, state, t, tol):
        torch.cuda.synchronize(); dist.barrier()
        ew = float((arena.W.double() - state[0])[real].abs().max())
        assert ew < tol, (tag, ew)
        assert int(arena.adam_t) == t, (tag, int(arena.adam_t))
        for name in ("W", "U", "V", "H"):                      # BN groups are per-rank by design
            x = getattr(arena, name)[exv].contiguous()
            xl = [torch.empty_like(x) for _ in range(world)]
            dist.all_gather(xl, x)
            assert all(torch.equal(xl[0], y) for y in xl), (tag, name, "differs across ranks")
        return ew

    algos = ["oneshot", "twoshot"] + (["nvls"] if gc.has_multicast else [])
    for algo in algos:
        for wire16 in (False, True):
            for pm in (0, 1):
                os.environ["TMPI_PUSH_MASTER"] = str(pm)
                strat = algo + ("16" if wire16 else "")
                ex = BSP_Exchanger(worker.comm, gc, strat, "cdd", dev, model, overlap=True, bucket_bytes=1 << 20, comm_blocks=24)
                assert len(ex.buckets) >= 2 and ex.push_master == bool(pm)
                state = reset()
                for t in range(1, 4):
                    g = grads(t)
                    arena.G.copy_(g)
                    ref_step(state, g, t, wire16)
                    torch.cuda.synchronize(); dist.barrier()
                    ex.fused_step()
                ex.sync_master()
                # fp32 kernel vs fp64 reference: ~1e-6 of a step of ~lr; wire16 with NVLS also rounds the reduced sum to bf16
                results["%s_pm%d" % (strat, pm)] = check(strat, state, 3, 2e-4 if wire16 else 2e-5)
    os.environ.pop("TMPI_PUSH_MASTER", None)

    # the 2-bucket step captured in a CUDA graph, replayed 5 times: the counter advances once per replay, not per bucket
    ex = BSP_Exchanger(worker.comm, gc, "fused", "cdd", dev, model, overlap=True, bucket_bytes=1 << 20, comm_blocks=24)
    state = reset()
    g = grads(1)
    arena.G.copy_(g)
    torch.cuda.synchronize(); dist.barrier()
    graph = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream(device=dev)
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        with torch.cuda.graph(graph, stream=s):
            ex.fused_step()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize(); dist.barrier()
    assert int(arena.adam_t) == 0, "capture must not run the step"
    for t in range(1, 6):
        graph.replay()
        ref_step(state, g, t, False)
    torch.cuda.synchronize(); dist.barrier()
    ex.sync_master()
    results["graph"] = check("graph", state, 5, 2e-5)
    del graph

    # checkpoint / resume: 3 steps, sync, save, scramble, load, 3 more == 6 uninterrupted steps
    import tempfile
    finals = []
    for resume in (False, True):
        ex = BSP_Exchanger(worker.comm, gc, "fused", "cdd", dev, model, overlap=True, bucket_bytes=1 << 20, comm_blocks=24)
        reset()
        for t in range(1, 7):
            arena.G.copy_(grads(t))
            torch.cuda.synchronize(); dist.barrier()
            ex.fused_step()
            if resume and t == 3:
                ex.sync_master()
                sd = arena.state_dict()
                with tempfile.TemporaryDirectory() as d:
                    torch.save(sd, os.path.join(d, "ckpt.pt"))
                    arena.W.normal_(); arena.U.normal_(); arena.V.uniform_(); arena.adam_t.fill_(99); arena.refresh_shadow()
                    arena.load_state_dict(torch.load(os.path.join(d, "ckpt.pt")))
                torch.cuda.synchronize(); dist.barrier()
        ex.sync_master()
        finals.append({k: getattr(arena, k).clone() for k in ("W", "U", "V")} | {"t": int(arena.adam_t)})
    assert finals[0]["t"] == finals[1]["t"] == 6
    for k in ("W", "U", "V"):
        assert torch.equal(finals[0][k], finals[1][k]), ("resume", k)
    results["resume"] = True

    try:
        BSP_Exchanger(worker.comm, gc, "fused_rs", "cdd", dev, model)
    except ValueError:
        results["fused_rs_rejected"] = True
    assert results.get("fused_rs_rejected"), "fused_rs must reject Adam"

    torch.cuda.synchronize(); dist.barrier()
    if rank == 0:
        print("MP_ADAM_CHECK_OK " + json.dumps(results))
    worker.finalize()


def case_wrn(strategy, steps):
    """Native Wide_ResNet (small), BSP cdd: the per-step training loss of rank 0."""
    rank = int(os.environ["RANK"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    from theanompi_b200.models.keras_model_zoo.wresnet import Wide_ResNet
    from theanompi_b200.worker import BSP_Worker
    steps = int(steps)
    worker = BSP_Worker("cuda%d" % local, "cdd", strategy)
    cfg = worker.model_config("Wide_ResNet", batch_size=32, file_batch_size=32, depth=10, widen=2, learning_rate=1e-3,
                              data_kwargs=dict(n_synthetic=32 * 2 * steps, synthetic=True))
    model = Wide_ResNet(cfg)
    worker.build(model, cfg)
    rec, ex = worker.recorder, worker.exchanger
    for i in range(steps):
        model.train_iter(i, rec)
        ex.exchange(rec)
    losses = [float(c) for c in rec.train_info["cost"]]
    if hasattr(ex, "sync_master"):
        ex.sync_master()
    if rank == 0:
        print("MP_ADAM_WRN " + json.dumps(dict(strategy=strategy, t=int(model.arena.adam_t), losses=losses)))
    model.cleanup()
    worker.finalize()


if __name__ == "__main__":
    globals()["case_" + sys.argv[1]](*sys.argv[2:])
