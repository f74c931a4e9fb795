"""Multi-process CPU (gloo) checks, launched by tests/test_distributed_cpu.py with RANK/WORLD_SIZE set.

    python tests/mp_cpu_checks.py <case> [case arguments]
"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def _proc():
    from theanompi_b200.parallel.base import MPI_GPU_Process
    rank = int(os.environ["RANK"])
    p = MPI_GPU_Process("cpu%d" % rank)
    p.get_intranode_comm()
    return p


def case_strategies():
    """Every allreduce strategy vs a ground-truth sum on the reference's 230,400-float vector
    (test/test-exchanger/test_exchanger.py:39-46) — BASELINE config #1."""
    from theanompi_b200.parallel import exchanger_strategy as ES
    p = _proc()
    rank, size = p.rank, p.size
    shapes = [(230400,), (96, 11, 11, 3), (37,), (1000, 129)]
    for name in ["ar", "nccl32", "nccl16", "asa32", "asa16", "copper", "copper16"]:
        for avg in (False, True):
            rs = np.random.RandomState(100 + rank)
            src = [torch.from_numpy(rs.randn(*s).astype(np.float32)) for s in shapes]
            dst = [torch.zeros_like(t) for t in src]
            all_src = []
            for r in range(size):
                rr = np.random.RandomState(100 + r)
                all_src.append([rr.randn(*s).astype(np.float32) for s in shapes])
            want = [sum(all_src[r][i] for r in range(size)) / (size if avg else 1.0) for i in range(len(shapes))]
            cls = {"ar": ES.Exch_allreduce, "nccl32": ES.Exch_nccl32, "nccl16": ES.Exch_nccl16, "asa32": ES.Exch_asa32,
                   "asa16": ES.Exch_asa16, "copper": ES.Exch_copper, "copper16": ES.Exch_copper16}[name]
            ex = cls(p.comm, avg=avg) if name not in ("nccl32", "nccl16") else cls(p.comm, None, avg=avg)
            ex.prepare(p.ctx, src, dst)
            ex.exchange()
            tol = 2e-2 if name.endswith("16") else 1e-5
            for d, w in zip(dst, want):
                err = float((d - torch.from_numpy(w)).abs().max())
                assert err < tol * max(1.0, float(np.abs(w).max())), (name, avg, err)
    # swap: partners exchange parameters
    ex = ES.Exch_swap(p.comm)
    mine = [torch.full((5,), float(rank))]
    ex.prepare(p.ctx, mine)
    ex.exchange()
    if size == 2:
        assert float(mine[0][0]) == float(1 - rank)
    ex.replace(winner_ranks=[0])
    p.comm.Barrier()
    print("OK strategies rank", rank)


def case_mailbox():
    p = _proc()
    c = p.comm
    if c.rank == 0:
        got = sorted(c.recv(tag=7) for _ in range(c.size - 1))            # ANY_SOURCE
        assert got == list(range(1, c.size)), got
        for r in range(1, c.size):
            c.send({"hello": r}, r, tag=8)
        assert not c.iprobe(tag=99)
    else:
        c.send(c.rank, 0, tag=7)
        assert c.recv(source=0, tag=8) == {"hello": c.rank}
    assert c.bcast("x" if c.rank == 0 else None, root=0) == "x"
    assert c.allgather(c.rank) == list(range(c.size))
    c.Barrier()
    print("OK mailbox rank", c.rank)


def _tiny_model(p, sync_type, strategy, n_steps=6, lr=0.02):
    from theanompi_b200.models.cifar10 import Cifar10_model
    from theanompi_b200.parallel.exchanger import BSP_Exchanger
    from theanompi_b200.utils.recorder import Recorder
    from theanompi_b200.models import layers2
    layers2.reseed()
    cfg = dict(verbose=False, rank=p.rank, size=p.size, device="cpu", batch_size=16, file_batch_size=16, learning_rate=lr,
               data_kwargs=dict(n_synthetic=640, synthetic=True))
    m = Cifar10_model(cfg)
    from theanompi_b200.models.layers2 import Dropout, Crop
    Dropout.SetDropoutOff(); Crop.SetRandCropOff()       # deterministic comparison
    m.compile_iter_fns(sync_type)
    ex = BSP_Exchanger(p.comm, None, strategy, sync_type, p.ctx, m)
    rec = Recorder(p.comm, 1000, "t", False, device="cpu")
    for i in range(n_steps):
        m.train_iter(i, rec)
        ex.exchange(rec)
    return m


def case_bsp_equivalence(out_dir):
    """2 ranks × batch 16 with cdd exchange ≡ 1 process × batch 32 (the reference's
    test-cdd-train idea with real asserts), for the host and 'nccl32'-semantics strategies.
    Rank 0 writes the final weights of each strategy to ``out_dir/bsp_<strategy>.pt``."""
    p = _proc()
    for strat in ("ar", "nccl32", "asa32"):
        m = _tiny_model(p, "cdd", strat)
        ws = p.comm.allgather(m.arena.W.clone())
        assert torch.equal(ws[0], ws[1]), "replicas diverged (%s)" % strat
        if p.rank == 0:
            torch.save(m.arena.W.clone(), os.path.join(out_dir, "bsp_%s.pt" % strat))
    p.comm.Barrier()
    print("OK bsp rank", p.rank)


def case_bsp_avg():
    p = _proc()
    m = _tiny_model(p, "avg", "ar")
    ws = p.comm.allgather(m.arena.W.clone())
    assert torch.equal(ws[0], ws[1])
    print("OK bsp avg rank", p.rank)


if __name__ == "__main__":
    globals()["case_" + sys.argv[1]](*sys.argv[2:])
    if dist.is_initialized():
        dist.barrier()
        dist.destroy_process_group()
