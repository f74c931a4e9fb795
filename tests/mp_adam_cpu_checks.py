"""Multi-process CPU (gloo) checks of data-parallel Adam, launched by tests/test_adam_bsp_cpu.py with RANK/WORLD_SIZE set.

    python tests/mp_adam_cpu_checks.py <case> [case arguments]
"""
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

LR = 1e-3
STEPS = 6


def _proc():
    from theanompi_b200.parallel.base import MPI_GPU_Process
    rank = int(os.environ["RANK"])
    p = MPI_GPU_Process("cpu%d" % rank)
    p.get_intranode_comm()
    return p


def _tiny_adam_model(p, strategy):
    from theanompi_b200.models import layers2
    from theanompi_b200.models.cifar10 import Cifar10_model
    from theanompi_b200.models.layers2 import Crop, Dropout
    from theanompi_b200.parallel.exchanger import BSP_Exchanger
    from theanompi_b200.utils.recorder import Recorder
    layers2.reseed()
    cfg = dict(verbose=False, rank=p.rank, size=p.size, device="cpu", batch_size=16, file_batch_size=16, learning_rate=LR,
               optimizer="adam", data_kwargs=dict(n_synthetic=640, synthetic=True))
    m = Cifar10_model(cfg)
    Dropout.SetDropoutOff(); Crop.SetRandCropOff()       # deterministic comparison
    m.compile_iter_fns("cdd")
    ex = BSP_Exchanger(p.comm, None, strategy, "cdd", p.ctx, m)
    rec = Recorder(p.comm, 1000, "t", False, device="cpu")
    for i in range(STEPS):
        m.train_iter(i, rec)
        ex.exchange(rec)
    return m


def case_bsp_equivalence(out_dir):
    """2 ranks x batch 16 with cdd Adam on classic strategies; rank 0 writes the final weights and the step counter of each
    strategy to ``out_dir/adam_<strategy>.pt``."""
    p = _proc()
    for strat in ("ar", "nccl32", "asa32"):
        m = _tiny_adam_model(p, strat)
        assert int(m.arena.adam_t) == STEPS, int(m.arena.adam_t)
        ws = p.comm.allgather((m.arena.W.clone(), m.arena.U.clone(), m.arena.V.clone()))
        for a, b in zip(ws[0], ws[1]):
            assert torch.equal(a, b), "replicas diverged (%s)" % strat
        if p.rank == 0:
            torch.save({"W": m.arena.W.clone(), "t": int(m.arena.adam_t)}, os.path.join(out_dir, "adam_%s.pt" % strat))
    p.comm.Barrier()
    print("OK adam bsp rank", p.rank)


if __name__ == "__main__":
    globals()["case_" + sys.argv[1]](*sys.argv[2:])
    if dist.is_initialized():
        dist.barrier()
        dist.destroy_process_group()
