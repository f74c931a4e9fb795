"""Synchronous data-parallel Adam on CPU (gloo): the classic cdd split (local Adam of the BN groups, all-reduce of G, Adam of
the exchanged groups on R / k) and the reference-path FlatAdam it is built from."""
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_PORT = [29760]


def run_ranks(n, case, *args, timeout=300):
    _PORT[0] += 1
    procs = []
    for r in range(n):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE=str(n), LOCAL_RANK=str(r), MASTER_ADDR="127.0.0.1",
                   MASTER_PORT=str(_PORT[0]), OMP_NUM_THREADS="2", PYTHONPATH=ROOT)
        procs.append(subprocess.Popen([sys.executable, os.path.join(ROOT, "tests", "mp_adam_cpu_checks.py"), case] + list(args),
                                      env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    outs = []
    for p in procs:
        try:
            o, _ = p.communicate(timeout=timeout)
        except subprocess.TimeoutExpired:
            for q in procs:
                q.kill()
            raise
        outs.append(o)
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0, "rank %d failed:\n%s" % (r, o[-3000:])
    return outs


def test_bsp_cdd_adam_two_ranks_equals_one_big_batch(tmp_path):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from mp_adam_cpu_checks import LR, STEPS
    run_ranks(2, "bsp_equivalence", str(tmp_path))
    # single process, batch 32 = the two shards of each step concatenated, then one Adam step on the mean gradient
    from theanompi_b200.models import layers2
    from theanompi_b200.models.cifar10 import Cifar10_model
    from theanompi_b200.models.layers2 import Crop, Dropout
    layers2.reseed()
    m = Cifar10_model(dict(verbose=False, rank=0, size=1, device="cpu", batch_size=16, file_batch_size=16, learning_rate=LR,
                           optimizer="adam", data_kwargs=dict(n_synthetic=640, synthetic=True)))
    Dropout.SetDropoutOff(); Crop.SetRandCropOff()
    m.compile_iter_fns("avg")
    d = m.data
    try:
        for step in range(STEPS):
            if step == 0:
                d.shuffle_data("train", common_seed=m.epoch)
            gsum = None
            for r in range(2):                               # what ranks 0 and 1 saw: shards [0::2] and [1::2]
                m.x_in.copy_(torch.from_numpy(np.ascontiguousarray(d.train_img_shuffle[2 * step + r])))
                m.y_in.copy_(torch.from_numpy(np.asarray(d.train_labels_shuffle[2 * step + r])))
                m._fwd_bwd_eager()
                gsum = m.arena.G.clone() if gsum is None else gsum + m.arena.G
            m.arena.G.copy_(gsum)
            m.adam.step(k=2)
    finally:
        Dropout.SetDropoutOn(); Crop.SetRandCropOn()
    assert int(m.arena.adam_t) == STEPS
    real = torch.zeros(m.arena.numel, dtype=torch.bool)
    for o, s in zip(m.arena.offsets, m.arena.sizes):
        real[o:o + s] = True
    for strat in ("ar", "nccl32", "asa32"):
        sd = torch.load(str(tmp_path / ("adam_%s.pt" % strat)))
        assert sd["t"] == STEPS
        diff = (sd["W"] - m.arena.W)[real].abs()
        # Adam normalises each element's step to about lr whatever the gradient's size, so an element whose averaged gradient
        # is ~0 moves by ~±lr on the sign of reduction-order noise (the two sides sum the shards in different orders).  Such
        # elements are rare; everywhere else the two computations agree to float32 rounding of a few steps.  One sign flip per
        # step bounds any element's difference by 2·lr per step.
        frac = float((diff <= 2e-5).float().mean())
        assert frac >= 0.9999, (strat, frac, float(diff.max()))
        assert float(diff.max()) <= 2 * LR * STEPS, (strat, float(diff.max()))


def test_flat_adam_split_matches_torch_adam():
    """Reference-path FlatAdam as the classic cdd split runs it: local step of the BN groups on G (no advance), then the
    exchanged groups on R with inv_k = 1/2 (advance) == torch.optim.Adam on the averaged gradient / the local one."""
    from theanompi_b200.parallel.arena import FlatArena
    from theanompi_b200.utils.opt import FlatAdam
    torch.manual_seed(11)
    shapes = [(37, 29), (37,), (19,), (19,), (5, 3, 3, 7)]
    names = [None, None, "gamma", "beta", None]
    params = []
    for s, n in zip(shapes, names):
        p = torch.randn(s) * 0.1
        p.pname = n
        params.append(p)
    wd = 5e-4
    arena = FlatArena(params, ["W", "b", "b", "b", "W"], "cpu", weight_decay=wd, bias_lr_mult=1.0, with_recv=True, optimizer="adam")
    exch = arena.exchanged_mask()
    assert exch == [True, True, False, False, True]
    ref = [p.detach().clone().double().requires_grad_(True) for p in arena.params]
    groups = [{"params": [q for q, wt in zip(ref, arena.weight_types) if wt == "W"], "weight_decay": wd},
              {"params": [q for q, wt in zip(ref, arena.weight_types) if wt != "W"], "weight_decay": 0.0}]
    lr = 1e-2
    opt = torch.optim.Adam(groups, lr=lr, betas=(0.9, 0.999), eps=1e-8)
    adam = FlatAdam(arena)
    arena.hyper[0] = lr
    for it in range(4):
        g_mine, g_peer = torch.randn(arena.numel), torch.randn(arena.numel)
        arena.G.copy_(g_mine)
        arena.R.copy_(g_mine + g_peer)
        for q, gv, rv, ex in zip(ref, arena.views("G"), arena.views("R"), exch):
            q.grad = (rv / 2 if ex else gv).double().clone().view_as(q)
        opt.step()
        adam.step(only_local=True, advance=False)
        assert int(arena.adam_t) == it
        adam.step(k=2, src="R", only_exchanged=True)
        assert int(arena.adam_t) == it + 1
    for q, p in zip(ref, arena.params):
        assert float((p.double() - q.detach()).abs().max()) < 1e-6, (p.shape, float((p.double() - q.detach()).abs().max()))


def test_flat_adam_checkpoint_roundtrip():
    """The arena's state dict carries both Adam moments and the step counter."""
    from theanompi_b200.parallel.arena import FlatArena
    from theanompi_b200.utils.opt import FlatAdam
    torch.manual_seed(3)
    a = FlatArena([torch.randn(40, 30), torch.randn(30)], device="cpu", optimizer="adam")
    adam = FlatAdam(a)
    a.hyper[0] = 1e-3
    for _ in range(3):
        a.G.normal_()
        adam.step()
    sd = a.state_dict()
    assert sd["t"] == 3 and torch.equal(sd["V"], a.V)
    b = FlatArena([torch.zeros(40, 30), torch.zeros(30)], device="cpu", optimizer="adam")
    b.load_state_dict(sd)
    assert torch.equal(b.W, a.W) and torch.equal(b.U, a.U) and torch.equal(b.V, a.V) and int(b.adam_t) == 3


def test_sgd_arena_layout_unchanged_and_fused_rs_rejects_adam():
    from theanompi_b200.parallel.arena import FlatArena
    from theanompi_b200.parallel.exchanger import BSP_Exchanger

    def arena(opt):
        return FlatArena([torch.randn(40, 30), torch.randn(30)], device="cpu", with_recv=True, shadow=True, optimizer=opt)
    sgd, adam = arena("msgd"), arena("adam")
    assert sgd.V is None and sgd.adam_t is None and "V" not in sgd.layout
    assert sgd.layout == {"W": 0, "G": sgd.numel * 4, "U": 2 * sgd.numel * 4, "R": 3 * sgd.numel * 4, "H": 4 * sgd.numel * 4}
    assert sgd.nbytes == 4 * sgd.numel * 4 + sgd.numel * 2
    assert {k: v for k, v in adam.layout.items() if k != "V"} == sgd.layout and adam.nbytes == sgd.nbytes + adam.numel * 4

    class _Comm(object):
        size, rank = 2, 0

    class _Model(object):
        optimizer = "adam"
        arena = adam
    try:
        BSP_Exchanger(_Comm(), object(), "fused_rs", "cdd", None, _Model())
    except ValueError as e:
        assert "Adam" in str(e)
    else:
        raise AssertionError("fused_rs must reject Adam")
