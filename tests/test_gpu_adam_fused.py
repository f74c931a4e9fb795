"""Data-parallel Adam on the GPU: the native adam_flat kernel's split form (group filter, inv_k, source R), the fused
all-reduce + Adam exchange kernels (multi-GPU) and native Wide_ResNet trained with BSP cdd through the Rule API."""
import json
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = "cuda:0"


def _torchrun(n, port, *args, timeout=600):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(n), "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "tests", "mp_adam_check.py")] + list(args)
    return subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=timeout, cwd=ROOT)


def test_adam_flat_split_matches_fp64():
    """The classic cdd split on the native kernel: BN groups on G without advancing t, then the exchanged groups on R with
    inv_k = 1/2 == fp64 Adam on the averaged gradient (exchanged) / the local gradient (BN)."""
    from theanompi_b200.parallel.arena import FlatArena
    from theanompi_b200.utils.opt import FlatAdam
    torch.manual_seed(5)
    shapes = [(300, 70), (300,), (64,), (64,), (64, 3, 3, 16)]
    names = [None, None, "gamma", "beta", None]
    params = []
    for s, n in zip(shapes, names):
        p = torch.randn(s) * 0.1
        p.pname = n
        params.append(p)
    arena = FlatArena(params, ["W", "b", "b", "b", "W"], torch.device(DEV), weight_decay=5e-4, with_recv=True, optimizer="adam")
    adam = FlatAdam(arena)
    lr, b1, b2, eps = 1e-2, adam.b1, adam.b2, adam.eps
    arena.hyper[0] = lr
    ex = arena.exch_vector()
    lrm, wd = arena.lr_mult_vector().double(), arena.wd_vector().double()
    w, m, v = arena.W.double(), torch.zeros(arena.numel, dtype=torch.float64, device=DEV), torch.zeros(arena.numel, dtype=torch.float64,
                                                                                                      device=DEV)
    for t in range(1, 5):
        g, r = torch.randn(arena.numel, device=DEV), torch.randn(arena.numel, device=DEV) * 2
        arena.G.copy_(g); arena.R.copy_(r)
        ge = torch.where(ex, r.double() / 2, g.double()) + wd * w
        m = b1 * m + (1 - b1) * ge
        v = b2 * v + (1 - b2) * ge * ge
        w = w - lr * lrm * (m / (1 - b1 ** t)) / ((v / (1 - b2 ** t)).sqrt() + eps)
        adam.step(only_local=True, advance=False)
        adam.step(k=2, src="R", only_exchanged=True)
    torch.cuda.synchronize()
    assert int(arena.adam_t) == 4
    real = torch.zeros(arena.numel, dtype=torch.bool, device=DEV)
    for o, s in zip(arena.offsets, arena.sizes):
        real[o:o + s] = True
    assert float((arena.W.double() - w)[real].abs().max()) < 2e-5
    assert float((arena.U.double() - m)[real].abs().max()) < 1e-5
    assert float((arena.H.float() - arena.W)[real].abs().max()) < 1e-2


@pytest.mark.multigpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_fused_adam_kernels_two_ranks():
    """Every algorithm x wire16 x push_master against fp64, the CUDA-graph replay of a 2-bucket step, checkpoint / resume."""
    r = _torchrun(2, 29781, "kernels")
    assert r.returncode == 0 and "MP_ADAM_CHECK_OK" in r.stdout, r.stdout[-4000:]


def _run_rule(strategy, monkeypatch, timeout=400):
    import theanompi_b200 as tm
    monkeypatch.setattr(tm.BSP, "sync_type", "cdd")
    monkeypatch.setattr(tm.BSP, "exch_strategy", strategy)
    rule = tm.BSP()
    rule.model_config = dict(batch_size=32, file_batch_size=32, n_epochs=1, learning_rate=1e-3, max_batches=6, printFreq=4, depth=10,
                             widen=2, data_kwargs=dict(n_synthetic=512, synthetic=True))
    rule.init(devices=["cuda0", "cuda1"], modelfile="theanompi_b200.models.keras_model_zoo.wresnet", modelclass="Wide_ResNet")
    try:
        return rule.proc.wait(timeout=timeout)
    except subprocess.TimeoutExpired:
        rule.proc.kill()
        raise


@pytest.mark.multigpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
@pytest.mark.parametrize("strategy", ["fused", "fused16", "nccl32"])
def test_rule_bsp_cdd_wide_resnet(tmp_path, monkeypatch, strategy):
    monkeypatch.chdir(tmp_path)
    assert _run_rule(strategy, monkeypatch) == 0
    assert os.path.exists(tmp_path / "snapshots" / "ckpt_0.pt")
    sd = torch.load(str(tmp_path / "snapshots" / "ckpt_0.pt"), map_location="cpu", weights_only=False)
    assert sd["arena"]["t"] == 6 and "V" in sd["arena"]


@pytest.mark.multigpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_fused_adam_follows_classic_trajectory():
    """Training-loss curves of native Wide_ResNet under the fused exchange and under the classic NCCL strategy (the Adam
    update runs after the all-reduce) coincide: same data, same init, same algorithm."""
    steps = 60
    curves = {}
    for k, strat in enumerate(("nccl32", "fused")):
        r = _torchrun(2, 29782 + k, "wrn", strat, str(steps))
        line = [l for l in r.stdout.splitlines() if l.startswith("MP_ADAM_WRN ")]
        assert r.returncode == 0 and line, r.stdout[-4000:]
        out = json.loads(line[-1][len("MP_ADAM_WRN "):])
        assert out["t"] == steps
        curves[strat] = out["losses"]
    w = 10

    def smooth(c):
        return [sum(c[i:i + w]) / w for i in range(0, len(c) - w + 1, w)]
    a, b = smooth(curves["nccl32"]), smooth(curves["fused"])
    for x, y in zip(a, b):
        assert abs(x - y) < 0.08 + 0.1 * x, curves
    assert a[-1] < a[0], curves                                    # and it learns
