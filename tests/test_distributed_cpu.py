"""world_size > 1 plumbing on CPU (gloo): strategies, mailbox control plane, BSP
equivalences, and the three rules end to end through the public Rule API."""
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_PORT = [29700]


def run_ranks(n, case, *args, timeout=240):
    _PORT[0] += 1
    procs = []
    for r in range(n):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE=str(n), LOCAL_RANK=str(r), MASTER_ADDR="127.0.0.1",
                   MASTER_PORT=str(_PORT[0]), OMP_NUM_THREADS="2", PYTHONPATH=ROOT)
        procs.append(subprocess.Popen([sys.executable, os.path.join(ROOT, "tests", "mp_cpu_checks.py"), case] + list(args), env=env,
                                      stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
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


def test_exchanger_strategies_world2():
    """BASELINE config #1: BSP allreduce correctness, world_size=2, CPU/gloo."""
    run_ranks(2, "strategies")


def test_mailbox_control_plane_world3():
    run_ranks(3, "mailbox")


def test_bsp_cdd_two_ranks_equals_one_big_batch(tmp_path):
    run_ranks(2, "bsp_equivalence", str(tmp_path))
    # single process, batch 32 = the two shards of each step concatenated
    from theanompi_b200.models import layers2
    from theanompi_b200.models.cifar10 import Cifar10_model
    from theanompi_b200.models.layers2 import Crop, Dropout
    from theanompi_b200.utils.recorder import Recorder
    layers2.reseed()
    m = Cifar10_model(dict(verbose=False, rank=0, size=1, device="cpu", batch_size=16, file_batch_size=16, learning_rate=0.02,
                           data_kwargs=dict(n_synthetic=640, synthetic=True)))
    Dropout.SetDropoutOff(); Crop.SetRandCropOff()
    m.compile_iter_fns("avg")
    d = m.data
    # emulate what ranks 0 and 1 saw: shards [0::2] and [1::2] of the commonly shuffled list
    rec = Recorder(None, 1000, "t", False, device="cpu")
    import numpy as np
    for step in range(6):
        if step == 0:
            d.shuffle_data("train", common_seed=m.epoch)
        xs = [d.train_img_shuffle[2 * step + r] for r in range(2)]
        ys = [d.train_labels_shuffle[2 * step + r] for r in range(2)]
        gsum = None
        for x, y in zip(xs, ys):
            m.x_in.copy_(torch.from_numpy(np.ascontiguousarray(x)))
            m.y_in.copy_(torch.from_numpy(np.asarray(y)))
            c, e = m._fwd_bwd_eager()
            gsum = m.arena.G.clone() if gsum is None else gsum + m.arena.G
        m.arena.G.copy_(gsum)
        m.sgd.step(m.shared_lr.get_value(), k=2)
    Dropout.SetDropoutOn(); Crop.SetRandCropOn()
    for strat in ("ar", "nccl32", "asa32"):
        w2 = torch.load(str(tmp_path / ("bsp_%s.pt" % strat)))
        err = float((w2 - m.arena.W).abs().max())
        assert err < 2e-5, (strat, err)


def test_bsp_avg_two_ranks():
    run_ranks(2, "bsp_avg")


def _run_rule(rule_cls, devices, extra_env=None, cfg=None, timeout=300):
    import theanompi_b200 as tm
    rule = rule_cls()
    rule.model_config = dict(batch_size=16, file_batch_size=16, n_epochs=1, learning_rate=0.01, max_batches=6,
                             printFreq=4, data_kwargs=dict(n_synthetic=320, synthetic=True))
    if cfg:
        rule.model_config.update(cfg)
    rule.env.update(extra_env or {})
    rule.env["OMP_NUM_THREADS"] = "2"
    rule.init(devices=devices, modelfile="theanompi_b200.models.cifar10", modelclass="Cifar10_model")
    try:
        rc = rule.proc.wait(timeout=timeout)
    except subprocess.TimeoutExpired:
        rule.proc.kill()
        raise
    return rc


def test_rule_bsp_cpu(tmp_path, monkeypatch):
    import theanompi_b200 as tm
    monkeypatch.chdir(tmp_path)
    tm.BSP.sync_type, tm.BSP.exch_strategy = "cdd", "ar"
    assert _run_rule(tm.BSP, ["cpu0", "cpu1"]) == 0
    assert os.path.exists(tmp_path / "inforec" / "inforec.pkl")
    assert os.path.exists(tmp_path / "snapshots" / "ckpt_0.pt")


def test_rule_easgd_cpu(tmp_path, monkeypatch):
    import theanompi_b200 as tm
    monkeypatch.chdir(tmp_path)
    assert _run_rule(tm.EASGD, ["cpu0", "cpu1", "cpu2"], extra_env={"TMPI_EASGD_TAU": "2"}) == 0


def test_rule_asgd_cpu(tmp_path, monkeypatch):
    """ASGD (delta-push exchanger behind the EASGD runtime) incl. validation / stop, which both copy the center to the worker."""
    import theanompi_b200 as tm
    monkeypatch.chdir(tmp_path)
    assert _run_rule(tm.ASGD, ["cpu0", "cpu1", "cpu2"], extra_env={"TMPI_EASGD_TAU": "2"}) == 0


def test_rule_gosgd_cpu(tmp_path, monkeypatch):
    import theanompi_b200 as tm
    monkeypatch.chdir(tmp_path)
    assert _run_rule(tm.GOSGD, ["cpu0", "cpu1", "cpu2"], cfg=dict(gosgd_p=0.5)) == 0


def test_failfast_teardown(tmp_path, monkeypatch):
    """A worker that dies takes the whole job down (parity with MPI abort semantics)."""
    import theanompi_b200 as tm
    monkeypatch.chdir(tmp_path)
    tm.BSP.sync_type, tm.BSP.exch_strategy = "cdd", "ar"
    rule = tm.BSP()
    rule.init(devices=["cpu0", "cpu1"], modelfile="theanompi_b200.models.cifar10", modelclass="NoSuchModel")
    rc = rule.proc.wait(timeout=120)
    assert rc != 0


def test_rule_bsp_two_hosts_through_remote_shell(tmp_path, monkeypatch):
    """The multi-host path (``host:device`` entries → one remote shell per worker, per-host LOCAL_RANK, rendezvous on the first
    host, NCCL/gloo strategy instead of the peer-memory one): two "hosts" that both resolve to this machine, reached through a
    local stand-in for ssh — the reference's ``mpirun -host`` MPMD launch (``rules.py:85-116``)."""
    import stat
    import theanompi_b200 as tm
    monkeypatch.chdir(tmp_path)
    shim = tmp_path / "fake_ssh"
    log = tmp_path / "ssh_calls.log"
    shim.write_text("#!/bin/sh\n# usage: fake_ssh HOST 'command line'\necho \"$1\" >> %s\nshift\nexec sh -c \"$*\"\n" % log)
    shim.chmod(shim.stat().st_mode | stat.S_IXUSR)
    monkeypatch.setenv("TMPI_SSH", str(shim))
    monkeypatch.setenv("TMPI_MASTER_ADDR", "127.0.0.1")
    tm.BSP.sync_type, tm.BSP.exch_strategy = "cdd", "fused"          # must fall back to a network strategy on its own
    try:
        assert _run_rule(tm.BSP, ["nodeA:cpu0", "nodeB:cpu0"]) == 0
    finally:
        tm.BSP.exch_strategy = "fused"
    assert sorted(log.read_text().split()) == ["nodeA", "nodeB"]
    assert os.path.exists(tmp_path / "inforec" / "inforec.pkl")
