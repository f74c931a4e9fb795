"""Every zoo model trains a few steps on the GPU path (native kernels / torch adapter) — smoke + sanity."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu


def _run(modelfile, modelclass, cfg, steps=3, sync="avg"):
    import importlib
    from theanompi_b200.models import layers2
    from theanompi_b200.utils.recorder import Recorder
    layers2.reseed(); layers2.Dropout.layers.clear(); layers2.Crop.layers.clear()
    base = dict(verbose=False, rank=0, size=1, device="cuda:0")
    base.update(cfg)
    m = getattr(importlib.import_module(modelfile), modelclass)(base)
    m.compile_iter_fns(sync)
    rec = Recorder(None, 10 ** 6, modelclass, False, device="cuda:0")
    w0 = m.arena.W.clone()
    c = 0
    for i in range(steps):
        out = m.train_iter(c, rec)
        c = out if isinstance(out, int) else c + 1
    m.val_iter(c, rec)
    torch.cuda.synchronize()
    loss = float(rec.train_info["cost"][-1])
    assert math.isfinite(loss), loss
    assert not torch.equal(w0, m.arena.W), "weights did not move"
    m.cleanup()
    return loss, m


IMNET = dict(n_class=16, data_kwargs=dict(n_train_files=4, n_val_files=1, synthetic=True))


def test_alexnet_graph_and_eager_agree():
    from theanompi_b200.ops import cuda_impl
    losses = []
    for graph in (False, True):
        cuda_impl._STEP.clear()
        l, m = _run("theanompi_b200.models.alex_net", "AlexNet", dict(batch_size=32, file_batch_size=32, cuda_graph=graph, **IMNET), steps=5)
        losses.append(l)
    assert abs(losses[0] - losses[1]) < 0.15, losses


def test_googlenet():
    _run("theanompi_b200.models.googlenet", "GoogLeNet", dict(batch_size=8, file_batch_size=16, **IMNET), steps=3)


def test_vgg16():
    _run("theanompi_b200.models.lasagne_model_zoo.vgg16", "VGG16", dict(batch_size=4, file_batch_size=8, **IMNET), steps=2)


def test_cifar10_model_learns():
    from theanompi_b200.models.cifar10 import Cifar10_model  # noqa: F401
    l, m = _run("theanompi_b200.models.cifar10", "Cifar10_model",
                dict(batch_size=64, file_batch_size=64, learning_rate=0.001, data_kwargs=dict(n_synthetic=1024, synthetic=True)), steps=40)
    assert l < 1.5, l                                   # synthetic classes are separable: loss must fall well below ln(10)


def test_resnet50_cdd_flat_sgd():
    _run("theanompi_b200.models.lasagne_model_zoo.resnet50", "ResNet50",
         dict(batch_size=4, file_batch_size=4, blocks=(1, 1, 1, 1), no_paraload=True, **IMNET), steps=2, sync="cdd")


def test_torch_adapter_models_still_run():
    """The torch-module variants (cuDNN / cuBLAS through TorchModelBase) stay available as library yardsticks."""
    _run("theanompi_b200.models.lasagne_model_zoo.resnet50", "ResNet50Torch",
         dict(batch_size=4, file_batch_size=4, blocks=(1, 1, 1, 1), no_paraload=True, **IMNET), steps=2, sync="cdd")
    _run("theanompi_b200.models.keras_model_zoo.wresnet", "Wide_ResNetTorch",
         dict(batch_size=16, file_batch_size=16, depth=10, widen=2, data_kwargs=dict(n_synthetic=128, synthetic=True)), steps=2)


@pytest.mark.parametrize("which", ["resnet", "wrn"])
def test_native_residual_nets_match_fp32_reference(which):
    """Native ResNet / Wide-ResNet (tcgen05 convs + fused BatchNormal kernels) vs the SAME model on the plain-torch fp32
    reference ops (CPU), same weights, same batch: loss of the first steps within bf16 accuracy, no library kernels launched."""
    import importlib
    from theanompi_b200.models import layers2
    from theanompi_b200.ops import native
    from theanompi_b200.utils.recorder import Recorder
    if which == "resnet":
        mod, cls = "theanompi_b200.models.lasagne_model_zoo.resnet50", "ResNet50"
        cfg = dict(batch_size=8, file_batch_size=8, blocks=(1, 1, 1, 1), no_paraload=True, n_class=16,
                   data_kwargs=dict(n_train_files=4, n_val_files=1, synthetic=True))
    else:
        mod, cls = "theanompi_b200.models.keras_model_zoo.wresnet", "Wide_ResNet"
        cfg = dict(batch_size=32, file_batch_size=32, depth=10, widen=2, data_kwargs=dict(n_synthetic=256, synthetic=True))
    losses = {}
    for dev in ("cpu", "cuda:0"):
        layers2.reseed(); layers2.Dropout.layers.clear(); layers2.Crop.layers.clear(); layers2.BatchNormal.layers.clear()
        m = getattr(importlib.import_module(mod), cls)(dict(verbose=False, rank=0, size=1, device=dev, cuda_graph=False, **cfg))
        m.rand_crop = False
        m.compile_iter_fns("avg")
        rec = Recorder(None, 10 ** 6, cls, False, device=dev)
        native.reset_launch_count()
        for i in range(3):
            m.train_iter(i, rec)
        losses[dev] = [float(c) for c in rec.train_info["cost"]]
        if dev != "cpu":
            torch.cuda.synchronize()
            assert native.launch_count() > 50
        m.cleanup()
    for a, b in zip(losses["cpu"], losses["cuda:0"]):
        assert abs(a - b) < 0.08 * max(1.0, abs(a)), losses


def test_wide_resnet_adam():
    _run("theanompi_b200.models.keras_model_zoo.wresnet", "Wide_ResNet",
         dict(batch_size=16, file_batch_size=16, depth=10, widen=2, data_kwargs=dict(n_synthetic=128, synthetic=True)), steps=3)


def test_gans_and_lstm():
    _run("theanompi_b200.models.lasagne_model_zoo.wgan", "WGAN", dict(critic_runs=2, data_kwargs=dict(n_synthetic=256)), steps=2)
    _run("theanompi_b200.models.lasagne_model_zoo.lsgan", "LSGAN", dict(data_kwargs=dict(n_synthetic=256)), steps=2)
    _run("theanompi_b200.models.lasagne_model_zoo.lsgan_cifar10", "LSGAN", dict(data_kwargs=dict(n_synthetic=256, synthetic=True)), steps=2)
    _run("theanompi_b200.models.lstm", "LSTM", dict(dim_proj=64, data_kwargs=dict(n_synthetic=128, n_words=500)), steps=3)
    _run("theanompi_b200.models.lstm", "LSTMTorch", dict(dim_proj=32, data_kwargs=dict(n_synthetic=128, n_words=500)), steps=3)


def test_loader_pipeline_matches_reference_crop():
    """GPU loader: pinned H2D + fused crop kernel == host reference of the same file."""
    import numpy as np
    from theanompi_b200.models.data.imagenet import ImageNet_data
    d = ImageNet_data(synthetic=True, n_train_files=3, n_val_files=1, file_batch_size=8, size_hw=64)
    d.batch_data(8)
    ld = d.para_load_init("cuda:0", 48, 48, rand_crop=False, batch_crop_mirror=False)
    ld.request(d.train_img[0], "val"); ld.request(d.train_img[1], "val")
    b = ld.get()
    torch.cuda.synchronize()
    raw = d.read(d.train_img[0], np.empty((8, 64, 64, 3), np.uint8)).numpy()
    want = ((raw.astype(np.float32) - 127.5) / 255.0 / np.array([0.229, 0.224, 0.225], np.float32))[:, 8:56, 8:56, :]
    assert np.abs(b.x.float().cpu().numpy() - want).max() < 1.2e-2     # bf16 ulp at |x| ~ 2.2
    ld.drain(); d.para_load_close()


def test_loader_process_mode_gpu(tmp_path, monkeypatch):
    """Loader process → page-locked shared-memory ring → H2D on the copy stream → fused crop kernel, with real batch files."""
    import numpy as np
    from theanompi_b200.models.data.loader import ParaLoader
    from theanompi_b200.models.data.proc_loader import ProcReader
    arrs = []
    for i in range(4):
        a = np.random.RandomState(i).randint(0, 256, (8, 64, 64, 3), dtype=np.uint8)
        np.save(str(tmp_path / ("b%d.npy" % i)), a)
        arrs.append(a)
    pr = ProcReader((8, 64, 64, 3), depth=2)
    assert all(t.is_pinned() for t in pr.tensors)
    ld = ParaLoader(pr.read, "cuda:0", (8, 64, 64, 3), (48, 48), mean=np.full((64, 64, 3), 127.5, np.float32), std_scale=1 / 255.0,
                    depth=2, rand_crop=False, host_buffers=pr.tensors, on_close=pr.close)
    try:
        ld.request(str(tmp_path / "b0.npy"), "val")
        for i in range(4):
            if i + 1 < 4:
                ld.request(str(tmp_path / ("b%d.npy" % (i + 1))), "val")
            b = ld.get()
            torch.cuda.synchronize()
            want = ((arrs[i].astype(np.float32) - 127.5) / 255.0)[:, 8:56, 8:56, :]
            assert np.abs(b.x.float().cpu().numpy() - want).max() < 4e-3, i
    finally:
        ld.close()


def test_deterministic_mode_is_bit_reproducible(tmp_path):
    """TMPI_DETERMINISTIC=1 (no split-K: every gradient element is produced by one CTA in a fixed k order) → two runs of the same
    training steps give bit-identical weights; the default (split-K with fp32 atomics in arrival order) is only close."""
    import os
    import subprocess
    import sys
    code = (
        "import torch, sys\n"
        "from theanompi_b200.models import layers2\n"
        "from theanompi_b200.models.cifar10 import Cifar10_model\n"
        "from theanompi_b200.utils.recorder import Recorder\n"
        "m = Cifar10_model(dict(verbose=False, rank=0, size=1, device='cuda:0', batch_size=64, file_batch_size=64, cuda_graph=False,\n"
        "                       data_kwargs=dict(n_synthetic=512, synthetic=True)))\n"
        "layers2.Dropout.SetDropoutOff(); layers2.Crop.SetRandCropOff()\n"
        "m.compile_iter_fns('avg'); rec = Recorder(None, 10**6, 'c', False, device='cuda:0')\n"
        "for i in range(4): m.train_iter(i, rec)\n"
        "torch.cuda.synchronize(); torch.save(m.arena.W.cpu(), sys.argv[1])\n")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    outs = []
    for k in range(2):
        f = str(tmp_path / ("w%d.pt" % k))
        env = dict(os.environ, TMPI_DETERMINISTIC="1", PYTHONPATH=root)
        r = subprocess.run([sys.executable, "-c", code, f], env=env, cwd=root, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=300)
        assert r.returncode == 0, r.stdout[-2000:]
        outs.append(torch.load(f))
    assert torch.equal(outs[0], outs[1])


def test_label_staging_survives_a_host_that_runs_ahead():
    """The host enqueues whole steps ahead of the device (always under CUDA graphs, and whenever a step is GPU-bound): the
    pinned label staging must not be overwritten with the next batch before the copy of the current one has executed —
    otherwise images and labels of consecutive steps get mixed (the 2-GPU trajectory regression this guards against)."""
    import numpy as np
    from theanompi_b200.models.cifar10 import Cifar10_model
    m = Cifar10_model(dict(verbose=False, rank=0, size=1, device="cuda:0", batch_size=64, file_batch_size=64, cuda_graph=False,
                           data_kwargs=dict(n_synthetic=256, synthetic=True)))
    B = int(m.shared_y.shape[0])
    torch.cuda.synchronize()
    torch.cuda._sleep(int(4e8))                       # the device is ~0.2 s behind the host from here on
    got = []
    for i in range(9):
        m._labels_to_device(np.full(B, i, dtype=np.int64))
        got.append(m.shared_y.clone())               # stream-ordered: sees what the i-th H2D copy delivered
    torch.cuda.synchronize()
    for i, g in enumerate(got):
        assert bool((g == i).all()), (i, g[:4].tolist())
