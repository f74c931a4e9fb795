"""Wide-ResNet WRN-28-4 on CIFAR-10 with Adam (ref ``keras_model_zoo/wresnet.py:37-82,159``):
pre-activation blocks, widths (16, 64, 128, 256), 4 blocks per group; params = all trainable
weights (``:257-263``).  The model of the GOSGD benchmark config (BASELINE.json).  The reference
only averages weights (``sync_type='avg'``, ``:152-153``); here ``'cdd'`` also works: gradients are
averaged across ranks, then one Adam step (inside the fused exchange kernels, or after a classic
strategy's all-reduce).

``Wide_ResNet`` runs on the hand-written sm_100a kernels (tcgen05 implicit-GEMM convolutions, fused BatchNormal+ReLU, native
residual add, one flat Adam kernel; CUDA-graph captured step).  ``Wide_ResNetTorch`` is the same network on torch modules
with ``torch.optim.Adam`` — the library yardstick and the numerical reference of the tests."""
from __future__ import annotations

import torch
import torch.nn as nn

from ..base import ModelBase
from ..layers2 import BatchNormal, Constant, Conv, Flatten, HeNormal, Normal, Pool, Softmax, get_params
from ..torch_base import TorchModelBase

n_epochs = 200
batch_size = 128
file_batch_size = 128
learning_rate = 1e-3
depth, widen = 28, 4


class PreActBlock(nn.Module):
    def __init__(self, cin, cout, stride):
        super().__init__()
        self.bn1, self.c1 = nn.BatchNorm2d(cin), nn.Conv2d(cin, cout, 3, stride, 1, bias=False)
        self.bn2, self.c2 = nn.BatchNorm2d(cout), nn.Conv2d(cout, cout, 3, 1, 1, bias=False)
        self.short = None if (stride == 1 and cin == cout) else nn.Conv2d(cin, cout, 1, stride, bias=False)

    def forward(self, x):
        o = torch.relu(self.bn1(x))
        s = x if self.short is None else self.short(o)
        o = self.c1(o)
        o = self.c2(torch.relu(self.bn2(o)))
        return o + s


class WRN(nn.Module):
    def __init__(self, depth=28, k=4, n_class=10):
        super().__init__()
        n = (depth - 4) // 6
        w = [16, 16 * k, 32 * k, 64 * k]
        layers = [nn.Conv2d(3, w[0], 3, 1, 1, bias=False)]
        cin = w[0]
        for g, (cout, stride) in enumerate(zip(w[1:], (1, 2, 2))):
            for j in range(n):
                layers.append(PreActBlock(cin, cout, stride if j == 0 else 1))
                cin = cout
        self.body = nn.Sequential(*layers)
        self.bn = nn.BatchNorm2d(cin)
        self.fc = nn.Linear(cin, n_class)

    def forward(self, x):
        return self.fc(torch.relu(self.bn(self.body(x))).mean((2, 3)))


class Wide_ResNet(ModelBase):
    n_epochs, batch_size, file_batch_size, learning_rate = n_epochs, batch_size, file_batch_size, learning_rate
    weight_decay, momentum = 0.0, 0.9
    optimizer = "adam"             # config['optimizer'] = 'sgd' / 'msgd' trains with momentum SGD instead
    bias_lr_mult = 1.0             # Adam: one learning rate for every parameter
    lr_policy = "step"
    lr_step = [60, 120, 160]
    lr_gamma = 0.2
    input_width = input_height = 32

    def __init__(self, config):
        super().__init__(config)
        self.name = "Wide_ResNet"
        for k in ("batch_size", "file_batch_size", "n_epochs", "learning_rate"):
            if k in config:
                setattr(self, k, config[k])
        self.base_lr = self.learning_rate
        from ..data.cifar10 import Cifar10_data
        from .. import layers2
        self.data = Cifar10_data(verbose=False, **config.get("data_kwargs", {}))
        self.channels = 3
        self.n_softmax_out = self.data.n_class
        self.setup_data_parallel(self.data)
        self._mean = torch.as_tensor(self.data.rawdata[4]).to(self.device)
        layers2.reseed()
        self.depth, self.widen = config.get("depth", depth), config.get("widen", widen)
        self.build_model()
        params, weight_types = get_params(self.layers)
        self.finalize(params, weight_types, (self.batch_size, 32, 32, 3))
        self.shared_lr.set_value(self.learning_rate)

    def _conv(self, inp, cout, k, stride, pad, input_shape=None):
        cin = (inp.output_shape if inp is not None else input_shape)[-1]
        c = Conv(inp, stride, pad, W=HeNormal((cout, k, k, cin)), b=False, relu=False, printinfo=False, input_shape=input_shape)
        self.layers.append(c)
        return c

    def _bn(self, inp):
        b = BatchNormal(inp, relu=True, printinfo=False)
        self.layers.append(b)
        return b

    def build_model(self):
        n = (self.depth - 4) // 6
        w = [16, 16 * self.widen, 32 * self.widen, 64 * self.widen]
        self.layers = []
        self.stem = self._conv(None, w[0], 3, 1, 1, input_shape=(self.batch_size, 32, 32, 3))
        cur = self.stem
        self.body = []
        for cout, stride0 in zip(w[1:], (1, 2, 2)):
            for j in range(n):
                stride = stride0 if j == 0 else 1
                cin = cur.output_shape[-1]
                bn1 = self._bn(cur)
                short = self._conv(bn1, cout, 1, stride, 0) if (stride != 1 or cin != cout) else None
                c1 = self._conv(bn1, cout, 3, stride, 1)
                bn2 = self._bn(c1)
                c2 = self._conv(bn2, cout, 3, 1, 1)
                self.body.append((bn1, short, c1, bn2, c2))
                cur = c2
        bn = self._bn(cur)
        gap = Pool(bn, bn.output_shape[1], 1, 0, "avg", printinfo=False)
        flat = Flatten(gap, axis=2, printinfo=False)
        sm = Softmax(flat, self.n_softmax_out, W=Normal((self.n_softmax_out, flat.output_shape[1]), std=0.05),
                     b=Constant((self.n_softmax_out,), 0.0), printinfo=False)
        self.layers += [gap, flat, sm]
        self.head = (bn, gap, flat, sm)
        self.output_layer = sm

    def forward(self, x):
        from ... import ops
        if x.is_cuda:
            # (x − mean) / 64 → activation dtype in ONE native kernel (the loader's normalise kernel with a full-image crop)
            if getattr(self, "_zero_off", None) is None or self._zero_off.shape[0] != x.shape[0]:
                self._zero_off = torch.zeros((x.shape[0], 2), dtype=torch.int32, device=x.device)
                self._zero_flip = torch.zeros((x.shape[0],), dtype=torch.uint8, device=x.device)
            x = ops.crop_mirror_normalize(x.float() if x.dtype not in (torch.float32, torch.bfloat16, torch.uint8) else x, self._mean,
                                          1.0 / 64.0, (x.shape[1], x.shape[2]), self._zero_off, self._zero_flip, out_dtype=self.act_dtype)
        else:
            x = ((x.float() - self._mean) / 64.0).to(self.act_dtype)
        x = self.stem.forward(x)
        for bn1, short, c1, bn2, c2 in self.body:                 # pre-activation block (ref :37-82)
            if short is None:
                x, s = ops.fork2(x)                               # identity shortcut: x feeds bn1 and the merge
                o = bn1.forward(x)
            else:
                o, o2 = ops.fork2(bn1.forward(x))                 # projection shortcut reads the pre-activated tensor
                s = short.forward(o2)
            o = c2.forward(bn2.forward(c1.forward(o)))
            x = ops.add(o, s)
        bn, gap, flat, sm = self.head
        return sm.forward(flat.forward(gap.forward(bn.forward(x))))

    def load_extra_state(self, sd):
        super().load_extra_state(sd)
        if "adam" in sd and self.adam is not None:      # checkpoints written before the moments moved into the arena
            self.adam.load_state_dict(sd["adam"])


class Wide_ResNetTorch(TorchModelBase):
    n_epochs, batch_size, file_batch_size, learning_rate = n_epochs, batch_size, file_batch_size, learning_rate
    weight_decay, momentum = 0.0, 0.9
    lr_policy = "step"
    lr_step = [60, 120, 160]
    lr_gamma = 0.2
    input_width = input_height = 32

    def __init__(self, config):
        super().__init__(config)
        self.name = "Wide_ResNetTorch"
        for k in ("batch_size", "file_batch_size", "n_epochs", "learning_rate"):
            if k in config:
                setattr(self, k, config[k])
        self.base_lr = self.learning_rate
        torch.manual_seed(23455)
        from ..data.cifar10 import Cifar10_data
        self.data = Cifar10_data(verbose=False, **config.get("data_kwargs", {}))
        self.channels = 3
        self.setup_data_parallel(self.data)
        self._mean = torch.as_tensor(self.data.rawdata[4]).to(self.device)
        net = WRN(config.get("depth", depth), config.get("widen", widen), self.data.n_class)
        self.finalize_torch(net, (self.batch_size, 32, 32, 3))

    def forward(self, x):
        x = (x.float() - self._mean) / 64.0
        return super().forward(x.to(self.act_dtype))

    def make_torch_optimizer(self, params):
        if self.config.get("optimizer", "adam") == "sgd":
            return None
        return torch.optim.Adam(params, lr=self.learning_rate)
