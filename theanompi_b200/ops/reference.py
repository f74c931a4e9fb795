"""Plain-PyTorch reference implementations of every op in :mod:`theanompi_b200.ops`.

These are (a) the CPU execution path (tests, gloo plumbing runs) and (b) the
fp32 ground truth every hand-written sm_100a kernel is tested against.

Layout convention for the whole framework: activations are **NHWC**
``[N, H, W, C]`` contiguous, conv filters are **OHWI** ``[O, kh, kw, C/groups]``,
FC weights are ``[n_out, n_in]`` (K-major for the tcgen05 GEMM).  The reference
used c01b / bc01 (``theanompi/models/layers2.py:430-560``).
"""
from __future__ import annotations

import torch
import torch.nn.functional as F


def _nchw(x):
    return x.permute(0, 3, 1, 2)


def _nhwc(x):
    return x.permute(0, 2, 3, 1).contiguous()


# --------------------------------------------------------------------------- conv
def conv2d_bias_act(x, w, b, stride=1, pad=0, groups=1, relu=True):
    """conv + bias + ReLU (ref ``layers2.py:380-388``)."""
    y = F.conv2d(_nchw(x), w.permute(0, 3, 1, 2), b, stride=stride, padding=pad, groups=groups)
    if relu:
        y = torch.relu(y)
    return _nhwc(y)


def conv2d_bias_act_bwd(x, w, y, dy, stride=1, pad=0, groups=1, relu=True, need_dx=True):
    """Returns (dx, dw, db) given the forward output ``y`` (for the ReLU mask)."""
    if relu:
        dy = dy * (y > 0).to(dy.dtype)
    xn, wn, dyn = _nchw(x), w.permute(0, 3, 1, 2), _nchw(dy)
    dx = None
    if need_dx:
        dx = torch.nn.grad.conv2d_input(xn.shape, wn, dyn, stride=stride, padding=pad, groups=groups)
        dx = _nhwc(dx)
    dw = torch.nn.grad.conv2d_weight(xn, wn.shape, dyn, stride=stride, padding=pad, groups=groups)
    dw = dw.permute(0, 2, 3, 1).contiguous()
    db = dy.sum(dim=(0, 1, 2))
    return dx, dw, db


# --------------------------------------------------------------------------- linear
def linear_bias_act(x, w, b, relu=True):
    """FC + bias + ReLU (ref ``layers2.py:927-929``); ``w`` is ``[n_out, n_in]``."""
    y = F.linear(x, w, b)
    return torch.relu(y) if relu else y


def linear_bias_act_bwd(x, w, y, dy, relu=True, need_dx=True):
    if relu:
        dy = dy * (y > 0).to(dy.dtype)
    dx = dy @ w if need_dx else None
    dw = dy.t() @ x
    db = dy.sum(0)
    return dx, dw, db


# --------------------------------------------------------------------------- pool
def pool2d(x, ksize, stride, pad=0, mode="max"):
    """max / average pooling (ref ``layers2.py:414-417``; cuDNN semantics: floor)."""
    xn = _nchw(x)
    if mode == "max":
        y = F.max_pool2d(xn, ksize, stride, pad)
    else:  # cuDNN 'average_exc_pad' is what theano's dnn_pool('average_exc_pad') used
        y = F.avg_pool2d(xn, ksize, stride, pad, count_include_pad=False)
    return _nhwc(y)


def pool2d_bwd(x, y, dy, ksize, stride, pad=0, mode="max"):
    xr = x.detach().clone().requires_grad_(True)
    with torch.enable_grad():
        yr = pool2d(xr, ksize, stride, pad, mode)
    (dx,) = torch.autograd.grad(yr, xr, dy)
    return dx


# --------------------------------------------------------------------------- LRN
def lrn(x, n=5, k=2.0, alpha=1e-4, beta=0.75):
    """Cross-channel LRN exactly as the reference writes it
    (``layers2.py:753-809``): ``x / (k + alpha * sum_{|j-i|<=n/2} x_j^2) ** beta``
    (alpha is NOT divided by n, unlike ``torch.nn.functional.local_response_norm``).
    Returns (y, scale)."""
    half = n // 2
    sq = x.float() ** 2
    C = x.shape[-1]
    padded = F.pad(sq, (half, half))
    s = torch.zeros_like(sq)
    for i in range(n):
        s = s + padded[..., i:i + C]
    scale = k + alpha * s
    y = x.float() * scale.pow(-beta)
    return y.to(x.dtype), scale


def lrn_bwd(x, dy, n=5, k=2.0, alpha=1e-4, beta=0.75):
    xr = x.detach().float().clone().requires_grad_(True)
    with torch.enable_grad():
        yr, _ = lrn(xr, n, k, alpha, beta)
    (dx,) = torch.autograd.grad(yr, xr, dy.float())
    return dx.to(x.dtype)


# --------------------------------------------------------------------------- dropout
def dropout_mask(shape, p_drop, seed, offset, device):
    """Deterministic keep-mask from (seed, offset) so CPU tests can reproduce it."""
    g = torch.Generator(device="cpu")
    g.manual_seed((int(seed) * 1000003 + int(offset)) & 0x7FFFFFFFFFFFFFFF)
    m = torch.rand(shape, generator=g) >= p_drop
    return m.to(device)


def dropout(x, p_drop, mask):
    """Inverted-scale-free dropout as in the reference (``layers2.py:885-891``):
    train: ``mask * x``; eval: ``(1-p) * x``."""
    return x * mask.to(x.dtype)


# --------------------------------------------------------------------------- softmax + NLL
def softmax_xent(logits, labels):
    """mean NLL, top-1 error, top-5 error, and d(mean NLL)/dlogits
    (ref ``layers2.py:952-997``)."""
    lg = logits.float()
    lsm = F.log_softmax(lg, dim=1)
    B = lg.shape[0]
    loss = -lsm[torch.arange(B, device=lg.device), labels].mean()
    pred = lg.argmax(1)
    err1 = (pred != labels).float().mean()
    k = min(5, lg.shape[1])
    topk = lg.topk(k, dim=1).indices
    err5 = 1.0 - (topk == labels[:, None]).any(1).float().mean()
    dlogits = lsm.exp()
    dlogits[torch.arange(B, device=lg.device), labels] -= 1.0
    dlogits = dlogits / B
    return loss, err1, err5, dlogits


# --------------------------------------------------------------------------- optimizer (flat arena)
def sgd_flat(w, g, u, lr_mult, wd, lr, mu, nesterov, inv_k, w_half=None):
    """One momentum-SGD step over flat fp32 buffers with per-element
    ``lr_mult`` / ``wd`` vectors (broadcastable).  Semantics of the reference's
    ``BSP_MSGD`` collapsed into one pass (``theanompi/lib/opt.py:181-268``):

        g_eff = g * inv_k + wd * w
        u     = mu * u + g_eff
        w    -= lr * lr_mult * (u            if not nesterov
                                g_eff + mu*u if nesterov)
    """
    g_eff = g * inv_k + wd * w
    u.mul_(mu).add_(g_eff)
    step = g_eff + mu * u if nesterov else u
    w.sub_(lr * lr_mult * step)
    if w_half is not None:
        w_half.copy_(w)
    return w, u


def adam_flat(w, g, m, v, lr_mult, wd, lr, b1, b2, eps, t, inv_k=1.0, w_half=None):
    """One Adam step (step number ``t`` >= 1) over flat fp32 buffers with per-element ``lr_mult`` / ``wd`` vectors, as the
    native ``adam_flat`` / fused Adam kernels compute it:

        ge = g * inv_k + wd * w
        m  = b1 * m + (1 - b1) * ge
        v  = b2 * v + (1 - b2) * ge^2
        w -= lr * lr_mult * (m / (1 - b1^t)) / (sqrt(v / (1 - b2^t)) + eps)
    """
    ge = g * inv_k + wd * w
    m.mul_(b1).add_(ge, alpha=1 - b1)
    v.mul_(b2).addcmul_(ge, ge, value=1 - b2)
    mh, vh = m / (1 - b1 ** t), v / (1 - b2 ** t)
    w.sub_(lr * lr_mult * mh / (vh.sqrt() + eps))
    if w_half is not None:
        w_half.copy_(w)
    return w, m, v


def easgd_elastic(w, c, alpha):
    """EASGD elastic move (ref ``exchanger.py:188-211``) with both sides updated
    from the SAME difference: ``d = alpha (w - c); w -= d; c += d``."""
    d = alpha * (w - c)
    w.sub_(d)
    c.add_(d)
    return w, c


def gosgd_merge(w, b, alpha_self, alpha_src):
    """GOSGD weighted merge (ref ``exchanger.py:450-462``)."""
    w.mul_(alpha_self).add_(b, alpha=alpha_src).div_(alpha_self + alpha_src)
    return w


# --------------------------------------------------------------------------- data aug
def crop_mirror_normalize(x_u8, mean, std_scale, crop_hw, offsets, flips, out_dtype=torch.float32):
    """``(x - mean) * std_scale`` → crop at per-image ``offsets`` → optional
    horizontal flip (ref ``data/utils.py:42-129`` + ``proc_load_mpi.py:99-104``).

    x_u8   : [N, H, W, C] uint8 or float
    mean   : [H, W, C] or [C] float
    offsets: [N, 2] int (y0, x0);  flips: [N] bool
    """
    N, H, W, C = x_u8.shape
    ch, cw = crop_hw
    if isinstance(std_scale, torch.Tensor):
        std_scale = std_scale.to(device=x_u8.device, dtype=torch.float32)
    x = (x_u8.float() - mean.float()) * std_scale
    out = torch.empty((N, ch, cw, C), dtype=torch.float32, device=x.device)
    for i in range(N):
        y0, x0 = int(offsets[i, 0]), int(offsets[i, 1])
        patch = x[i, y0:y0 + ch, x0:x0 + cw, :]
        if bool(flips[i]):
            patch = patch.flip(1)
        out[i] = patch
    return out.to(out_dtype)


# --------------------------------------------------------------------------- batch norm (+ residual)(+ ReLU), NHWC
def batch_norm_fwd(x, gamma, beta, run_mean, run_var, training, momentum, eps, relu, res=None):
    """y = γ·(x − mean)·rstd + β [+ res] [ReLU]; statistics over all but the last (channel) axis.  Updates the running
    statistics in place (momentum form, unbiased variance) when training.  Returns (y, mean, rstd)."""
    xf = x.float()
    C = x.shape[-1]
    x2 = xf.reshape(-1, C)
    R = x2.shape[0]
    if training:
        mean = x2.mean(0)
        var = (x2 * x2).mean(0) - mean * mean
        var = var.clamp_min(0)
        if run_mean is not None:
            with torch.no_grad():
                run_mean.mul_(1 - momentum).add_(momentum * mean)
                run_var.mul_(1 - momentum).add_(momentum * var * (R / max(1, R - 1)))
    else:
        mean, var = run_mean.float(), run_var.float()
    rstd = torch.rsqrt(var + eps)
    y = (xf - mean) * (rstd * gamma.float()) + beta.float()
    if res is not None:
        y = y + res.float()
    if relu:
        y = torch.relu(y)
    return y.to(x.dtype), mean, rstd


def batch_norm_bwd(x, dy, y, gamma, mean, rstd, relu, need_dres):
    """Returns (dx, dres, dgamma, dbeta) for :func:`batch_norm_fwd` in training mode."""
    C = x.shape[-1]
    g = dy.float()
    if relu:
        g = g * (y.float() > 0)
    xh = (x.float() - mean) * rstd
    g2, xh2 = g.reshape(-1, C), xh.reshape(-1, C)
    R = g2.shape[0]
    dbeta = g2.sum(0)
    dgamma = (g2 * xh2).sum(0)
    dx = (gamma.float() * rstd) * (g - dbeta / R - xh * (dgamma / R))
    return dx.to(x.dtype), (g.to(x.dtype) if need_dres else None), dgamma, dbeta
