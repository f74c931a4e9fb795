"""Optimizer split for BSP ("cdd" mode) and the flat fused SGD.

Reference: ``theanompi/lib/opt.py`` builds two Theano functions per model,
``get_vel`` (fwd + bwd + *pre* update into the send buffers ``vels``) and
``descent_vel`` (*post* update from the receive buffers ``vels2``), with one
elementwise kernel per tensor per buffer (``opt.py:2-52,181-330``).

Here the three reference optimizers keep their names and algebra but act on the
flat arena (one launch each):

``BSP_MSGD``   aggregate *momentum*  (``opt.py:181-268``)
               pre : U ← μU + (G + ηW)            send = U
               post: W ← W − lr·m · R / k          (R = Σ_ranks U)
``_BSP_MSGD``  aggregate *gradient*  (``opt.py:78-177``)
               pre : G ← (G + ηW) / k              send = G
               post: U ← μU + R ;  W ← W − lr·m · U
``BSP_SGD``    no momentum           (``opt.py:271-330``)
               pre : G ← lr·m · (G + ηW) / k       send = G
               post: W ← W − R

(m = per-group lr multiplier: 1 for 'W', 2 for 'b'; η only on 'W'; BN gamma/beta
are updated locally in the pre step and never exchanged, ``opt.py:207-226``.)

Models with ``optimizer = 'adam'`` use :func:`_pre_post_adam` instead (send = G, Adam
on R / k after the exchange, :class:`FlatAdam`).

The B200 fast path does not use the split at all: the fused exchanger kernels
(``csrc/comm_kernels.cu``) read every peer's G over NVLink, average, and apply
the momentum/weight-decay/lr update in the same pass — :class:`FlatSGD` is the
k = 1 (single GPU) instance of that kernel.

Reference bug fixed (SURVEY §2.9 #8): ``cdd_iter_fn`` applied ``descent_vel()``
*before* the next ``get_vel()``; here the post step runs right after the exchange,
so validation and checkpoints always see fully-updated weights.  The reference's
Nesterov expression (``mu**2*u - (1+mu)*g`` followed by ``w - lr*u``) has the
wrong sign; we implement the standard form  ``w ← w − lr (g_eff + μ u_new)``.
"""
from __future__ import annotations

import torch

from ..ops import reference as ref


class SharedScalar(object):
    """``theano.shared`` look-alike backed by one element of a device tensor so
    CUDA graphs pick up new values without re-capture (``model.shared_lr``)."""

    def __init__(self, buf, index, value=0.0):
        self._buf, self._i = buf, index
        self._host = float(value)
        self.set_value(value)

    def get_value(self):
        return self._host

    def set_value(self, v):
        self._host = float(v)
        self._buf[self._i] = float(v)


def _native_for(t):
    if t.is_cuda:
        from ..ops import cuda_impl
        return cuda_impl
    return None


class FlatSGD(object):
    """Fused momentum-SGD over the whole arena (or a block range)."""

    def __init__(self, arena, mu=0.9, nesterov=False, use_momentum=True):
        self.arena = arena
        self.mu = mu if use_momentum else 0.0
        self.nesterov = nesterov

    def step(self, lr, k=1, src="G", lo=0, hi=None, only_local=False, only_exchanged=False):
        a = self.arena
        hi = a.numel if hi is None else hi
        g = getattr(a, src)
        nat = _native_for(a.W)
        if nat is not None:
            nat.sgd_flat(a, g, lr, self.mu, self.nesterov, 1.0 / k, lo, hi,
                         only_local=only_local, only_exchanged=only_exchanged)
            return
        sl = slice(lo, hi)
        lrm, wd = a.lr_mult_vector()[sl], a.wd_vector()[sl]
        w, gg, u = a.W[sl], g[sl], a.U[sl]
        if only_local or only_exchanged:
            ex = a.exch_vector()[sl]
            m = ~ex if only_local else ex
            idx = m.nonzero().squeeze(1)
            if idx.numel() == 0:
                return
            w2, u2 = w[idx].clone(), u[idx].clone()
            ref.sgd_flat(w2, gg[idx], u2, lrm[idx], wd[idx], lr, self.mu, self.nesterov, 1.0 / k)
            w[idx] = w2
            u[idx] = u2
        else:
            ref.sgd_flat(w, gg, u, lrm, wd, lr, self.mu, self.nesterov, 1.0 / k)
        if a.H is not None:
            a.H[sl].copy_(w)


class FlatAdam(object):
    """Adam over the arena in one native kernel (``csrc/comm_kernels.cu: adam_flat_kernel``): first moment in the arena's U
    region, second moment in its V region, step counter (``arena.adam_t``) and lr in device memory — the step is CUDA-graph
    capturable.  The reference's Wide-ResNet uses Keras Adam (``keras_model_zoo/wresnet.py:159``)."""

    def __init__(self, arena, b1=0.9, b2=0.999, eps=1e-8):
        arena.ensure_adam_state()
        self.arena, self.b1, self.b2, self.eps = arena, b1, b2, eps

    @property
    def V(self):
        return self.arena.V

    @property
    def t(self):
        return self.arena.adam_t

    def step(self, lr=None, k=1, src="G", only_local=False, only_exchanged=False, advance=True):
        """Adam on ``src / k`` (``src`` = the G or R region) for all groups, only the non-exchanged (BN) ones or only the
        exchanged ones; ``advance=False`` leaves the step counter for a later call of the same step."""
        a = self.arena
        g = getattr(a, src)
        nat = _native_for(a.W)
        if nat is not None:
            from ..ops.cuda_impl import L, _table, _p, _st
            lrm, wd, ex = _table(a)
            filt = 1 if only_local else (2 if only_exchanged else 0)
            L().adam_flat(a.W.data_ptr(), g.data_ptr(), a.U.data_ptr(), a.V.data_ptr(), _p(a.H), a.block_group.data_ptr(), lrm, wd, ex,
                          a.hyper.data_ptr(), a.adam_t.data_ptr(), float(self.b1), float(self.b2), float(self.eps), 0, int(a.numel),
                          _st(a.W), inv_k=1.0 / k, filter=filt, advance=int(bool(advance)))
            return
        lr = float(a.hyper[0]) if lr is None else lr
        t = float(int(a.adam_t) + 1)
        lrm, wd = a.lr_mult_vector(), a.wd_vector()
        if only_local or only_exchanged:
            ex = a.exch_vector()
            idx = (~ex if only_local else ex).nonzero().squeeze(1)
            if idx.numel():
                w2, m2, v2 = a.W[idx].clone(), a.U[idx].clone(), a.V[idx].clone()
                ref.adam_flat(w2, g[idx], m2, v2, lrm[idx], wd[idx], lr, self.b1, self.b2, self.eps, t, 1.0 / k)
                a.W[idx], a.U[idx], a.V[idx] = w2, m2, v2
        else:
            ref.adam_flat(a.W, g, a.U, a.V, lrm, wd, lr, self.b1, self.b2, self.eps, t, 1.0 / k)
        if advance:
            a.adam_t += 1
        if a.H is not None:
            a.H.copy_(a.W)

    def state_dict(self):
        return {"V": self.V.detach().cpu().clone(), "t": int(self.t)}

    def load_state_dict(self, sd):
        self.V.copy_(sd["V"].to(self.V.device)); self.t.fill_(int(sd["t"]))


# --------------------------------------------------------------------------- classic split (API parity)
def _ex(a):
    return a.exch_vector()


def _pre_post_msgd(model, use_nesterov, k):
    """BSP_MSGD: aggregate momentum."""
    a, mu = model.arena, (model.mu if model.use_momentum else 0.0)
    sgd = FlatSGD(a, mu, use_nesterov, True)

    def pre():
        lr = model.shared_lr.get_value()
        if k == 1:
            sgd.step(lr, 1)
            return
        sgd.step(lr, 1, only_local=True)                      # BN params: full local update
        ex = _ex(a)
        g_eff = a.G + a.wd_vector() * a.W
        a.U.copy_(torch.where(ex, mu * a.U + g_eff, a.U))
        model._send_region = "U"

    def post():
        if k == 1:
            return
        lr = model.shared_lr.get_value()
        ex = _ex(a)
        a.W.sub_(torch.where(ex, lr * a.lr_mult_vector() * a.R / float(k), torch.zeros_like(a.W)))
        a.refresh_shadow()

    return pre, post, "U"


def _pre_post_msgd_grad(model, use_nesterov, k):
    """_BSP_MSGD: aggregate gradient."""
    a, mu = model.arena, (model.mu if model.use_momentum else 0.0)
    sgd = FlatSGD(a, mu, use_nesterov, True)

    def pre():
        lr = model.shared_lr.get_value()
        if k == 1:
            sgd.step(lr, 1)
            return
        sgd.step(lr, 1, only_local=True)
        ex = _ex(a)
        a.G.copy_(torch.where(ex, (a.G + a.wd_vector() * a.W) / float(k), a.G))

    def post():
        if k == 1:
            return
        lr = model.shared_lr.get_value()
        ex = _ex(a)
        u_new = mu * a.U + a.R
        step = a.R + mu * u_new if use_nesterov else u_new
        a.U.copy_(torch.where(ex, u_new, a.U))
        a.W.sub_(torch.where(ex, lr * a.lr_mult_vector() * step, torch.zeros_like(a.W)))
        a.refresh_shadow()

    return pre, post, "G"


def _pre_post_sgd(model, k):
    a = model.arena
    sgd = FlatSGD(a, 0.0, False, False)

    def pre():
        lr = model.shared_lr.get_value()
        if k == 1:
            sgd.step(lr, 1)
            return
        sgd.step(lr, 1, only_local=True)
        ex = _ex(a)
        a.G.copy_(torch.where(ex, lr * a.lr_mult_vector() * (a.G + a.wd_vector() * a.W) / float(k), a.G))

    def post():
        if k == 1:
            return
        ex = _ex(a)
        a.W.sub_(torch.where(ex, a.R, torch.zeros_like(a.W)))
        a.refresh_shadow()

    return pre, post, "G"


def _pre_post_adam(model, k):
    """Synchronous data-parallel Adam: average the gradients, then one Adam step (= single-process Adam on the global batch).
    pre : local Adam step of the non-exchanged (BN) groups on the rank's own G            send = G
    post: Adam step of the exchanged groups on R / k (R = Σ_ranks G), then t += 1
    The fused strategies compute the same thing inside the exchange kernels."""
    adam = model.adam

    def pre():
        if k == 1:
            adam.step()
            return
        adam.step(only_local=True, advance=False)

    def post():
        if k == 1:
            return
        adam.step(k=k, src="R", only_exchanged=True)

    return pre, post, "G"


def _publish(model, pre, post, send_region, k):
    a = model.arena
    mask = a.exchanged_mask()
    if k > 1:
        model.vels = [v for v, m in zip(a.views(send_region), mask) if m]
        model.vels2 = [v for v, m in zip(a.views("R"), mask) if m]
    else:
        model.vels, model.vels2 = [], []
    model._send_region = send_region
    return pre, post


def BSP_MSGD(model, use_nesterov_momentum, k=1):
    return _publish(model, *_pre_post_msgd(model, use_nesterov_momentum, k), k)


def _BSP_MSGD(model, use_nesterov_momentum, k=1):
    return _publish(model, *_pre_post_msgd_grad(model, use_nesterov_momentum, k), k)


def BSP_SGD(model, k=1):
    return _publish(model, *_pre_post_sgd(model, k), k)


def _clip_paramlist(param_list, scale=10):
    """``T.clip(param,-10,10)`` helper (ref ``opt.py:67-75``; unused there too)."""
    with torch.no_grad():
        for p in param_list:
            p.clamp_(-scale, scale)
    return param_list


def prepare_update_dict(model, k=1, aggregate="momentum"):
    if getattr(model, "optimizer", "msgd") == "adam":
        return _publish(model, *_pre_post_adam(model, k), k)
    if model.use_momentum:
        if aggregate == "gradient":
            return _BSP_MSGD(model, model.use_nesterov_momentum, k=k)
        return BSP_MSGD(model, model.use_nesterov_momentum, k=k)
    return BSP_SGD(model, k=k)


def pre_model_iter_fn(model, k=1, f_train=True, f_val=True, aggregate="momentum", fused_tail=None):
    """Build ``model.get_vel / descent_vel / train_iter_fn / val_iter_fn``
    (ref ``opt.py:2-52``).  ``get_vel(subb)`` = forward + backward + pre update and
    returns ``(cost, error)``; ``descent_vel()`` = post update.

    When the update is self-contained (k = 1) or a fused exchanger supplies
    ``fused_tail`` (allreduce + SGD in one kernel family) the update is registered as
    the model's *step tail* so it is part of the CUDA-graph-captured step, and
    ``descent_vel`` is a no-op."""
    if f_train:
        pre, post = prepare_update_dict(model, k=k, aggregate=aggregate)
        tail = fused_tail if fused_tail is not None else (pre if k == 1 else None)
        model.set_step_tail(tail)

        def get_vel(subb_ind=0):
            cost, err = model.forward_backward(subb_ind)
            if tail is None:
                with torch.no_grad():
                    pre()
            return cost, err

        def descent_vel():
            if tail is None:
                with torch.no_grad():
                    post()

        model.get_vel, model.descent_vel = get_vel, descent_vel
        model.compiled_train_fn_list = [get_vel, descent_vel]
        model.train_iter_fn = choose_iter_fn(model)
    if f_val:
        model.compile_val()
        model.val_iter_fn = model.val_fn


def choose_iter_fn(model):
    """The reference returns ``cdd_iter_fn`` = descent_vel(); get_vel() (one step
    late).  We return get_vel only — the exchanger calls ``descent_vel`` right after
    the collective (see module docstring)."""

    def cdd_iter_fn(subb_ind=0):
        return model.get_vel(subb_ind)

    return cdd_iter_fn
