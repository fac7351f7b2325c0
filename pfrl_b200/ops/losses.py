"""Fused loss ops (forward + backward CUDA kernels in csrc/losses.cu) as
torch.autograd Functions.  Inputs are CUDA tensors of any float (or bool / integer
for ``terminal``) dtype and any layout; each is converted to a contiguous fp32 copy
that stays referenced until the launch has been enqueued.  There is no CPU path
here -- agents fall back to their torch formulation on CPU."""
import ctypes

import torch

from pfrl_b200 import _lib


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _f32(t):
    t = t.detach()
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


class _C51Loss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, y, next_p, reward, discount, terminal, weights, z, mean):
        L = _lib.load()
        B, n = y.shape
        # every converted input stays bound to a local until the launch: _p keeps only the
        # address, and a temporary freed early is handed to the next conversion
        yc, pc, rc, dc, tc = _f32(y), _f32(next_p), _f32(reward), _f32(discount), _f32(terminal)
        w = None if weights is None else _f32(weights)
        zc = _f32(z)
        t = torch.empty_like(yc)
        delta = torch.empty(B, dtype=torch.float32, device=y.device)
        scratch = torch.empty(B, dtype=torch.float32, device=y.device)
        loss = torch.empty((), dtype=torch.float32, device=y.device)
        _lib.check(L.b2rl_c51_loss_fwd(
            _p(yc), _p(pc), _p(rc), _p(dc), _p(tc), _p(w),
            _p(zc), B, n, int(mean), _p(t), _p(delta), _p(scratch), _p(loss), _stream()))
        ctx.save_for_backward(yc, t, w if w is not None else torch.empty(0, device=y.device))
        ctx.has_w = w is not None
        ctx.mean = int(mean)
        ctx.mark_non_differentiable(delta, t)
        return loss, delta, t

    @staticmethod
    def backward(ctx, g_loss, g_delta, g_t):
        L = _lib.load()
        y, t, w = ctx.saved_tensors
        B, n = y.shape
        grad_y = torch.empty_like(y)
        g = _f32(g_loss).reshape(1)
        _lib.check(L.b2rl_c51_loss_bwd(_p(y), _p(t), _p(w) if ctx.has_w else None, _p(g), B, n,
                                       ctx.mean, _p(grad_y), _stream()))
        return grad_y, None, None, None, None, None, None, None


def c51_loss(y, next_p, reward, discount, terminal, weights, v_min=None, v_max=None, mean=True,
             z=None, return_target=False):
    """Categorical projection + cross entropy.  Returns (loss, per-sample
    priority errors[, projected target])."""
    if z is None:
        z = torch.linspace(v_min, v_max, y.shape[1], dtype=torch.float32, device=y.device)
    loss, delta, t = _C51Loss.apply(y, next_p, reward, discount, terminal, weights, z, mean)
    return (loss, delta, t) if return_target else (loss, delta)


class _TdLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, q, action, next_q, reward, discount, terminal, weights, clip_delta, mean):
        L = _lib.load()
        B, nA = q.shape
        # converted inputs stay referenced until the launch (see _C51Loss.forward)
        qc, nqc, rc, dc, tc = _f32(q), _f32(next_q), _f32(reward), _f32(discount), _f32(terminal)
        act = action.detach().long().contiguous()
        w = None if weights is None else _f32(weights)
        dev = q.device
        y = torch.empty(B, dtype=torch.float32, device=dev)
        t = torch.empty(B, dtype=torch.float32, device=dev)
        delta = torch.empty(B, dtype=torch.float32, device=dev)
        scratch = torch.empty(B, dtype=torch.float32, device=dev)
        loss = torch.empty((), dtype=torch.float32, device=dev)
        _lib.check(L.b2rl_td_loss_fwd(
            _p(qc), _p(act), _p(nqc), _p(rc), _p(dc), _p(tc), _p(w), B, nA, int(clip_delta),
            int(mean), _p(y), _p(t), _p(delta), _p(scratch), _p(loss), _stream()))
        ctx.save_for_backward(y, t, act, w if w is not None else torch.empty(0, device=dev))
        ctx.has_w = w is not None
        ctx.cfg = (B, nA, int(clip_delta), int(mean))
        ctx.mark_non_differentiable(delta, y, t)
        return loss, delta, y, t

    @staticmethod
    def backward(ctx, g_loss, *unused):
        L = _lib.load()
        y, t, act, w = ctx.saved_tensors
        B, nA, clip_delta, mean = ctx.cfg
        grad_q = torch.empty((B, nA), dtype=torch.float32, device=y.device)
        g = _f32(g_loss).reshape(1)
        _lib.check(L.b2rl_td_loss_bwd(_p(y), _p(t), _p(w) if ctx.has_w else None, _p(act), _p(g),
                                      B, nA, clip_delta, mean, _p(grad_q), _stream()))
        return grad_q, None, None, None, None, None, None, None, None


def td_loss(q, action, next_q, reward, discount, terminal, weights, clip_delta=True, mean=True):
    """Scalar TD loss.  Returns (loss, |y - t|, y, t)."""
    return _TdLoss.apply(q, action, next_q, reward, discount, terminal, weights, clip_delta, mean)


class _QuantileHuber(torch.autograd.Function):
    @staticmethod
    def forward(ctx, y, t, taus, weights, mean):
        L = _lib.load()
        B, N = y.shape
        Np = t.shape[1]
        yc, tc, tau = _f32(y), _f32(t), _f32(taus)
        w = None if weights is None else _f32(weights)
        dev = y.device
        delta = torch.empty(B, dtype=torch.float32, device=dev)
        scratch = torch.empty(B, dtype=torch.float32, device=dev)
        loss = torch.empty((), dtype=torch.float32, device=dev)
        _lib.check(L.b2rl_quantile_huber_fwd(_p(yc), _p(tc), _p(tau), _p(w), B, N, Np, int(mean),
                                             _p(delta), _p(scratch), _p(loss), _stream()))
        ctx.save_for_backward(yc, tc, tau, w if w is not None else torch.empty(0, device=dev))
        ctx.has_w = w is not None
        ctx.mean = int(mean)
        ctx.mark_non_differentiable(delta)
        return loss, delta

    @staticmethod
    def backward(ctx, g_loss, g_delta):
        L = _lib.load()
        y, t, tau, w = ctx.saved_tensors
        B, N = y.shape
        Np = t.shape[1]
        grad_y = torch.empty_like(y)
        g = _f32(g_loss).reshape(1)
        _lib.check(L.b2rl_quantile_huber_bwd(_p(y), _p(t), _p(tau), _p(w) if ctx.has_w else None,
                                             _p(g), B, N, Np, ctx.mean, _p(grad_y), _stream()))
        return grad_y, None, None, None, None


def quantile_huber_loss(y, t, taus, weights, mean=True):
    """IQN loss.  Returns (loss, per-sample mean error)."""
    return _QuantileHuber.apply(y, t, taus, weights, mean)
