"""PPO kernels (csrc/ppo.cu) behind torch: GAE over a [T, E] rollout and the
fused clipped-surrogate loss as an autograd Function.  Inputs are CUDA tensors of any
float dtype and any layout (``cut``/``valid``: bool or integer); each is converted to a
contiguous fp32 (uint8) copy that stays referenced until the launch has been enqueued."""
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


def gae(reward, nonterminal, v, v_next, cut, gamma, lambd, valid=None):
    """reward/nonterminal/v/v_next: float CUDA [T, E]; cut/valid: bool or uint8 [T, E].
    Returns (adv [T, E], v_teacher [T, E], stats [2] = mean, std)."""
    L = _lib.load()
    T, E = reward.shape
    dev = reward.device
    adv = torch.zeros((T, E), dtype=torch.float32, device=dev)
    vt = torch.zeros((T, E), dtype=torch.float32, device=dev)
    stats = torch.empty(2, dtype=torch.float32, device=dev)
    scratch = torch.empty(((E + 127) // 128) * 3, dtype=torch.float64, device=dev)
    # every converted input stays bound to a local until the launch: _p keeps only the
    # address, and a temporary freed early is handed to the next conversion
    rc, ntc, vc, vnc = _f32(reward), _f32(nonterminal), _f32(v), _f32(v_next)
    cut = cut.to(torch.uint8).contiguous()
    if valid is not None:
        valid = valid.to(torch.uint8).contiguous()
    _lib.check(L.b2rl_gae(_p(rc), _p(ntc), _p(vc), _p(vnc), _p(cut), _p(valid), T, E,
                          float(gamma), float(lambd), _p(adv), _p(vt), _p(scratch), _p(stats),
                          _stream()))
    return adv, vt, stats


class _PpoLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, log_prob, entropy, v_pred, log_prob_old, v_pred_old, adv, v_teacher,
                adv_stats, clip_eps, clip_eps_vf, value_coef, entropy_coef):
        L = _lib.load()
        M = log_prob.numel()
        dev = log_prob.device
        g_lp = torch.empty(M, dtype=torch.float32, device=dev)
        g_en = torch.empty(M, dtype=torch.float32, device=dev)
        g_v = torch.empty(M, dtype=torch.float32, device=dev)
        losses = torch.empty(4, dtype=torch.float32, device=dev)
        scratch = torch.empty(((M + 255) // 256) * 3, dtype=torch.float64, device=dev)
        # converted inputs stay referenced until the launch (see gae)
        args = [None if x is None else _f32(x).view(-1)
                for x in (log_prob, entropy, v_pred, log_prob_old, v_pred_old, adv, v_teacher,
                          adv_stats)]
        _lib.check(L.b2rl_ppo_loss(
            *[_p(x) for x in args], M, float(clip_eps),
            -1.0 if clip_eps_vf is None else float(clip_eps_vf), float(value_coef),
            float(entropy_coef), _p(g_lp), _p(g_en), _p(g_v), _p(scratch), _p(losses),
            _stream()))
        ctx.save_for_backward(g_lp, g_en, g_v)
        ctx.shapes = (log_prob.shape, entropy.shape, v_pred.shape)
        ctx.mark_non_differentiable(losses)
        return losses[0].clone(), losses

    @staticmethod
    def backward(ctx, g_total, g_losses):
        g_lp, g_en, g_v = ctx.saved_tensors
        s_lp, s_en, s_v = ctx.shapes
        return ((g_lp * g_total).view(s_lp), (g_en * g_total).view(s_en),
                (g_v * g_total).view(s_v), None, None, None, None, None, None, None, None, None)


def ppo_loss(log_prob, entropy, v_pred, log_prob_old, v_pred_old, adv, v_teacher, adv_stats,
             clip_eps, clip_eps_vf, value_coef, entropy_coef):
    """Returns (total loss (differentiable), losses[4] = total/policy/value/entropy)."""
    return _PpoLoss.apply(log_prob, entropy, v_pred, log_prob_old, v_pred_old, adv, v_teacher,
                          adv_stats, clip_eps, clip_eps_vf, value_coef, entropy_coef)
