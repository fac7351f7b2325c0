"""torch-float64 restatements of the reference's loss, GAE and PPO formulas (test
infrastructure only), with autograd for the gradients.

The inputs are the fp32 values a kernel reads, widened exactly to fp64, and every
operation runs in fp64.  Two exceptions keep the reference's fp32 semantics where a
value or gradient is discontinuous, so that the selection made here is the one the
kernel makes:
- constants the kernels hold in fp32 (the C51 clamp bound float32(1e-10), the PPO
  clip range 1 -+ float32(clip_eps), the value clip bounds v_old -+ clip_eps_vf) are
  rounded to fp32 first;
- the PPO value loss picks max(unclipped, clipped) from the fp32 squared errors,
  with autograd's rule for torch.max (half the gradient to each side of a tie).
Everything else goes through torch's own min / max / clamp / smooth_l1_loss, so
ties and boundaries follow autograd: half-and-half at a min / max tie, gradient
passed at both ends of a clamp.

Differentiable inputs: pass an fp64 leaf (``x.double().requires_grad_()``); the
conversion below leaves fp64 tensors as they are."""
import numpy as np
import torch
import torch.nn.functional as F

F64 = torch.float64
C51_Y_MIN = float(np.float32(1e-10))  # torch.clamp(y, 1e-10, 1.0) on an fp32 y
PPO_STD_EPS = float(np.float32(1e-8))  # (advs - mean) / (std + 1e-8) on fp32 tensors


def _d(x):
    return None if x is None else torch.as_tensor(x).to(F64)


def _f32(x):
    return float(np.float32(x))


def _reduce(per, weights, mean):
    """compute_weighted_value_loss / compute_value_loss: sum (weighted), / B for mean."""
    s = (per * weights).sum() if weights is not None else per.sum()
    return s / per.shape[0] if mean else s


def td_loss(q, action, next_q, reward, discount, terminal, weights, clip_delta, mean):
    """pfrl/agents/dqn.py:44-104 with t = r + discount * (1 - terminal) * next_q
    (dqn.py:405).  Returns loss, |y - t|, y, t."""
    q = _d(q)
    next_q, reward, discount, terminal, weights = map(
        _d, (next_q, reward, discount, terminal, weights))
    y = q.gather(1, torch.as_tensor(action).long().view(-1, 1).to(q.device)).view(-1)
    t = reward + discount * (1.0 - terminal) * next_q
    if clip_delta:
        per = F.smooth_l1_loss(y, t, reduction="none")
    else:
        per = F.mse_loss(y, t, reduction="none") / 2
    return _reduce(per, weights, mean), (y - t).abs(), y, t


def categorical_projection(Tz, p, z):
    """pfrl/agents/categorical_dqn.py:7-57 (1 - (bj - l) onto l, bj - l onto u)."""
    Tz, p, z = _d(Tz), _d(p), _d(z)
    n = z.numel()
    v_min, v_max = float(z[0]), float(z[-1])
    dz = float(z[1] - z[0])
    bj = ((Tz.clamp(v_min, v_max) - v_min) / dz).clamp(0, n - 1)
    lo, up = bj.floor(), bj.ceil()
    out = torch.zeros_like(p)
    out.scatter_add_(1, lo.long(), p * (1 - (bj - lo)))
    out.scatter_add_(1, up.long(), p * (bj - lo))
    return out


def c51_loss(y, next_p, reward, discount, terminal, weights, z, mean):
    """categorical_dqn.py:140-152 (Tz), :7-57 (projection), :178-204 (cross entropy,
    per-sample error, weighted sum).  Returns loss, per-sample error, target."""
    y = _d(y)
    reward, discount, terminal, weights, z = map(_d, (reward, discount, terminal, weights, z))
    Tz = reward[:, None] + (1.0 - terminal[:, None]) * discount[:, None] * z[None]
    t = categorical_projection(Tz, next_p, z)
    elt = -t * torch.log(torch.clamp(y, C51_Y_MIN, 1.0))
    per = elt.sum(1)
    return _reduce(per, weights, mean), per, t


def quantile_huber(y, t, taus, weights, mean):
    """pfrl/agents/iqn.py:176-250: elementwise |tau - 1[t < y]| * smooth_l1(y, t), mean
    over N', sum over N.  Returns loss, per-sample mean error (iqn.py:388)."""
    y = _d(y)
    t, taus, weights = map(_d, (t, taus, weights))
    yy, tt, ta = torch.broadcast_tensors(y[:, :, None], t[:, None, :], taus[:, :, None])
    ind = (tt < yy).to(F64)
    elt = torch.abs(ta - ind) * F.smooth_l1_loss(yy, tt, reduction="none")
    return _reduce(elt.mean(2).sum(1), weights, mean), elt.mean((1, 2))


def gae(reward, nonterminal, v, v_next, cut, gamma, lambd, valid=None):
    """pfrl/agents/ppo.py:36-53 per episode segment on time-major [T, E] arrays.  ``cut``
    marks the last transition of a segment; a slot with ``valid`` false holds no
    transition: adv = v_teacher = 0 there, and the segment before it ends.

    Returns adv, v_teacher and sum_k (gamma lambda)^k |delta_{t+k}| over the same
    segment (the magnitude the fp32 rounding of adv is measured against)."""
    reward, nonterminal, v, v_next = map(_d, (reward, nonterminal, v, v_next))
    cut = torch.as_tensor(cut).bool()
    valid = torch.ones_like(cut) if valid is None else torch.as_tensor(valid).bool()
    T, E = reward.shape
    adv = torch.zeros_like(reward)
    mag = torch.zeros_like(reward)
    a = torch.zeros(E, dtype=F64, device=reward.device)
    m = torch.zeros_like(a)
    gl = gamma * lambd
    for t in range(T - 1, -1, -1):
        keep = (valid[t] & ~cut[t]).to(F64)  # the carry from t + 1 ends at a cut
        a, m = a * keep, m * keep
        delta = reward[t] + gamma * nonterminal[t] * v_next[t] - v[t]
        a = torch.where(valid[t], delta + gl * a, torch.zeros_like(a))
        m = torch.where(valid[t], delta.abs() + gl * m, torch.zeros_like(m))
        adv[t], mag[t] = a, m
    vt = torch.where(valid, adv + v, torch.zeros_like(adv))
    return adv, vt, mag


def ppo_loss(log_prob, entropy, v_pred, log_prob_old, v_pred_old, adv, v_teacher, adv_stats,
             clip_eps, clip_eps_vf, value_coef, entropy_coef):
    """pfrl/agents/ppo.py:495 (standardised advantages) and :634-671 (_lossfun).
    Returns total, policy, value and entropy losses."""
    log_prob, entropy, v_pred = _d(log_prob), _d(entropy), _d(v_pred)
    a = _d(adv)
    if adv_stats is not None:
        st = _d(adv_stats)
        a = (a - st[0]) / (st[1] + PPO_STD_EPS)
    ratio = torch.exp(log_prob - _d(log_prob_old))
    eps = np.float32(clip_eps)
    rc = torch.clamp(ratio, float(np.float32(1) - eps), float(np.float32(1) + eps))
    loss_policy = -torch.mean(torch.min(ratio * a, rc * a))
    vt = _d(v_teacher)
    l_plain = (v_pred - vt) ** 2
    if clip_eps_vf is None:
        lv = l_plain
    else:
        vo32 = torch.as_tensor(v_pred_old).float()
        lo32, hi32 = vo32 - _f32(clip_eps_vf), vo32 + _f32(clip_eps_vf)
        vc = torch.min(torch.max(v_pred, lo32.to(F64)), hi32.to(F64))  # ppo.py:28-33
        l_clip = (vc - vt) ** 2
        # torch.max(l_plain, l_clip), branch taken on the fp32 squared errors
        v32, vt32 = torch.as_tensor(v_pred).float(), torch.as_tensor(v_teacher).float()
        vc32 = torch.min(torch.max(v32, lo32), hi32)
        p32, c32 = (v32 - vt32) * (v32 - vt32), (vc32 - vt32) * (vc32 - vt32)
        sel = (c32 > p32).to(F64) + 0.5 * (c32 == p32).to(F64)
        lv = l_plain * (1 - sel) + l_clip * sel
    loss_value = torch.mean(lv)
    loss_entropy = -torch.mean(entropy)
    total = loss_policy + value_coef * loss_value + entropy_coef * loss_entropy
    return total, loss_policy, loss_value, loss_entropy
