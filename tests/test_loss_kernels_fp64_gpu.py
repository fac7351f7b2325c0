"""GPU: the fused loss kernels (csrc/losses.cu), GAE and the PPO loss (csrc/ppo.cu),
forward and backward through their autograd Functions, against the fp64
restatements in tests/fp64_losses.py at the edges of each launch shape and at the
shapes the agents run.

Tolerances follow from fp32 rounding, u = 2^-24.  Each bound below counts the
roundings on the kernel's path and is then doubled; every case prints the worst
ratio of error to bound, and a ratio above 1 fails.
- TD: t = r + disc (1 - term) next_q rounds three times, err_t <= 3u (|r| + |disc
  next_q|); d = y - t adds u |d|.  Huber' and clamp(d, -1, 1) are 1-Lipschitz, so a
  per-sample loss moves by at most min(|d|, 1) err_d + 2u l and a gradient entry by
  |g| (err_d + 3u) with g = 0.37 w / B.
- C51: fp32 bj = (Tz - v_min) / delta_z is off by at most
  K_j = u (3 (|r| + |s z_j|) + 3 (v_max - v_min)) / delta_z, s = (1 - term) disc.
  The projection is piecewise linear with slope 1 in bj, so a row's target moves by
  at most sum_j p_j (2 K_j + u (4 + n)) in total (n: the most shared-memory adds onto
  one atom); that bounds each entry and, times max |log clamp(y)|, the per-sample
  error, which adds u (n / 32 + 8) sum_k t_k |log y_k| for logf and the warp sum.
  Gradient -g t / y: (g / y) (that target bound + 5u t).
- Quantile Huber: each pair |tau - I| huber(d) is within 8u of itself (huber is
  within 2u |huber| of itself under a relative error u in d); a thread adds
  ceil(N N' / 256) of them and the tree 8 more levels: u (ceil(N N' / 256) + 16)
  sum |pair|.  Gradient: |g / N'| u (N' + 8) sum_m |tau - I| |clamp(d)|.
- Batch reductions (TD, C51, QH finish_sum: ceil(B / 256) adds per thread, 8 tree
  levels, the weight product and the division): the per-sample bounds, weighted,
  plus u (ceil(B / 256) + 10) sum_i |w_i l_i|, over B for mean, plus u |loss|.
- GAE runs in fp64 and rounds once to fp32: |adv - adv64| <= u |adv64| <= u
  sum_k (gamma lambda)^k |delta_{t+k}| over the segment; v_teacher adds u |v|.
  stats: mean and std (fp64 sums, T + 40 adds deep) of the kernel's own fp32
  advantages over the valid slots, rounded once to fp32.
- PPO: ratio = expf(x), x = lp - lp_old, is within u (|x| + 4) of exp(x) (2 ulp
  expf); the standardised advantage within 3u; each surrogate within
  u (|x| + 9) |ratio adv|, each squared error within 3u; per-row sums are fp64,
  and the four losses round to fp32 (three more roundings for the total).  Gradient
  rows add the 1 / M and the upstream-gradient products (two or three u).

Discontinuities (the Huber kink has none; the C51 y clamp, PPO's clip range,
min / max selection) are taken from the same fp32 quantities the kernel compares,
see tests/fp64_losses.py; PPO rows whose fp32 ratio lies within 1e-5 of a clip
bound are moved onto lp == lp_old, since expf and exp may round such a ratio to
either side.  Every backward is driven with 0.37 * loss, so that a kernel that
ignores grad_loss fails."""
import math

import numpy as np
import pytest
import torch

import fp64_losses as R
from pfrl_b200.ops.losses import c51_loss, quantile_huber_loss, td_loss
from pfrl_b200.ops.ppo import gae, ppo_loss

pytestmark = pytest.mark.gpu
U = 2.0 ** -24
F64 = torch.float64
GL = float(np.float32(0.37))  # upstream gradient of every backward


def _check(case, name, got, want, bound):
    err = (got.detach().double() - want.detach().double()).abs()
    ratio = (err / (2 * bound).clamp_min(1e-300)).max().item()
    print("%s %-8s worst err/bound %.3g" % (case, name, ratio))
    assert ratio <= 1.0, (case, name, ratio)


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _leaf(x):
    return x.detach().double().requires_grad_(True)


def _grad(loss, x):
    (g,) = torch.autograd.grad(GL * loss, x)
    return g


def _reduce_bound(per_bound, per, w, mean):
    """Bound on a finish_sum batch reduction of w_i * per_i (see the module doc)."""
    B = per.shape[0]
    wa = torch.ones_like(per) if w is None else w.double().abs()
    b = (wa * per_bound).sum() + U * (math.ceil(B / 256) + 10) * (wa * per.abs()).sum()
    return b / B if mean else b


# ---------------------------------------------------------------------------
# TD
# ---------------------------------------------------------------------------
def _td_inputs(B, nA, seed):
    g = _gen(seed)
    q = 3 * torch.randn(B, nA, device="cuda", generator=g)
    action = torch.randint(0, nA, (B,), device="cuda", generator=g)
    next_q = 3 * torch.randn(B, device="cuda", generator=g)
    reward = torch.randn(B, device="cuda", generator=g)
    discount = 0.9 + 0.1 * torch.rand(B, device="cuda", generator=g)
    terminal = (torch.rand(B, device="cuda", generator=g) < 0.2).float()
    weights = 0.1 + 2 * torch.rand(B, device="cuda", generator=g)
    # planted: t = r exactly (terminal), d = y - t in {1, -1, 0} exactly
    for row, (r, y) in enumerate([(0.5, 1.5), (0.5, -0.5), (0.25, 0.25)][:B]):
        terminal[row], reward[row] = 1.0, r
        q[row, action[row]] = y
    return q, action, next_q, reward, discount, terminal, weights


@pytest.mark.parametrize("B,nA", [(1, 1), (1, 18), (31, 18), (256, 1), (256, 18), (257, 18),
                                  (512, 18), (4097, 1), (4097, 18)])
def test_td_loss_vs_fp64(B, nA):
    q, action, next_q, reward, discount, terminal, weights = _td_inputs(B, nA, B * 100 + nA)
    for clip in (True, False):
        for mean in (True, False):
            for w in (None, weights):
                case = "td B=%d nA=%d clip=%d mean=%d w=%d" % (B, nA, clip, mean, w is not None)
                qk = q.clone().requires_grad_(True)
                loss, delta, y, t = td_loss(qk, action, next_q, reward, discount, terminal, w,
                                            clip, mean)
                gq = _grad(loss, qk)
                q64 = _leaf(q)
                loss64, delta64, y64, t64 = R.td_loss(q64, action, next_q, reward, discount,
                                                      terminal, w, clip, mean)
                g64 = _grad(loss64, q64)
                err_t = 3 * U * (reward.double().abs() +
                                 (discount.double() * next_q.double()).abs())
                err_d = err_t + U * delta64.detach()
                ad = delta64.detach()
                per64 = (torch.where(ad < 1, 0.5 * ad * ad, ad - 0.5) if clip else 0.5 * ad * ad)
                per_b = (ad.clamp(max=1) if clip else ad) * err_d + 2 * U * per64
                _check(case, "t", t, t64, err_t)
                _check(case, "y", y, y64, torch.zeros_like(y64))
                _check(case, "delta", delta, delta64, err_d)
                _check(case, "loss", loss, loss64,
                       _reduce_bound(per_b, per64, w, mean) + U * loss64.abs())
                gs = GL * (torch.ones_like(ad) if w is None else w.double()) / (B if mean else 1)
                gb = torch.zeros_like(g64)
                gb.scatter_(1, action.view(-1, 1), (gs.abs() * (err_d + 3 * U)).view(-1, 1))
                _check(case, "grad", gq, g64, gb)


# ---------------------------------------------------------------------------
# C51
# ---------------------------------------------------------------------------
Y_PLANTS = [0.0, 1e-12, float(np.float32(1e-10)), 1.0, float(np.nextafter(np.float32(1),
                                                                          np.float32(2)))]


def _support(n, kind):
    if kind == "linspace":
        return torch.linspace(-10, 10, n, dtype=torch.float32, device="cuda")
    return (torch.arange(n, dtype=torch.float32, device="cuda") - (n - 1) / 2) * 0.5


def _c51_inputs(B, n, kind, seed):
    g = _gen(seed)
    z = _support(n, kind)
    y = torch.softmax(2 * torch.randn(B, n, device="cuda", generator=g), 1)
    next_p = torch.softmax(2 * torch.randn(B, n, device="cuda", generator=g), 1)
    reward = 2 * torch.randn(B, device="cuda", generator=g)
    discount = torch.where(torch.rand(B, device="cuda", generator=g) < 0.5,
                           torch.full((B,), 0.99, device="cuda"),
                           0.9 + 0.1 * torch.rand(B, device="cuda", generator=g))
    terminal = (torch.rand(B, device="cuda", generator=g) < 0.2).float()
    weights = 0.1 + 2 * torch.rand(B, device="cuda", generator=g)
    # planted rows: Tz on an atom (terminal, r = z_k), below v_min, above v_max, and
    # Tz_j = z_{j+1} on every atom (discount 1, r = one spacing)
    plants = [(1.0, 1.0, float(z[n // 3])), (0.0, 0.99, -1e3), (0.0, 0.99, 1e3),
              (0.0, 1.0, float(z[1] - z[0]))]
    for k, (term, disc, r) in enumerate(plants):
        row = (k + 3) % B
        terminal[row], discount[row], reward[row] = term, disc, r
    # planted y at the atom with the largest target mass of rows 0..4
    _, _, t64 = R.c51_loss(y, next_p, reward, discount, terminal, None, z, True)
    for k, val in enumerate(Y_PLANTS):
        row = k % B
        y[row, int(t64[row].argmax())] = val
    return y, next_p, reward, discount, terminal, weights, z


C51_CASES = ([(B, 51, "linspace") for B in (1, 7, 8, 9, 32, 512, 4097)] +
             [(512, n, "linspace") for n in (2, 31, 32, 33, 64, 200, 256)] +
             [(9, 51, "exact"), (512, 51, "exact"), (512, 2, "exact"), (512, 256, "exact")])


@pytest.mark.parametrize("B,n,kind", C51_CASES)
def test_c51_loss_vs_fp64(B, n, kind):
    y, next_p, reward, discount, terminal, weights, z = _c51_inputs(B, n, kind, B * 1000 + n)
    z64 = z.double()
    s = (1 - terminal.double()) * discount.double()
    dz = float(z64[1] - z64[0])
    K = U * (3 * (reward.double().abs()[:, None] + (s[:, None] * z64[None]).abs()) +
             3 * float(z64[-1] - z64[0])) / dz
    t_b = (next_p.double() * (2 * K + U * (4 + n))).sum(1)  # per-row target bound
    logy = torch.log(y.double().clamp(R.C51_Y_MIN, 1.0)).abs()
    for mean in (True, False):
        for w in (None, weights):
            case = "c51 B=%d n=%d %s mean=%d w=%d" % (B, n, kind, mean, w is not None)
            yk = y.clone().requires_grad_(True)
            loss, delta, t = c51_loss(yk, next_p, reward, discount, terminal, w, z=z, mean=mean,
                                      return_target=True)
            gy = _grad(loss, yk)
            y64 = _leaf(y)
            loss64, delta64, t64 = R.c51_loss(y64, next_p, reward, discount, terminal, w, z, mean)
            g64 = _grad(loss64, y64)
            d_b = t_b * logy.max(1).values + U * (n / 32 + 8) * (t64.detach() * logy).sum(1)
            _check(case, "target", t, t64, t_b[:, None].expand_as(t64))
            _check(case, "delta", delta, delta64, d_b)
            _check(case, "loss", loss, loss64,
                   _reduce_bound(d_b, delta64.detach(), w, mean) + U * loss64.abs())
            gs = GL * (torch.ones(B, dtype=F64, device="cuda") if w is None else w.double())
            gs = (gs / (B if mean else 1))[:, None]
            inside = (y.double() >= R.C51_Y_MIN) & (y.double() <= 1.0)
            gb = torch.where(inside, gs / y.double() * (t_b[:, None] + 5 * U * t64.detach()),
                             torch.zeros_like(g64))
            _check(case, "grad", gy, g64, gb)
    # the planted y values take the clamp's branches exactly as autograd does
    assert (gy[(y == 0) | (y == 1e-12) | (y > 1)] == 0).all()


# ---------------------------------------------------------------------------
# Quantile Huber
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("B,N,Np", [(1, 1, 1), (24, 16, 12), (32, 64, 64), (512, 64, 64),
                                    (3, 300, 1), (5, 1, 300), (2, 17, 257)])
def test_quantile_huber_vs_fp64(B, N, Np):
    g = _gen(B * N + Np)
    y = torch.randn(B, N, device="cuda", generator=g)
    t = 1.5 * torch.randn(B, Np, device="cuda", generator=g)
    taus = torch.rand(B, N, device="cuda", generator=g)
    weights = 0.1 + 2 * torch.rand(B, device="cuda", generator=g)
    # planted: d = t - y = 0 and |d| = 1 exactly
    y[0, 0] = t[0, 0]
    if N > 1 and Np > 1:
        y[0, 1], t[0, 1] = 0.25, 1.25
    y64d, t64d, tau64 = y.double(), t.double(), taus.double()
    dd = t64d[:, None, :] - y64d[:, :, None]
    wt = (tau64[:, :, None] - (dd < 0).double()).abs()
    A = (wt * torch.where(dd.abs() < 1, 0.5 * dd * dd, dd.abs() - 0.5)).sum((1, 2))
    s_b = U * (math.ceil(N * Np / 256) + 16) * A
    G = (wt * dd.clamp(-1, 1).abs()).sum(2)
    for mean in (True, False):
        for w in (None, weights):
            case = "qh B=%d N=%d N'=%d mean=%d w=%d" % (B, N, Np, mean, w is not None)
            yk = y.clone().requires_grad_(True)
            loss, err = quantile_huber_loss(yk, t, taus, w, mean)
            gy = _grad(loss, yk)
            y64 = _leaf(y)
            loss64, err64 = R.quantile_huber(y64, t, taus, w, mean)
            g64 = _grad(loss64, y64)
            _check(case, "err", err, err64, s_b / (N * Np) + U * err64.detach().abs())
            per = A / Np
            _check(case, "loss", loss, loss64,
                   _reduce_bound(s_b / Np, per, w, mean) + U * loss64.abs())
            gs = GL * (torch.ones(B, dtype=F64, device="cuda") if w is None else w.double())
            gs = (gs / Np / (B if mean else 1))[:, None]
            _check(case, "grad", gy, g64, gs.abs() * U * (Np + 8) * G)


# ---------------------------------------------------------------------------
# GAE
# ---------------------------------------------------------------------------
def _rollout(T, E, seed, with_valid):
    """Columns [0, E/3): cut on the last row only; [E/3, 2E/3): every row cut;
    the rest: random cuts and terminals, independent of each other (truncations and
    terminals that do not end the stored segment)."""
    g = _gen(seed)
    reward = torch.randn(T, E, device="cuda", generator=g)
    v = torch.randn(T, E, device="cuda", generator=g)
    v_next = torch.randn(T, E, device="cuda", generator=g)
    nonterminal = (torch.rand(T, E, device="cuda", generator=g) > 0.05).float()
    cut = torch.rand(T, E, device="cuda", generator=g) < 0.05
    a, b = E // 3, 2 * E // 3
    cut[:, :a] = False
    cut[:, a:b] = True
    cut[-1] = True
    valid = None
    if with_valid:
        valid = torch.rand(T, E, device="cuda", generator=g) > 0.05
        valid[T - T // 4:, ::7] = False  # partly filled columns
    return reward, nonterminal, v, v_next, cut, valid


@pytest.mark.parametrize("T,E", [(1, 1), (1, 129), (8, 256), (2048, 256), (7, 4097)])
@pytest.mark.parametrize("gamma,lambd", [(0.99, 0.95), (1.0, 1.0), (0.995, 0.0)])
def test_gae_vs_fp64(T, E, gamma, lambd):
    for with_valid in (False, True):
        case = "gae T=%d E=%d g=%g l=%g valid=%d" % (T, E, gamma, lambd, with_valid)
        reward, nonterminal, v, v_next, cut, valid = _rollout(T, E, T * E, with_valid)
        adv, vt, stats = gae(reward, nonterminal, v, v_next, cut, gamma, lambd, valid)
        adv64, vt64, mag = R.gae(reward, nonterminal, v, v_next, cut, gamma, lambd, valid)
        _check(case, "adv", adv, adv64, U * mag)
        _check(case, "v_teach", vt, vt64, U * (mag + v.double().abs()))
        sel = torch.ones_like(cut) if valid is None else valid
        if valid is not None:
            assert (adv[~valid] == 0).all() and (vt[~valid] == 0).all()
        a = adv.double()[sel]
        m, m2 = a.mean(), (a * a).mean()
        sd = a.std(unbiased=False)
        deep = (T + 40) * 2.0 ** -53
        _check(case, "mean", stats[0], m, U * m.abs() + deep * a.abs().mean())
        var_err = 4 * deep * (m2 + m * m)
        _check(case, "std", stats[1], sd,
               U * sd + torch.minimum(var_err.sqrt(), var_err / (2 * sd).clamp_min(1e-300)))


# ---------------------------------------------------------------------------
# PPO loss
# ---------------------------------------------------------------------------
CLIP_EPS, VALUE_COEF, ENTROPY_COEF = 0.15, float(np.float32(0.7)), float(np.float32(0.013))


def _ppo_inputs(M, seed, with_stats):
    T, E = (2048, 256) if M == 2048 * 256 else (1, M)
    reward, nonterminal, v_, v_next, cut, _ = _rollout(T, E, seed, False)
    adv, _, stats = gae(reward, nonterminal, v_, v_next, cut, 0.99, 0.95)
    adv = adv.reshape(-1).clone()
    g = _gen(seed + 1)
    lp_old = 0.5 * torch.randn(M, device="cuda", generator=g) - 1
    lp = lp_old + 0.3 * torch.randn(M, device="cuda", generator=g)
    ent = torch.rand(M, device="cuda", generator=g)
    v_old = torch.randn(M, device="cuda", generator=g)
    v = v_old + 0.3 * torch.randn(M, device="cuda", generator=g)
    vt = torch.randn(M, device="cuda", generator=g)
    eps = np.float32(CLIP_EPS)
    ratio = torch.exp(lp - lp_old)
    near = ((ratio - float(np.float32(1) - eps)).abs() < 1e-5) | (
        (ratio - float(np.float32(1) + eps)).abs() < 1e-5)
    lp[near] = lp_old[near]
    # planted rows: lp == lp_old, v == v_old, v on either value clip bound, adv = 0
    # (after standardisation when stats are given)
    i = torch.arange(M, device="cuda")
    lp[i % 8 == 0] = lp_old[i % 8 == 0]
    v[i % 8 == 1] = v_old[i % 8 == 1]
    v[i % 16 == 2] = v_old[i % 16 == 2] - float(np.float32(0.2))
    v[i % 16 == 3] = v_old[i % 16 == 3] + float(np.float32(0.2))
    adv[i % 16 == 4] = stats[0] if with_stats else 0.0
    return lp, ent, v, lp_old, v_old, adv, vt, (stats if with_stats else None)


@pytest.mark.parametrize("M", [1, 64, 255, 256, 257, 2048, 524288])
def test_ppo_loss_vs_fp64(M):
    for clip_vf in (None, 0.2):
        for with_stats in (False, True):
            case = "ppo M=%d vf=%s stats=%d" % (M, clip_vf, with_stats)
            lp, ent, v, lp_old, v_old, adv, vt, stats = _ppo_inputs(M, M, with_stats)
            ins = [x.clone().requires_grad_(True) for x in (lp, ent, v)]
            total, parts = ppo_loss(ins[0], ins[1], ins[2], lp_old, v_old, adv, vt, stats,
                                    CLIP_EPS, clip_vf, VALUE_COEF, ENTROPY_COEF)
            grads = torch.autograd.grad(GL * total, ins)
            ins64 = [_leaf(x) for x in (lp, ent, v)]
            ref = R.ppo_loss(ins64[0], ins64[1], ins64[2], lp_old, v_old, adv, vt, stats,
                             CLIP_EPS, clip_vf, VALUE_COEF, ENTROPY_COEF)
            grads64 = torch.autograd.grad(GL * ref[0], ins64)

            x = (lp.double() - lp_old.double()).abs()
            a = adv.double()
            if stats is not None:
                a = (a - stats[0].double()) / (stats[1].double() + R.PPO_STD_EPS)
            ra = (torch.exp(lp.double() - lp_old.double()) * a).abs()
            b_p = U * ((x + 9) * ra).sum() / M + U * ref[1].detach().abs()
            d = (v.double() - vt.double()).abs()
            if clip_vf is None:
                dc = d
            else:
                lo = (v_old - float(np.float32(clip_vf))).double()
                hi = (v_old + float(np.float32(clip_vf))).double()
                dc = (torch.min(torch.max(v.double(), lo), hi) - vt.double()).abs()
            b_v = 3 * U * torch.max(d * d, dc * dc).sum() / M + U * ref[2].detach().abs()
            b_e = 2 * U * ref[3].detach().abs()
            b_t = (b_p + VALUE_COEF * b_v + ENTROPY_COEF * b_e +
                   3 * U * (ref[1].abs() + VALUE_COEF * ref[2].abs() +
                            ENTROPY_COEF * ref[3].abs()).detach())
            for k, (name, b) in enumerate([("total", b_t), ("policy", b_p), ("value", b_v),
                                           ("entropy", b_e)]):
                _check(case, name, parts[k], ref[k], b)
            _check(case, "total'", total, ref[0], b_t)
            _check(case, "g_lp", grads[0], grads64[0], U * (x + 11) * grads64[0].abs())
            _check(case, "g_ent", grads[1], grads64[1], 4 * U * grads64[1].abs())
            _check(case, "g_v", grads[2], grads64[2],
                   8 * U * GL * VALUE_COEF / M * 2 * (d + dc))


# ---------------------------------------------------------------------------
# determinism, CUDA graphs, concurrent streams, converted inputs
# ---------------------------------------------------------------------------
def _run_td(q, *rest):
    qk = q.detach().clone().requires_grad_(True)
    loss, delta, _, _ = td_loss(qk, *rest)
    return loss, delta, _grad(loss, qk)


def _run_c51(y, *rest):
    yk = y.detach().clone().requires_grad_(True)
    loss, delta = c51_loss(yk, *rest)
    return loss, delta, _grad(loss, yk)


def _run_qh(y, *rest):
    yk = y.detach().clone().requires_grad_(True)
    loss, err = quantile_huber_loss(yk, *rest)
    return loss, err, _grad(loss, yk)


def _run_ppo(lp, ent, v, *rest):
    ins = [x.detach().clone().requires_grad_(True) for x in (lp, ent, v)]
    total, parts = ppo_loss(*ins, *rest)
    return (parts,) + torch.autograd.grad(GL * total, ins)


def _run_gae(*args):
    return gae(*args)


def _cases():
    td = _td_inputs(4097, 18, 1)
    c51 = _c51_inputs(4097, 51, "linspace", 2)
    g = _gen(3)
    qh = (torch.randn(512, 64, device="cuda", generator=g),
          torch.randn(512, 64, device="cuda", generator=g),
          torch.rand(512, 64, device="cuda", generator=g),
          torch.rand(512, device="cuda", generator=g))
    ppo = _ppo_inputs(524288, 4, True)
    roll = _rollout(2048, 256, 5, True)
    return [
        ("td", _run_td, td + (True, True)),
        ("c51", _run_c51, c51[:6] + (None, None, True, c51[6])),
        ("qh", _run_qh, qh + (True,)),
        ("ppo", _run_ppo, ppo + (CLIP_EPS, 0.2, VALUE_COEF, ENTROPY_COEF)),
        ("gae", _run_gae, roll[:5] + (0.99, 0.95, roll[5])),
    ]


def _same(a, b):
    return all(torch.equal(x, y) for x, y in zip(a, b))


def test_identical_calls_are_bit_identical():
    for name, run, args in _cases():
        first = run(*args)
        torch.cuda.synchronize()
        assert _same(first, run(*args)), name


def test_cuda_graph_replay_matches_eager():
    """Captured the way DQN / PPO capture their update: the ticket of each reduction
    is fixed at capture and reused on every replay."""
    cases = {name: (run, args) for name, run, args in _cases() if name in ("td", "c51", "ppo")}
    for name, (run, args) in cases.items():
        static = [a.clone() if torch.is_tensor(a) else a for a in args]
        B = args[0].shape[0]
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            run(*static)
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            out = run(*static)
        for k in range(3):
            g = _gen(100 + k)
            with torch.no_grad():
                for s, a in zip(static, args):
                    if torch.is_tensor(s) and s.is_floating_point() and s.shape[0] == B:
                        s.copy_(a * (1 + 0.1 * torch.rand(a.shape, device="cuda", generator=g)))
            graph.replay()
            torch.cuda.synchronize()
            assert _same(out, run(*[s.clone() if torch.is_tensor(s) else s for s in static])), \
                (name, k)


def test_concurrent_streams_match_eager():
    """Two batches of every reduction kernel in flight on two streams at once."""
    a, b = _cases(), _cases()
    for (_, _, args) in b:  # a second, different batch of the same shapes
        for x in args:
            if torch.is_tensor(x) and x.is_floating_point() and x.numel() > 2:
                x.mul_(1.25)
    eager = [(run(*x1), run(*x2)) for (_, run, x1), (_, _, x2) in zip(a, b)]
    torch.cuda.synchronize()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    s1.wait_stream(torch.cuda.current_stream())
    s2.wait_stream(torch.cuda.current_stream())
    outs = []
    for (_, run, x1), (_, _, x2) in zip(a, b):
        with torch.cuda.stream(s1):
            o1 = run(*x1)
        with torch.cuda.stream(s2):
            o2 = run(*x2)
        outs.append((o1, o2))
    torch.cuda.synchronize()
    for (name, _, _), (e1, e2), (o1, o2) in zip(a, eager, outs):
        assert _same(e1, o1) and _same(e2, o2), name


def _strided(x):
    """The same values behind a non-contiguous view."""
    w = torch.zeros(*x.shape, 2, dtype=x.dtype, device=x.device)
    w[..., 1] = x
    return w[..., 1]


def _widen(x):
    return _strided(x.double())


def test_converted_inputs_match_fp32_contiguous():
    """fp64, bool and strided inputs give the bits of the fp32 contiguous call."""
    q, action, next_q, reward, discount, terminal, weights = _td_inputs(999, 18, 7)
    ref = _run_td(q, action, next_q, reward, discount, terminal, weights)
    got = _run_td(q, action, _widen(next_q), reward.double(), discount.double(),
                  terminal.bool(), _widen(weights))
    assert _same(ref, got)

    y, next_p, reward, discount, terminal, weights, z = _c51_inputs(300, 51, "linspace", 8)
    ref = _run_c51(y, next_p, reward, discount, terminal, weights, None, None, True, z)
    got = _run_c51(y, _widen(next_p), reward.double(), _widen(discount),
                   terminal.to(torch.uint8), weights.double(), None, None, True, z.double())
    assert _same(ref, got)

    g = _gen(9)
    yq, tq, tau, wq = (torch.randn(40, 16, device="cuda", generator=g),
                       torch.randn(40, 12, device="cuda", generator=g),
                       torch.rand(40, 16, device="cuda", generator=g),
                       torch.rand(40, device="cuda", generator=g))
    assert _same(_run_qh(yq, tq, tau, wq, True),
                 _run_qh(_widen(yq), tq.double(), _widen(tau), wq.double(), True))

    reward, nonterminal, v, v_next, cut, valid = _rollout(64, 300, 10, True)
    ref = gae(reward, nonterminal, v, v_next, cut, 0.99, 0.95, valid)
    got = gae(reward.double(), nonterminal.double(), _widen(v), _widen(v_next), _strided(cut),
              0.99, 0.95, valid.to(torch.uint8))
    assert _same(ref, got)

    lp, ent, v, lp_old, v_old, adv, vt, stats = _ppo_inputs(3000, 11, True)
    ref = _run_ppo(lp, ent, v, lp_old, v_old, adv, vt, stats, CLIP_EPS, 0.2, VALUE_COEF,
                   ENTROPY_COEF)
    got = _run_ppo(lp, ent, v, lp_old.double(), _widen(v_old), adv.double(), _widen(vt),
                   stats.double(), CLIP_EPS, 0.2, VALUE_COEF, ENTROPY_COEF)
    assert _same(ref, got)
