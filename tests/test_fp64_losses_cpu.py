"""CPU: the fp64 restatements in tests/fp64_losses.py (the reference side of
test_loss_kernels_fp64_gpu.py) against the real reference's own fp32 outputs
(tests/golden/losses.npz), at the tolerances test_losses_gpu.py holds the kernels to."""
import os

import numpy as np
import pytest
import torch

import fp64_losses as R

G = np.load(os.path.join(os.path.dirname(__file__), "golden", "losses.npz"))
TOL = dict(rtol=1e-5, atol=1e-6)


def t64(x):
    return torch.as_tensor(np.asarray(x)).double()


def leaf(x):
    return t64(x).requires_grad_(True)


@pytest.mark.parametrize("clip", [True, False])
@pytest.mark.parametrize("acc", ["mean", "sum"])
@pytest.mark.parametrize("use_w", [True, False])
def test_td_loss(clip, acc, use_w):
    q = leaf(G["td_q"])
    loss, delta, _, _ = R.td_loss(q, G["td_action"], G["td_next_q"], G["td_reward"],
                                  G["td_discount"], G["td_terminal"],
                                  G["td_weights"] if use_w else None, clip, acc == "mean")
    key = "td_%d_%s_%d" % (clip, acc, use_w)
    np.testing.assert_allclose(loss.item(), G[key + "_loss"], **TOL)
    np.testing.assert_allclose(delta.detach().numpy(), G["td_delta"], **TOL)
    loss.backward()
    np.testing.assert_allclose(q.grad.numpy(), G[key + "_grad"], **TOL)


def test_projection():
    z = G["proj_z"]
    Tz = (np.float32(0.1) + np.float32(0.9) * z).astype(np.float32)[None]
    from oracle.losses import categorical_projection

    np.testing.assert_allclose(R.categorical_projection(Tz, G["proj_p"], z).numpy(),
                               categorical_projection(Tz, G["proj_p"], z), rtol=1e-6, atol=1e-7)


@pytest.mark.parametrize("acc", ["mean", "sum"])
@pytest.mark.parametrize("use_w", [True, False])
def test_c51_loss(acc, use_w):
    y = leaf(G["c51_y"])
    loss, delta, t = R.c51_loss(y, G["c51_next_p"], G["c51_reward"], G["c51_discount"],
                                G["c51_terminal"], G["c51_weights"] if use_w else None,
                                G["c51_z"], acc == "mean")
    key = "c51_%s_%d" % (acc, use_w)
    # the reference's fp32 bj = (Tz - v_min) / delta_z carries ~2^-24 * (|Tz| + |v_min|) /
    # delta_z ~ 1e-6 absolute with this support; the fp64 target does not, so the target
    # is held to that (the kernel, which rounds like the reference, meets atol=1e-7)
    np.testing.assert_allclose(t.numpy(), G["c51_target"], rtol=1e-5, atol=2e-6)
    np.testing.assert_allclose(delta.detach().numpy(), G["c51_delta"], **TOL)
    np.testing.assert_allclose(loss.item(), G[key + "_loss"], **TOL)
    loss.backward()
    # d/dy = -scale * t / y: the target's 2e-6 becomes 2e-6 * scale / y
    yv = G["c51_y"].astype(np.float64)
    scale = (G["c51_weights"] if use_w else np.ones(len(yv)))[:, None] / (
        len(yv) if acc == "mean" else 1)
    want = G[key + "_grad"].astype(np.float64)
    ratio = np.abs(y.grad.numpy() - want) / (1e-7 + 1e-5 * np.abs(want) + 2e-6 * scale / yv)
    assert ratio.max() <= 1, ratio.max()


@pytest.mark.parametrize("acc", ["mean", "sum"])
@pytest.mark.parametrize("use_w", [True, False])
def test_quantile_huber(acc, use_w):
    y = leaf(G["qh_y"])
    loss, err = R.quantile_huber(y, G["qh_t"], G["qh_taus"], G["qh_weights"] if use_w else None,
                                 acc == "mean")
    key = "qh_%s_%d" % (acc, use_w)
    np.testing.assert_allclose(loss.item(), G[key + "_loss"], **TOL)
    np.testing.assert_allclose(err.detach().numpy(), G["qh_delta"], **TOL)
    loss.backward()
    np.testing.assert_allclose(y.grad.numpy(), G[key + "_grad"], rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize("tag", ["a", "b", "c"])
def test_gae(tag):
    gamma, lambd = [float(x) for x in G["gae_%s_params" % tag]]
    adv, vt, mag = R.gae(G["gae_reward"], G["gae_nonterminal"], G["gae_v"], G["gae_v_next"],
                         G["gae_cut"], gamma, lambd)
    np.testing.assert_allclose(adv.numpy(), G["gae_%s_adv" % tag], rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(vt.numpy(), G["gae_%s_vt" % tag], rtol=1e-12, atol=1e-12)
    assert (mag >= adv.abs()).all()


def test_gae_valid_mask_ends_segment():
    """An invalid slot holds nothing and cuts the segment before it."""
    T, E = 6, 1
    r = np.arange(1, T + 1, dtype=np.float64)[:, None]
    zeros = np.zeros((T, E))
    valid = np.ones((T, E), bool)
    valid[3] = False
    cut = np.zeros((T, E), bool)
    cut[-1] = True
    adv, vt, _ = R.gae(r, np.ones((T, E)), zeros, zeros, cut, 0.5, 1.0, valid)
    want = np.zeros(T)
    for lo, hi in ((0, 3), (4, 6)):  # two segments: [0, 3) and [4, 6)
        acc = 0.0
        for t in range(hi - 1, lo - 1, -1):
            acc = r[t, 0] + 0.5 * acc
            want[t] = acc
    np.testing.assert_array_equal(adv.numpy()[:, 0], want)
    np.testing.assert_array_equal(vt.numpy()[:, 0], want)


@pytest.mark.parametrize("tag,clip_vf", [("a", None), ("b", 0.2)])
def test_ppo_loss(tag, clip_vf):
    lp, ent, v = leaf(G["ppo_lp"]), leaf(G["ppo_ent"]), leaf(G["ppo_v"])
    total, policy, value, _ = R.ppo_loss(lp, ent, v, G["ppo_lp_old"], G["ppo_v_old"],
                                         G["ppo_adv"], G["ppo_vt"], G["ppo_mean_std"], 0.2,
                                         clip_vf, 0.5, 0.01)
    np.testing.assert_allclose(total.item(), G["ppo_%s_loss" % tag], **TOL)
    np.testing.assert_allclose(policy.item(), G["ppo_%s_policy" % tag], **TOL)
    np.testing.assert_allclose(value.item(), G["ppo_%s_value" % tag], **TOL)
    total.backward()
    np.testing.assert_allclose(lp.grad.numpy(), G["ppo_%s_g_lp" % tag], rtol=1e-4, atol=1e-7)
    np.testing.assert_allclose(ent.grad.numpy(), G["ppo_%s_g_ent" % tag], rtol=1e-5, atol=1e-9)
    np.testing.assert_allclose(v.grad.numpy(), G["ppo_%s_g_v" % tag], rtol=1e-4, atol=1e-7)


def test_ppo_value_clip_boundary_follows_autograd():
    """At v == v_old -+ clip_eps_vf (in fp32) the value gradient is the one autograd
    gives the reference's fp32 formula: half through each side of the max / min ties."""
    vo = torch.tensor([0.3, 0.3, 0.3, 0.3])
    v32 = torch.stack([vo[0] - 0.2, vo[1] + 0.2, vo[2], vo[3] + 0.1])
    vt = torch.tensor([0.9, -0.5, 0.3, -2.0])
    zeros = torch.zeros(4)

    v = v32.double().requires_grad_(True)
    R.ppo_loss(zeros, zeros, v, zeros, vo, zeros, vt, None, 0.2, 0.2, 1.0, 0.0)[2].backward()

    w = v32.clone().requires_grad_(True)  # the reference's own expression, in fp32
    vc = torch.min(torch.max(w, vo - 0.2), vo + 0.2)
    torch.mean(torch.max((w - vt) ** 2, (vc - vt) ** 2)).backward()
    np.testing.assert_allclose(v.grad.numpy(), w.grad.double().numpy(), rtol=1e-6)
