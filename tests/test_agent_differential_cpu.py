"""Randomised differential tests of PPO, A2C and the DQN family against the REAL reference:
scripted random observations / rewards with random `done` and `reset` patterns over several
environments, so that episode segmentation, the flush of unfinished episodes at update time,
the dataset order that fixes what ``random.sample`` draws, GAE, advantage standardisation, the
value-clipped loss and the normaliser all have to agree.  Both agents sample their actions
from torch's global generator; statistics are compared after every step and the parameters at
the end.

The reference's side of every scenario is tests/golden/ref_agent_differential.npz, recorded by
oracle/gen_golden_differential.py running the `_run_*` functions below with lib = pfrl."""
import os
import random
import sys
from unittest import mock

import numpy as np
import pytest
import torch
from torch import nn

sys.path.insert(0, os.path.dirname(__file__))
from fake_store import OracleBackedStore  # noqa: E402

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _golden(key):
    """(actions, statistics, parameters) the reference recorded for scenario `key`."""
    g = np.load(os.path.join(GOLD, "ref_agent_differential.npz"))
    params = [g["%s_param%d" % (key, i)] for i in range(int(g[key + "_n_params"]))]
    return g[key + "_actions"], g[key + "_stats"], params


def _is_reference(lib):
    return lib.__name__ == "pfrl"


def _agent(lib, n_envs, seed, **kw):
    torch.manual_seed(seed)
    model = nn.Sequential(nn.Linear(6, 24), nn.Tanh(), lib.nn.Branched(
        nn.Sequential(nn.Linear(24, 3), lib.policies.SoftmaxCategoricalHead()), nn.Linear(24, 1)))
    return model, lib.agents.PPO(
        model, torch.optim.Adam(model.parameters(), lr=2e-3),
        obs_normalizer=lib.nn.EmpiricalNormalization(6, clip_threshold=5), gamma=0.9,
        phi=lambda x: x.astype(np.float32, copy=False), update_interval=48, minibatch_size=16,
        epochs=2, **kw)


def _run_ppo(lib, seed):
    n_envs = 1 + seed % 3
    kw = [dict(lambd=0.95, clip_eps_vf=None, standardize_advantages=True, entropy_coef=0.01),
          dict(lambd=0.8, clip_eps_vf=0.2, standardize_advantages=False, entropy_coef=0.0,
               max_grad_norm=0.5, value_func_coef=0.5)][seed % 2]
    rng = np.random.RandomState(seed)
    T = 160
    obs = rng.randn(T + 1, n_envs, 6).astype(np.float32)
    rew = rng.randn(T, n_envs)
    done = rng.rand(T, n_envs) < 0.08
    reset = (rng.rand(T, n_envs) < 0.05) & ~done
    model, agent = _agent(lib, n_envs, 100 + seed, **kw)
    torch.manual_seed(7)
    random.seed(7)
    np.random.seed(7)
    cur = [obs[0, i] for i in range(n_envs)]
    acts, stats = [], []
    for t in range(T):
        a = np.asarray(agent.batch_act(cur))
        acts.append(a.copy())
        nxt = [obs[t + 1, i] for i in range(n_envs)]
        agent.batch_observe(nxt, list(rew[t]), list(done[t]), list(reset[t]))
        # an env that ended starts its next episode from a fresh observation
        cur = [obs[t + 1, i] * (-1.0 if (done[t, i] or reset[t, i]) else 1.0)
               for i in range(n_envs)]
        stats.append([float(v) for _, v in agent.get_statistics()])
    return np.asarray(acts), np.asarray(stats), [p.detach().numpy().copy()
                                                 for p in model.parameters()]


@pytest.mark.parametrize("seed", range(6))
def test_ppo_random_done_reset_patterns(seed):
    import pfrl_b200

    a_ref, s_ref, p_ref = _golden("ppo%d" % seed)
    a_me, s_me, p_me = _run_ppo(pfrl_b200, seed)
    assert np.array_equal(a_ref, a_me)
    both_nan = np.isnan(s_ref) & np.isnan(s_me)
    np.testing.assert_allclose(np.where(both_nan, 0, s_me), np.where(both_nan, 0, s_ref),
                               rtol=5e-5, atol=1e-6)
    assert len(p_ref) == len(p_me)
    for x, y in zip(p_ref, p_me):
        np.testing.assert_allclose(y, x, rtol=1e-5, atol=2e-6)
    assert s_ref[-1][4] >= 3          # n_updates: several updates happened


def _run_a2c(lib, seed):
    n_envs = 2 + seed
    rng = np.random.RandomState(50 + seed)
    T = 90
    obs = rng.randn(T + 1, n_envs, 6).astype(np.float32)
    rew = rng.randn(T, n_envs)
    done = rng.rand(T, n_envs) < 0.1
    torch.manual_seed(200 + seed)
    model = nn.Sequential(nn.Linear(6, 16), nn.Tanh(), lib.nn.Branched(
        nn.Sequential(nn.Linear(16, 3), lib.policies.SoftmaxCategoricalHead()),
        nn.Linear(16, 1)))
    agent = lib.agents.A2C(
        model, torch.optim.RMSprop(model.parameters(), lr=3e-3, eps=1e-5), gamma=0.95,
        num_processes=n_envs, update_steps=3 + seed, use_gae=bool(seed % 2), tau=0.9,
        max_grad_norm=[None, 0.5][seed % 2], average_actor_loss_decay=0.5,
        average_entropy_decay=0.5, average_value_decay=0.5,
        phi=lambda x: x.astype(np.float32, copy=False))
    torch.manual_seed(9)
    acts, stats = [], []
    for t in range(T):
        acts.append(np.asarray(agent.batch_act(list(obs[t]))).copy())
        agent.batch_observe(list(obs[t + 1]), list(rew[t]), list(done[t]), [False] * n_envs)
        stats.append([float(v) for _, v in agent.get_statistics()])
    return np.asarray(acts), np.asarray(stats), [p.detach().numpy().copy()
                                                 for p in model.parameters()]


@pytest.mark.parametrize("seed", range(4))
def test_a2c_random_done_patterns(seed):
    import pfrl_b200

    a_ref, s_ref, p_ref = _golden("a2c%d" % seed)
    a_me, s_me, p_me = _run_a2c(pfrl_b200, seed)
    assert np.array_equal(a_ref, a_me)
    np.testing.assert_allclose(s_me, s_ref, rtol=5e-5, atol=1e-6)
    assert len(p_ref) == len(p_me)
    for x, y in zip(p_ref, p_me):
        np.testing.assert_allclose(y, x, rtol=1e-5, atol=2e-6)


def _run_dqn_family(lib, kind):
    from oracle.gen_golden_losses import TRACE_PER, _make_trace_agent

    n_envs, T = 3, 120
    rng = np.random.RandomState(len(kind))
    obs = rng.randn(T + 1, n_envs, 5).astype(np.float32)
    rew = rng.randn(T, n_envs)
    done = rng.rand(T, n_envs) < 0.1
    reset = (rng.rand(T, n_envs) < 0.07) & ~done
    with mock.patch("pfrl_b200.replay_buffers.device_buffer.DeviceReplayStore", OracleBackedStore):
        if _is_reference(lib):
            rbuf = lib.replay_buffers.PrioritizedReplayBuffer(100, **TRACE_PER)
            raw = rbuf.update_errors
            rbuf.update_errors = lambda e, raw=raw: raw([float(x) for x in e])
        else:
            rbuf = lib.replay_buffers.PrioritizedReplayBuffer(100, device=0, **TRACE_PER)
        torch.manual_seed(5)
        q, agent = _make_trace_agent(lib, kind, rbuf)
        np.random.seed(6)
        torch.manual_seed(6)
        cur = [obs[0, i] for i in range(n_envs)]
        acts, stats = [], []
        for t in range(T):
            a = [int(x) for x in agent.batch_act(cur)]
            acts.append(a)
            agent.batch_observe([obs[t + 1, i] for i in range(n_envs)], list(rew[t]),
                                list(done[t]), list(reset[t]))
            cur = [obs[t + 1, i] * (-1.0 if (done[t, i] or reset[t, i]) else 1.0)
                   for i in range(n_envs)]
            st = dict(agent.get_statistics())
            stats.append([st["average_q"], st["average_loss"], st["n_updates"], st["rlen"]])
    return (np.asarray(acts, dtype=np.int64), np.asarray(stats, dtype=np.float64),
            [p.detach().numpy().copy() for p in q.parameters()])


@pytest.mark.parametrize("kind", ["ddqn", "rainbow", "c51"])
def test_dqn_family_random_done_reset_patterns(kind):
    """DoubleDQN / Rainbow / C51 + 3-step prioritised replay (device buffer over the
    host store emulation) on scripted random transitions of three environments with
    random terminals AND random non-terminal resets."""
    import pfrl_b200

    a_ref, s_ref, p_ref = _golden(kind)
    a_me, s_me, p_me = _run_dqn_family(pfrl_b200, kind)
    assert np.array_equal(a_ref, a_me)
    assert np.array_equal(s_ref[:, 2:], s_me[:, 2:])
    live = s_ref[:, 2] > 0
    np.testing.assert_allclose(s_me[live, :2], s_ref[live, :2], rtol=5e-5, atol=1e-6)
    assert len(p_ref) == len(p_me)
    for x, y in zip(p_ref, p_me):
        np.testing.assert_allclose(y, x, rtol=1e-5, atol=2e-6)


def _run_uniform_replay_agent(lib, kind):
    from oracle.gen_golden_losses import _make_more_agent, _module_attrs

    n_envs, T = 2, 110
    rng = np.random.RandomState(len(kind) + 40)
    obs = rng.randn(T + 1, n_envs, 5).astype(np.float32)
    rew = rng.randn(T, n_envs)
    done = rng.rand(T, n_envs) < 0.1
    reset = (rng.rand(T, n_envs) < 0.07) & ~done
    with mock.patch("pfrl_b200.replay_buffers.device_buffer.DeviceReplayStore", OracleBackedStore):
        rbuf = lib.replay_buffers.ReplayBuffer(90) if _is_reference(lib) else \
            lib.replay_buffers.ReplayBuffer(90, device=0)
        torch.manual_seed(21)
        agent = _make_more_agent(lib, kind, rbuf)
        np.random.seed(22)
        torch.manual_seed(22)
        cur = [obs[0, i] for i in range(n_envs)]
        acts, stats = [], []
        for t in range(T):
            acts.append(np.asarray(agent.batch_act(cur), dtype=np.float64).copy())
            agent.batch_observe([obs[t + 1, i] for i in range(n_envs)], list(rew[t]),
                                list(done[t]), list(reset[t]))
            cur = [obs[t + 1, i] * (-1.0 if (done[t, i] or reset[t, i]) else 1.0)
                   for i in range(n_envs)]
            stats.append([float(v) for _, v in agent.get_statistics()])
        params = [p.detach().numpy().copy() for _, m in _module_attrs(agent)
                  for p in m.parameters()]
    return np.asarray(acts), np.asarray(stats), params


@pytest.mark.parametrize("kind", ["sac", "td3", "ddpg", "iqn"])
def test_uniform_replay_agents_random_done_reset_patterns(kind):
    """SAC / TD3 / DDPG / IQN on the uniform device buffer (host store emulation) with
    scripted random transitions, random terminals and random non-terminal resets."""
    import pfrl_b200

    a_ref, s_ref, p_ref = _golden(kind)
    a_me, s_me, p_me = _run_uniform_replay_agent(pfrl_b200, kind)
    np.testing.assert_allclose(a_me, a_ref, rtol=1e-5, atol=2e-6)
    both_nan = np.isnan(s_ref) & np.isnan(s_me)
    np.testing.assert_allclose(np.where(both_nan, 0, s_me), np.where(both_nan, 0, s_ref),
                               rtol=5e-5, atol=2e-6)
    assert len(p_ref) == len(p_me)
    for x, y in zip(p_ref, p_me):
        np.testing.assert_allclose(y, x, rtol=1e-5, atol=2e-6)
