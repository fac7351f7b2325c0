"""CPU: remaining host-side pieces of the path -- EmpiricalNormalization vs
the reference (golden), the Evaluator / train_agent_batch_with_evaluation
flow, explorers' RNG stream, sample_n_k's stream, batch_experiences on lists."""
import os

import numpy as np
import torch

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def test_empirical_normalization_matches_reference_golden():
    from pfrl_b200.nn import EmpiricalNormalization

    g = np.load(os.path.join(GOLD, "empirical_normalization.npz"))
    en = EmpiricalNormalization(7, clip_threshold=5)
    for i in range(4):
        y = en(torch.tensor(g["x%d" % i]), update=True).numpy()
        np.testing.assert_allclose(y, g["y%d" % i], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(en.mean.numpy(), g["mean"], rtol=1e-6, atol=1e-7)
    np.testing.assert_allclose(en.std.numpy(), g["std"], rtol=1e-6)
    assert int(en.count) == int(g["count"])
    out = en(torch.tensor(g["probe"]), update=False).numpy()
    np.testing.assert_allclose(out, g["probe_out"], rtol=1e-5, atol=1e-6)


def test_sample_n_k_consumes_the_reference_stream():
    """Same draws as pfrl/utils/random.py for both branches (k << n and 3k >= n)."""
    from oracle.replay import sample_n_k as oracle_sample
    from pfrl_b200.utils.random import sample_n_k

    for n, k in ((1000, 10), (1000, 400), (50, 50), (10 ** 6, 1024), (7, 0)):
        np.random.seed(n + k)
        a = sample_n_k(n, k)
        sa = np.random.get_state()[1][:5].copy()
        np.random.seed(n + k)
        b = oracle_sample(n, k)
        sb = np.random.get_state()[1][:5].copy()
        assert np.array_equal(a, b) and np.array_equal(sa, sb)
        assert len(set(a.tolist())) == k


def test_epsilon_greedy_uses_one_global_draw_per_decision():
    from pfrl_b200 import explorers

    ex = explorers.LinearDecayEpsilonGreedy(1.0, 0.1, 100, lambda: 7)
    np.random.seed(0)
    ref = np.random.RandomState(0)
    for t in (0, 10, 50, 100, 500):
        eps = ex.compute_epsilon(t)
        expect = 7 if ref.rand() < eps else 3
        assert ex.select_action(t, lambda: 3) == expect
    assert ex.compute_epsilon(1000) == 0.1 and abs(ex.compute_epsilon(50) - 0.55) < 1e-12


def test_batch_experiences_known_answer_on_lists():
    """The reference's KAT (tests/replay_buffers_test/test_replay_buffer.py:803-864):
    terminal flags, gamma ** len, last next_state."""
    from pfrl_b200.replay_buffer import batch_experiences

    def tr(s, r, term):
        return dict(state=np.float32([s]), action=s, reward=r, next_state=np.float32([s + 1]),
                    next_action=None, is_state_terminal=term)

    exps = [[tr(0, 1.0, False), tr(1, 2.0, False), tr(2, 4.0, True)], [tr(5, -1.0, False)]]
    b = batch_experiences(exps, torch.device("cpu"), lambda x: x, 0.5)
    assert b["state"].tolist() == [[0.0], [5.0]] and b["next_state"].tolist() == [[3.0], [6.0]]
    assert b["reward"].tolist() == [1.0 + 0.5 * 2.0 + 0.25 * 4.0, -1.0]
    assert b["discount"].tolist() == [0.125, 0.5]
    assert b["is_state_terminal"].tolist() == [1.0, 0.0]
    assert b["action"].tolist() == [0, 5] and "next_action" not in b


def test_train_agent_batch_with_evaluation_writes_scores(tmp_path):
    from pfrl_b200 import agents, experiments, explorers, q_functions
    from pfrl_b200.envs import ChainEnv, SerialVectorEnv
    from pfrl_b200.replay_buffers import HostReplayBuffer
    from pfrl_b200.utils import set_random_seed

    set_random_seed(0)
    q = q_functions.FCStateQFunctionWithDiscreteAction(5, 2, 16, 1)
    agent = agents.DoubleDQN(
        q, torch.optim.Adam(q.parameters(), lr=3e-3), HostReplayBuffer(2000), 0.95,
        explorers.ConstantEpsilonGreedy(0.3, lambda: np.random.randint(2)), replay_start_size=20,
        minibatch_size=8, target_update_interval=20,
        phi=lambda x: x.astype(np.float32, copy=False))
    env = SerialVectorEnv([ChainEnv(seed=i) for i in range(2)])
    eval_env = SerialVectorEnv([ChainEnv(seed=10 + i) for i in range(2)])
    agent2, history = experiments.train_agent_batch_with_evaluation(
        agent, env, steps=300, eval_n_steps=None, eval_n_episodes=4, eval_interval=100,
        outdir=str(tmp_path), eval_env=eval_env, max_episode_len=30)
    assert agent2 is agent and len(history) == 3
    rows = open(os.path.join(str(tmp_path), "scores.txt")).read().strip().split("\n")
    assert rows[0].split("\t")[:8] == ["steps", "episodes", "elapsed", "mean", "median", "stdev",
                                       "max", "min"]
    assert len(rows) == 4 and rows[0].split("\t")[8:] == [n for n, _ in agent.get_statistics()]
    assert os.path.isdir(os.path.join(str(tmp_path), "best"))
    assert os.path.isdir(os.path.join(str(tmp_path), "300_finish"))


def test_vector_frame_stack_shares_frame_objects():
    """reference: tests/wrappers_tests/test_vector_frame_stack.py (needs gym
    there); here: frames are shared between consecutive observations and a
    reset repeats the first frame k times."""
    from pfrl_b200.envs import SerialVectorEnv
    from pfrl_b200.wrappers import VectorFrameStack

    class ImgEnv:
        def __init__(self, seed):
            self.rng = np.random.RandomState(seed)
            self.t = 0

        def reset(self):
            self.t = 0
            return self.rng.randint(0, 256, size=(1, 6, 6)).astype(np.uint8)

        def step(self, a):
            self.t += 1
            return (self.rng.randint(0, 256, size=(1, 6, 6)).astype(np.uint8), 1.0, self.t == 5, {})

        def close(self):
            pass

    venv = VectorFrameStack(SerialVectorEnv([ImgEnv(i) for i in range(3)]), k=4)
    obs = venv.reset()
    assert len(obs) == 3 and np.asarray(obs[0]).shape == (4, 6, 6)
    assert all(f is obs[0]._frames[0] for f in obs[0]._frames)  # first frame repeated
    obs2, r, d, info = venv.step([0, 0, 0])
    assert obs2[1]._frames[:3] == obs[1]._frames[1:] or all(
        a is b for a, b in zip(obs2[1]._frames[:3], obs[1]._frames[1:]))
    assert obs2[1]._frames[3] is not obs[1]._frames[3]
    for _ in range(4):
        obs2, r, d, info = venv.step([0, 0, 0])
    assert all(d)
    obs3 = venv.reset(np.logical_not(d))
    assert all(f is obs3[2]._frames[0] for f in obs3[2]._frames)
    assert venv.num_envs == 3


EXPLORER_CASES = [
    ("ConstantEpsilonGreedy", (0.3, lambda: np.random.randint(4)), "discrete"),
    ("LinearDecayEpsilonGreedy", (1.0, 0.1, 20, lambda: np.random.randint(4)), "discrete"),
    ("ExponentialDecayEpsilonGreedy", (1.0, 0.05, 0.9, lambda: np.random.randint(4)), "discrete"),
    ("Boltzmann", (0.7,), "discrete"),
    ("Greedy", (), "discrete"),
    ("AdditiveGaussian", (0.3, -1, 1), "continuous"),
    ("AdditiveOU", (0.1, 0.2, 0.4), "continuous"),
]


def _explorer_trace(explorers, av_cls, name):
    """40 actions of explorer `name` from `explorers` (the reference's module or
    this package's), the position of numpy's global stream after them, and its repr."""
    (args, kind), = [(a, k) for n, a, k in EXPLORER_CASES if n == name]
    q = torch.tensor([[0.3, -0.2, 1.1, 0.4]])
    ex = getattr(explorers, name)(*args)
    np.random.seed(5)
    acts = []
    for t in range(40):
        if kind == "discrete":
            a = ex.select_action(t, lambda: 2, action_value=av_cls(q))
        else:
            a = ex.select_action(t, lambda: np.float32([0.2, -0.4]))
        acts.append(np.asarray(a, dtype=np.float64))
    return np.stack(acts), np.random.get_state()[1][:8].copy(), repr(ex)


def test_explorers_consume_the_reference_stream():
    """Every explorer against the real reference (tests/golden/ref_explorers.npz,
    oracle/gen_golden_differential.py): same actions, same position of numpy's
    global stream and the same repr."""
    from pfrl_b200 import action_value, explorers

    g = np.load(os.path.join(GOLD, "ref_explorers.npz"))
    for name, _, _ in EXPLORER_CASES:
        acts, stream, rep = _explorer_trace(explorers, action_value.DiscreteActionValue, name)
        np.testing.assert_array_equal(g[name + "_actions"], acts, err_msg=name)
        assert np.array_equal(g[name + "_stream"], stream), name
        assert str(g[name + "_repr"]) == rep, name


def test_linear_interpolation_hook():
    """reference: tests/experiments_tests/test_hooks.py (values at the ends,
    in between, and clamped outside [1, total_steps])."""
    from pfrl_b200.experiments import LinearInterpolationHook, StepHook

    seen = []
    hook = LinearInterpolationHook(11, 1.0, 0.0, lambda env, agent, v: seen.append((env, agent, v)))
    assert isinstance(hook, StepHook)
    for step in (0, 1, 2, 6, 11, 50):
        hook("env", "agent", step)
    assert [s[:2] for s in seen] == [("env", "agent")] * 6
    np.testing.assert_allclose([s[2] for s in seen], [1.0, 1.0, 0.9, 0.5, 0.0, 0.0], atol=1e-12)
