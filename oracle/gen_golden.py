"""Generate tests/golden/*.npz from the REAL reference (pfnet/pfrl).

TEST INFRASTRUCTURE ONLY.  Run in the build container (needs /root/reference):

    python oracle/gen_golden.py

Each fixture is a scripted trace (inputs) plus what the unmodified reference
produced for it (outputs).  The GPU box has no reference tree, so these files
are how `-m gpu` tests check the CUDA path against the reference itself, and
how `-m "not gpu"` tests pin the oracle.  numpy version matters for the
reference's scalar promotion (SURVEY.md section 7.1): generated with the numpy
printed below; all priorities are fed as Python floats (fp64).
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle.refimport import import_reference  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")

OP_APPEND, OP_STOP, OP_SAMPLE = 0, 1, 2


def make_state(sid, shape):
    """Deterministic uint8 observation for state id ``sid``."""
    n = int(np.prod(shape))
    return ((np.arange(n, dtype=np.int64) * 31 + sid * 17 + (sid * sid) % 251) % 256).astype(
        np.uint8).reshape(shape)


def gen_per_trace(name, seed, capacity, num_steps, n_envs, steps, batch, alpha, beta0,
                  betasteps, normalize_by_max, gamma, obs_shape=(4, 6, 6), lazy=False):
    import torch

    from pfrl.replay_buffer import batch_experiences
    from pfrl.replay_buffers import PrioritizedReplayBuffer
    from pfrl.wrappers.atari_wrappers import LazyFrames

    rng = np.random.RandomState(seed)
    rbuf = PrioritizedReplayBuffer(capacity, alpha=alpha, beta0=beta0, betasteps=betasteps,
                                   normalize_by_max=normalize_by_max, num_steps=num_steps)
    np.random.seed(seed)
    phi = lambda x: np.asarray(x, dtype=np.float32) / 255  # noqa: E731

    ops = []          # rows: op, env, sid, next_sid, action, terminal, n
    rewards = []      # per append
    errors = []       # per sample: list of floats
    out_idx, out_w, out_reward, out_disc, out_term, out_action = [], [], [], [], [], []
    out_state_sum, out_next_sum = [], []
    out_len = []
    frame_shape = (1,) + tuple(obs_shape[1:])
    k = obs_shape[0]
    next_sid = [1000 * (e + 1) for e in range(n_envs)]
    cur = {}
    frames = {}

    def obs_of(e, sid, reset=False):
        if not lazy:
            return make_state(sid, obs_shape)
        f = make_state(sid, frame_shape)
        if reset:
            frames[e] = [f] * k
        else:
            frames[e] = frames[e][1:] + [f]
        return LazyFrames(list(frames[e]), stack_axis=0)

    for e in range(n_envs):
        cur[e] = (next_sid[e], obs_of(e, next_sid[e], reset=True))
        next_sid[e] += 1
    for t in range(steps):
        for e in range(n_envs):
            sid, sobs = cur[e]
            nsid = next_sid[e]
            next_sid[e] += 1
            nobs = obs_of(e, nsid)
            action = int(rng.randint(0, 6))
            reward = float(rng.choice([-1.0, 0.0, 1.0, 0.5]))
            terminal = bool(rng.rand() < 0.06)
            rbuf.append(sobs, action, reward, nobs, None, terminal, env_id=e)
            ops.append((OP_APPEND, e, sid, nsid, action, int(terminal), 0))
            rewards.append(reward)
            reset = (not terminal) and rng.rand() < 0.03
            if terminal or reset:
                rbuf.stop_current_episode(env_id=e)
                ops.append((OP_STOP, e, 0, 0, 0, 0, 0))
                rsid = next_sid[e]
                next_sid[e] += 1
                cur[e] = (rsid, obs_of(e, rsid, reset=True))
            else:
                cur[e] = (nsid, nobs)
            out_len.append(len(rbuf))
            if len(rbuf) >= max(batch, 8) and rng.rand() < 0.35:
                n = int(min(batch, len(rbuf)))
                exps = rbuf.sample(n)
                ops.append((OP_SAMPLE, 0, 0, 0, 0, 0, n))
                out_idx.append(np.array(rbuf.memory.sampled_indices, dtype=np.int64))
                out_w.append(np.array([x[0]["weight"] for x in exps], dtype=np.float64))
                b = batch_experiences(exps, torch.device("cpu"), phi, gamma)
                out_reward.append(b["reward"].numpy())
                out_disc.append(b["discount"].numpy())
                out_term.append(b["is_state_terminal"].numpy())
                out_action.append(b["action"].numpy())
                out_state_sum.append(b["state"].numpy().reshape(n, -1).astype(np.float64).sum(1))
                out_next_sum.append(
                    b["next_state"].numpy().reshape(n, -1).astype(np.float64).sum(1))
                err = [float(x) for x in np.abs(rng.randn(n)) * 0.7]
                errors.append(np.array(err, dtype=np.float64))
                rbuf.update_errors(err)

    def ragged(lst, dtype):
        flat = np.concatenate(lst) if lst else np.zeros(0, dtype)
        return flat.astype(dtype)

    sizes = np.array([len(x) for x in out_idx], dtype=np.int64)
    np.savez_compressed(
        os.path.join(OUT, name + ".npz"),
        meta=np.array([seed, capacity, num_steps, n_envs, batch, int(lazy)], dtype=np.int64),
        params=np.array([alpha, beta0, betasteps, gamma], dtype=np.float64),
        normalize_by_max=np.array(str(normalize_by_max)),
        obs_shape=np.array(obs_shape, dtype=np.int64),
        ops=np.array(ops, dtype=np.int64), rewards=np.array(rewards, dtype=np.float64),
        sample_sizes=sizes, errors=ragged(errors, np.float64),
        idx=ragged(out_idx, np.int64), weight=ragged(out_w, np.float64),
        reward=ragged(out_reward, np.float32), discount=ragged(out_disc, np.float32),
        terminal=ragged(out_term, np.float32), action=ragged(out_action, np.int64),
        state_sum=ragged(out_state_sum, np.float64), next_sum=ragged(out_next_sum, np.float64),
        length=np.array(out_len, dtype=np.int64),
        final_max_priority=np.float64(rbuf.memory.max_priority),
        final_total=np.float64(rbuf.memory.priority_sums.sum()),
        final_min=np.float64(rbuf.memory.priority_mins.min()),
        numpy_version=np.array(np.__version__), reference_commit=np.array("c8cb332"),
    )
    print("wrote", name, "samples:", len(sizes), "draws:", int(sizes.sum()), "len:", len(rbuf))


def gen_uniform_trace(name, seed, capacity, num_steps, steps, batch, gamma):
    import torch
    from pfrl.replay_buffer import batch_experiences
    from pfrl.replay_buffers import ReplayBuffer

    rng = np.random.RandomState(seed)
    rbuf = ReplayBuffer(capacity, num_steps=num_steps)
    np.random.seed(seed)
    phi = lambda x: x  # noqa: E731
    obs = rng.randn(steps + 1, 17).astype(np.float32)
    acts = rng.randn(steps, 6).astype(np.float32)
    rews = rng.randn(steps)
    terms = rng.rand(steps) < 0.05
    out_state, out_next, out_action, out_reward, out_disc, out_term, sizes = [], [], [], [], [], [], []
    sample_at = []
    for t in range(steps):
        rbuf.append(obs[t], acts[t], float(rews[t]), obs[t + 1], None, bool(terms[t]))
        if terms[t]:
            rbuf.stop_current_episode()
        if len(rbuf) >= batch and t % 7 == 3:
            exps = rbuf.sample(batch)
            b = batch_experiences(exps, torch.device("cpu"), phi, gamma)
            sample_at.append(t)
            sizes.append(batch)
            out_state.append(b["state"].numpy())
            out_next.append(b["next_state"].numpy())
            out_action.append(b["action"].numpy())
            out_reward.append(b["reward"].numpy())
            out_disc.append(b["discount"].numpy())
            out_term.append(b["is_state_terminal"].numpy())
    np.savez_compressed(
        os.path.join(OUT, name + ".npz"),
        meta=np.array([seed, capacity, num_steps, steps, batch], dtype=np.int64),
        gamma=np.float64(gamma), obs=obs, acts=acts, rews=rews, terms=terms,
        sample_at=np.array(sample_at, dtype=np.int64),
        state=np.concatenate(out_state), next_state=np.concatenate(out_next),
        action=np.concatenate(out_action), reward=np.concatenate(out_reward),
        discount=np.concatenate(out_disc), terminal=np.concatenate(out_term),
        numpy_version=np.array(np.__version__),
    )
    print("wrote", name, "samples:", len(sizes))


def gen_reference_checkpoints():
    """replay_buffer.pkl files exactly as the reference writes them
    (replay_buffers/replay_buffer.py:85-87) plus what the reference says they
    hold: batch_experiences over every experience in queue order, leaf
    priorities, max_priority."""
    import torch

    from pfrl.replay_buffer import batch_experiences
    from pfrl.replay_buffers import PrioritizedReplayBuffer, ReplayBuffer
    from pfrl.wrappers.atari_wrappers import LazyFrames

    phi = lambda x: np.asarray(x, dtype=np.float32)  # noqa: E731
    cpu = torch.device("cpu")

    def expected(memory_items, gamma):
        b = batch_experiences(list(memory_items), cpu, phi, gamma)
        return {k: v.numpy() for k, v in b.items()}

    # uniform, 3-step, float32 vector observations, two interleaved env ids
    rng = np.random.RandomState(41)
    rbuf = ReplayBuffer(capacity=50, num_steps=3)
    obs = [rng.randn(4).astype(np.float32) for _ in range(2)]
    for t in range(90):
        e = t % 2
        nxt = rng.randn(4).astype(np.float32)
        done = rng.rand() < 0.12
        rbuf.append(obs[e], np.float32(rng.randn(2)), float(rng.randn()), nxt,
                    is_state_terminal=done, env_id=e)
        if done or rng.rand() < 0.05:
            rbuf.stop_current_episode(env_id=e)
            nxt = rng.randn(4).astype(np.float32)
        obs[e] = nxt
    rbuf.save(os.path.join(OUT, "ref_uniform_3step.pkl"))
    exp = expected(rbuf.memory, 0.9)
    np.savez_compressed(os.path.join(OUT, "ref_uniform_3step_expected.npz"),
                        n=len(rbuf), capacity=50, **exp)

    # prioritised, 1-step, LazyFrames uint8 observations sharing frames
    rng = np.random.RandomState(42)
    np.random.seed(42)
    rbuf = PrioritizedReplayBuffer(capacity=40, alpha=0.6, beta0=0.4, betasteps=100, num_steps=1)
    sid = 0

    def fresh():
        nonlocal sid
        sid += 1
        return make_state(sid, (1, 6, 6))

    frames = [fresh() for _ in range(4)]
    cur = LazyFrames(list(frames), stack_axis=0)
    for t in range(75):
        done = rng.rand() < 0.1
        frames = frames[1:] + [fresh()]
        nxt = LazyFrames(list(frames), stack_axis=0)
        rbuf.append(cur, int(rng.randint(6)), float(rng.choice([-1.0, 0.0, 1.0])), nxt,
                    is_state_terminal=done)
        cur = nxt
        if done:
            rbuf.stop_current_episode()
            frames = [fresh() for _ in range(4)]
            cur = LazyFrames(list(frames), stack_axis=0)
        if t >= 20 and t % 5 == 0:
            rbuf.sample(8)
            rbuf.update_errors([float(x) for x in np.abs(rng.randn(8)) * 3])
    rbuf.save(os.path.join(OUT, "ref_per_lazyframes.pkl"))
    sums = rbuf.memory.priority_sums
    pri = []
    for i in range(len(rbuf)):
        v = sums._write(i, 0.0)
        sums._write(i, v)
        pri.append(v)
    exp = expected(rbuf.memory.data, 0.99)
    np.savez_compressed(os.path.join(OUT, "ref_per_lazyframes_expected.npz"),
                        n=len(rbuf), capacity=40, priority=np.asarray(pri, dtype=np.float64),
                        max_priority=np.float64(rbuf.memory.max_priority),
                        total=np.float64(sums.sum()), **exp)
    print("wrote reference checkpoints:", len(rbuf), "PER experiences")


def main():
    import_reference()
    os.makedirs(OUT, exist_ok=True)
    print("numpy", np.__version__)
    gen_reference_checkpoints()
    gen_state_dict_layouts()
    gen_seeded_init()
    gen_per_trace("per_trace_1step", seed=11, capacity=300, num_steps=1, n_envs=1, steps=900,
                  batch=16, alpha=0.6, beta0=0.4, betasteps=200, normalize_by_max=True,
                  gamma=0.99)
    gen_per_trace("per_trace_3step_memory", seed=12, capacity=500, num_steps=3, n_envs=3,
                  steps=500, batch=32, alpha=0.5, beta0=0.4, betasteps=100,
                  normalize_by_max="memory", gamma=0.99)
    gen_per_trace("per_trace_lazyframes", seed=13, capacity=257, num_steps=3, n_envs=2,
                  steps=500, batch=24, alpha=0.5, beta0=0.5, betasteps=None,
                  normalize_by_max=False, gamma=0.9, lazy=True)
    gen_uniform_trace("uniform_trace_sac", seed=21, capacity=400, num_steps=1, steps=1200,
                      batch=32, gamma=0.99)
    gen_uniform_trace("uniform_trace_3step", seed=22, capacity=1000, num_steps=3, steps=900,
                      batch=16, gamma=0.97)
    try:
        from oracle import gen_golden_losses  # noqa: E402
    except ImportError:
        return
    gen_golden_losses.main(OUT)


if __name__ == "__main__":
    main()


def gen_state_dict_layouts():
    """Parameter names and shapes of the reference's model classes (what its
    <attr>.pt checkpoints contain), plus one real Rainbow checkpoint directory
    written by the reference's Agent.save (agent.py:81-106)."""
    import json

    import torch
    from torch import nn

    import pfrl

    def layout(m):
        return {k: list(v.shape) for k, v in m.state_dict().items()}

    torch.manual_seed(0)
    noisy_ddqn = pfrl.q_functions.DistributionalDuelingDQN(18, 51, -10, 10)
    pfrl.nn.to_factorized_noisy(noisy_ddqn, sigma_scale=0.5)
    models = {
        "LargeAtariCNN": pfrl.nn.LargeAtariCNN(),
        "SmallAtariCNN": pfrl.nn.SmallAtariCNN(),
        "MLP(7,3,(16,8))": pfrl.nn.MLP(7, 3, (16, 8)),
        "EmpiricalNormalization(6)": pfrl.nn.EmpiricalNormalization(6),
        "FCStateQFunctionWithDiscreteAction(5,3,16,2)":
            pfrl.q_functions.FCStateQFunctionWithDiscreteAction(5, 3, 16, 2),
        "DistributionalFCStateQFunctionWithDiscreteAction(5,3,11,-1,1,16,2)":
            pfrl.q_functions.DistributionalFCStateQFunctionWithDiscreteAction(5, 3, 11, -1, 1, 16, 2),
        "DuelingDQN(6)": pfrl.q_functions.DuelingDQN(6),
        "DistributionalDuelingDQN(18,51,-10,10)":
            pfrl.q_functions.DistributionalDuelingDQN(18, 51, -10, 10),
        "DistributionalDuelingDQN(18,51,-10,10)+noisy": noisy_ddqn,
        "GaussianHeadWithStateIndependentCovariance(3,diagonal)":
            pfrl.policies.GaussianHeadWithStateIndependentCovariance(3, var_type="diagonal"),
        "Branched(Linear(4,2),Linear(4,1))": pfrl.nn.Branched(nn.Linear(4, 2), nn.Linear(4, 1)),
    }
    with open(os.path.join(OUT, "ref_state_dict_layouts.json"), "w") as f:
        json.dump({k: layout(m) for k, m in models.items()}, f, indent=1, sort_keys=True)

    # a real checkpoint: small Rainbow agent after a few updates
    torch.manual_seed(1)
    np.random.seed(1)
    q = pfrl.q_functions.DistributionalFCStateQFunctionWithDiscreteAction(5, 2, 11, -1, 2, 16, 2)
    pfrl.nn.to_factorized_noisy(q, sigma_scale=0.5)
    rbuf = pfrl.replay_buffers.PrioritizedReplayBuffer(100, num_steps=2)
    agent = pfrl.agents.CategoricalDoubleDQN(
        q, torch.optim.Adam(q.parameters(), lr=1e-3), rbuf, 0.9, pfrl.explorers.Greedy(),
        replay_start_size=20, minibatch_size=8, target_update_interval=10,
        phi=lambda x: x.astype(np.float32, copy=False))
    rng = np.random.RandomState(2)
    obs = [rng.randn(5).astype(np.float32)]
    for t in range(60):
        a = agent.batch_act(obs)
        nobs = [rng.randn(5).astype(np.float32)]
        done = t % 17 == 16
        agent.batch_observe(nobs, [float(rng.randn())], [done], [False])
        obs = nobs
    ckpt = os.path.join(OUT, "ref_ckpt_rainbow")
    agent.save(ckpt)
    probe = rng.randn(4, 5).astype(np.float32)
    torch.manual_seed(123)  # the noisy layers draw fresh noise at every forward
    with torch.no_grad(), pfrl.utils.evaluating(agent.model):
        out = agent.model(torch.tensor(probe))
    np.savez_compressed(os.path.join(OUT, "ref_ckpt_rainbow_expected.npz"), probe=probe,
                        q_values=out.q_values.numpy(), q_dist=out.q_dist.numpy(),
                        optim_steps=np.int64(agent.optim_t))
    print("wrote state-dict layouts and", sorted(os.listdir(ckpt)))


def gen_seeded_init():
    """Initial parameters the reference's constructors produce under
    torch.manual_seed(11) (same-seed reproducibility of a drop-in)."""
    import torch

    import pfrl

    from oracle.digest import store_exact

    g = {}

    def rec(name, make):
        torch.manual_seed(11)
        for k, v in make().state_dict().items():
            store_exact(g, name + "__" + k, v.numpy())

    def noisy():
        q = pfrl.q_functions.DistributionalFCStateQFunctionWithDiscreteAction(
            5, 2, 11, -1.0, 2.0, 16, 2)
        pfrl.nn.to_factorized_noisy(q, sigma_scale=0.5)
        return q

    rec("FCQ", lambda: pfrl.q_functions.FCStateQFunctionWithDiscreteAction(5, 2, 32, 2))
    rec("DistFCQ", lambda: pfrl.q_functions.DistributionalFCStateQFunctionWithDiscreteAction(
        5, 2, 21, -1.0, 2.0, 32, 2))
    rec("MLP", lambda: pfrl.nn.MLP(7, 3, (16, 8)))
    rec("SmallAtariCNN", lambda: pfrl.nn.SmallAtariCNN())
    rec("NoisyDistFCQ", noisy)
    np.savez_compressed(os.path.join(OUT, "ref_seeded_init.npz"), **g)
    print("wrote ref_seeded_init.npz with", len(g), "arrays")
