"""Randomised differential test of the device buffers' host logic against
the REAL reference buffers: random interleavings of append (several env ids,
terminals), stop_current_episode, sample and update_errors, with small
capacities so that eviction, n-step tails and the sample / update protocol all
interact.  Compared: lengths after every op, sampled batches (through each
side's batch_experiences), importance weights, and the trees' total at the
end.  The store is tests/fake_store.OracleBackedStore.

The reference's side is tests/golden/ref_buffer_differential.npz, recorded by
oracle/gen_golden_differential.py running `_trace` below with lib = pfrl."""
import os
import sys
from unittest import mock

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.dirname(__file__))
from fake_store import OracleBackedStore  # noqa: E402

from oracle.digest import assert_exact  # noqa: E402

GOLD = os.path.join(os.path.dirname(__file__), "golden")
EXACT_FIELDS = ("state", "next_state", "action", "discount", "is_state_terminal")


def _config(seed):
    prioritized = seed % 2 == 0
    num_steps = [1, 2, 3, 5][seed % 4]
    capacity = [7, 16, 33, 50][(seed // 2) % 4]
    return prioritized, num_steps, capacity, 1 + seed % 3


def _trace(lib, seed, n_ops=400):
    """Drive one buffer of `lib` (pfrl or pfrl_b200) through the scripted ops of `seed`.
    Returns the length after every op, each sampled batch's fields concatenated in
    order with the batch sizes, and for prioritized buffers the trees' total and
    max priority at the end."""
    prioritized, num_steps, capacity, n_envs = _config(seed)
    reference = lib.__name__ == "pfrl"
    if prioritized:
        kw = dict(alpha=0.7, beta0=0.5, betasteps=50, num_steps=num_steps,
                  normalize_by_max=[True, "memory", False][seed % 3])
        if reference:
            buf = lib.replay_buffers.PrioritizedReplayBuffer(capacity, **kw)
            raw = buf.update_errors
            buf.update_errors = lambda e: raw([float(x) for x in e])
        else:
            buf = lib.replay_buffers.PrioritizedReplayBuffer(capacity, device=0, **kw)
    elif reference:
        buf = lib.replay_buffers.ReplayBuffer(capacity, num_steps)
    else:
        buf = lib.replay_buffers.ReplayBuffer(capacity, num_steps, device=0)
    if reference:
        phi = lambda x: np.asarray(x, dtype=np.float32)  # noqa: E731
    else:
        phi = lib.utils.phi.Identity()
    rng = np.random.RandomState(seed)
    np.random.seed(seed)  # the stream sample() draws from
    cur = [rng.randn(3).astype(np.float32) for _ in range(n_envs)]
    cpu = torch.device("cpu")
    lens, sizes = [], []
    out = {k: [] for k in EXACT_FIELDS + ("reward", "weights")}
    for step in range(n_ops):
        op = rng.rand()
        if op < 0.7:
            e = rng.randint(n_envs)
            nxt = rng.randn(3).astype(np.float32)
            done = rng.rand() < 0.15
            buf.append(cur[e], int(rng.randint(4)), float(rng.randn()), nxt, None, bool(done),
                       env_id=e)
            cur[e] = rng.randn(3).astype(np.float32) if done else nxt
            if done or rng.rand() < 0.05:
                buf.stop_current_episode(env_id=e)
        elif op < 0.8:
            buf.stop_current_episode(env_id=rng.randint(n_envs))
        elif len(buf) > 0:
            n = int(rng.randint(1, min(len(buf), 6) + 1))
            exps = buf.sample(n)
            b = lib.replay_buffer.batch_experiences(exps, cpu, phi, 0.9)
            sizes.append(n)
            for k in EXACT_FIELDS:
                out[k].append(b[k].float().numpy())
            out["reward"].append(b["reward"].numpy())
            if prioritized:
                if reference:
                    out["weights"].append(np.asarray([x[0]["weight"] for x in exps],
                                                     dtype=np.float32))
                else:
                    out["weights"].append(b["weights"].numpy())
                buf.update_errors([float(x) for x in np.abs(rng.randn(n)) * 2])
        lens.append(len(buf))
    tr = {k: np.concatenate(v) for k, v in out.items() if v}
    tr.update(lens=np.asarray(lens, dtype=np.int64), sizes=np.asarray(sizes, dtype=np.int64))
    if prioritized and len(buf) > 0:
        if reference:
            tr["total"] = np.float64(buf.memory.priority_sums.sum())
            tr["max_priority"] = np.float64(buf.memory.max_priority)
        else:
            buf._flush()
            info = buf.store.info()
            tr["total"], tr["max_priority"] = np.float64(info["total"]), np.float64(info["max_priority"])
    return tr


@pytest.mark.parametrize("seed", range(12))
def test_random_interleavings_match_the_reference(seed):
    import pfrl_b200

    g = np.load(os.path.join(GOLD, "ref_buffer_differential.npz"))
    key = lambda k: "s%d_%s" % (seed, k)  # noqa: E731
    with mock.patch("pfrl_b200.replay_buffers.device_buffer.DeviceReplayStore", OracleBackedStore):
        mine = _trace(pfrl_b200, seed)
    recorded = {k[len(key("")):].removesuffix("_sha256") for k in g.files if k.startswith(key(""))}
    assert recorded == set(mine), (seed, sorted(recorded), sorted(mine))
    lens = g[key("lens")]
    if not np.array_equal(mine["lens"], lens):
        raise AssertionError("lengths diverge: seed %d, op %d"
                             % (seed, int(np.argmax(mine["lens"] != lens))))
    assert np.array_equal(mine["sizes"], g[key("sizes")]), seed
    for k in EXACT_FIELDS:
        assert_exact(g, key(k), mine[k], "seed %d" % seed)
    ends = np.cumsum(mine["sizes"])
    for j, (lo, hi) in enumerate(zip(ends - mine["sizes"], ends)):
        torch.testing.assert_close(torch.from_numpy(mine["reward"][lo:hi]),
                                   torch.from_numpy(g[key("reward")][lo:hi]), rtol=1e-6, atol=1e-7)
        if "weights" in mine:
            np.testing.assert_allclose(mine["weights"][lo:hi], g[key("weights")][lo:hi],
                                       rtol=2e-6, err_msg="seed %d, sample %d" % (seed, j))
    if "total" in mine:
        assert mine["total"] == g[key("total")]
        assert mine["max_priority"] == g[key("max_priority")]
