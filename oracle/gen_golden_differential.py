"""Record the REAL reference's side of the randomised differential tests.

TEST INFRASTRUCTURE ONLY.  Run in the build container (needs the reference tree):

    python oracle/gen_golden_differential.py

The scenarios are the tests' own functions, called here with the reference's
package; the tests call them with pfrl_b200 and compare against these files:

  tests/golden/ref_agent_differential.npz   tests/test_agent_differential_cpu.py
  tests/golden/ref_buffer_differential.npz  tests/test_buffer_differential_cpu.py
  tests/golden/ref_dense_heap.npz           tests/test_oracle_vs_reference.py
  tests/golden/ref_explorers.npz            tests/test_host_logic_cpu.py
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TESTS = os.path.join(ROOT, "tests")
sys.path.insert(0, ROOT)
sys.path.insert(0, TESTS)
from oracle.digest import store_exact  # noqa: E402
from oracle.refimport import import_reference  # noqa: E402

OUT = os.path.join(TESTS, "golden")


def agent_differential(pfrl):
    import test_agent_differential_cpu as t

    runs = [("ppo%d" % s, t._run_ppo, s) for s in range(6)]
    runs += [("a2c%d" % s, t._run_a2c, s) for s in range(4)]
    runs += [(k, t._run_dqn_family, k) for k in ("ddqn", "rainbow", "c51")]
    runs += [(k, t._run_uniform_replay_agent, k) for k in ("sac", "td3", "ddpg", "iqn")]
    g = {}
    for key, run, arg in runs:
        acts, stats, params = run(pfrl, arg)
        g[key + "_actions"], g[key + "_stats"] = acts, stats
        g[key + "_n_params"] = np.int64(len(params))
        for i, p in enumerate(params):
            g["%s_param%d" % (key, i)] = p
    np.savez_compressed(os.path.join(OUT, "ref_agent_differential.npz"), **g)


def buffer_differential(pfrl):
    import test_buffer_differential_cpu as t

    g = {}
    for seed in range(12):
        for k, v in t._trace(pfrl, seed).items():
            if k in t.EXACT_FIELDS:
                store_exact(g, "s%d_%s" % (seed, k), v)
            else:
                g["s%d_%s" % (seed, k)] = v
    np.savez_compressed(os.path.join(OUT, "ref_buffer_differential.npz"), **g)


class _ReferenceHeap:
    """The reference's PrioritizedBuffer behind the calls tests/test_oracle_vs_reference.py's
    `_trace` makes (the sample half of PrioritizedReplayBuffer.sample, uniform_ratio 0)."""

    def __init__(self, pfrl, cap):
        self.buf = pfrl.collections.prioritized.PrioritizedBuffer(capacity=cap)

    def __len__(self):
        return len(self.buf)

    def append(self, value, priority):
        self.buf.append(value, priority)

    def sample(self, n):
        idx, probs, min_prob = self.buf._sample_indices_and_probabilities(n, 0)
        self.buf.sampled_indices, self.buf.flag_wait_priority = idx, True
        return idx, probs, min_prob

    def set_last_priority(self, priority):
        self.buf.set_last_priority(priority)

    @property
    def max_priority(self):
        return self.buf.max_priority

    def total(self):
        return self.buf.priority_sums.sum()


def dense_heap(pfrl):
    import test_oracle_vs_reference as t

    g = {}
    for cap in t.CAPACITIES:
        for k, v in t._trace(_ReferenceHeap(pfrl, cap), cap).items():
            store_exact(g, "c%d_%s" % (cap, k), v)
    np.savez_compressed(os.path.join(OUT, "ref_dense_heap.npz"), **g)


def explorers(pfrl):
    import test_host_logic_cpu as t

    g = {}
    for name, _, _ in t.EXPLORER_CASES:
        acts, stream, rep = t._explorer_trace(pfrl.explorers, pfrl.action_value.DiscreteActionValue,
                                              name)
        g[name + "_actions"], g[name + "_stream"], g[name + "_repr"] = acts, stream, np.str_(rep)
    np.savez_compressed(os.path.join(OUT, "ref_explorers.npz"), **g)


def main():
    pfrl = import_reference()
    import pfrl.collections.prioritized  # noqa: F401

    print("numpy", np.__version__)
    for gen in (agent_differential, buffer_differential, dense_heap, explorers):
        gen(pfrl)
        print("wrote", gen.__name__)


if __name__ == "__main__":
    main()
