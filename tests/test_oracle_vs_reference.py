"""CPU: the oracle's dense-heap restatement against the REAL reference's
PrioritizedBuffer (pfrl/collections/prioritized.py), bit for bit.  The
reference's side is tests/golden/ref_dense_heap.npz, recorded by
oracle/gen_golden_differential.py running `_trace` below on the reference."""
import os

import numpy as np
import pytest

from oracle.digest import assert_exact
from oracle.replay import OraclePrioritizedBuffer

GOLD = os.path.join(os.path.dirname(__file__), "golden")
CAPACITIES = [1, 2, 3, 7, 64, 100, 777, 1024, 1025]


class _Oracle:
    """OraclePrioritizedBuffer behind the calls `_trace` makes of the reference's class."""

    def __init__(self, cap):
        self.buf = OraclePrioritizedBuffer(cap)

    def __len__(self):
        return len(self.buf)

    def append(self, value, priority):
        self.buf.append(value, priority)

    def sample(self, n):
        idx, pr, tot, mn = self.buf.sample_indices(n)
        return list(idx), [p / tot for p in pr.tolist()], mn / tot

    def set_last_priority(self, priority):
        self.buf.set_last_priority(priority)

    @property
    def max_priority(self):
        return self.buf.max_priority

    def total(self):
        return self.buf.total()


def _trace(buf, cap):
    """A random mix of appends (default and explicit priorities), samples and priority
    updates.  Returns the length after every op, each sample's indices, probabilities
    and min probability, the max priority after each update and the final total."""
    rng = np.random.RandomState(cap)
    lens, sizes, idx, probs, pmin, maxp = [], [], [], [], [], []
    for t in range(1200):
        if rng.rand() < 0.6 or len(buf) < min(4, cap):
            for _ in range(int(rng.randint(1, 8))):
                pr = None if rng.rand() < 0.7 else float(rng.rand() * 3 + 1e-3)
                buf.append(t, pr)
        else:
            n = int(rng.randint(1, min(len(buf), 40) + 1))
            np.random.seed(int(rng.randint(1 << 30)))
            i, p, m = buf.sample(n)
            sizes.append(n)
            idx.extend(i)
            probs.extend(p)
            pmin.append(m)
            buf.set_last_priority([float(x) for x in (rng.rand(n) * 2 + 1e-6) ** 0.6])
            maxp.append(buf.max_priority)
        lens.append(len(buf))
    return dict(lens=np.asarray(lens, dtype=np.int64), sizes=np.asarray(sizes, dtype=np.int64),
                indices=np.asarray(idx, dtype=np.int64), probs=np.asarray(probs, dtype=np.float64),
                min_prob=np.asarray(pmin, dtype=np.float64),
                max_priority=np.asarray(maxp, dtype=np.float64), total=np.float64(buf.total()))


@pytest.mark.parametrize("cap", CAPACITIES)
def test_dense_heap_oracle_is_bit_identical_to_reference_tree(cap):
    g = np.load(os.path.join(GOLD, "ref_dense_heap.npz"))
    mine = _trace(_Oracle(cap), cap)
    for k, v in mine.items():
        assert_exact(g, "c%d_%s" % (cap, k), v)
    assert len(mine["indices"]) > 0 or cap == 1
