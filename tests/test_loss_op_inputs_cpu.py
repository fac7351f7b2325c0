"""CPU: the loss / GAE / PPO wrappers hand the C ABI one live fp32 (or uint8 / int64)
copy per input, whatever dtype and layout the caller passed.

The library is replaced by a fake whose ``b2rl_*`` entry points check, at call time,
that the input pointers are pairwise distinct and that the memory behind each holds the
expected converted values.  A wrapper that converts inside the argument list
(``_p(_f32(x))``) frees each copy before the next conversion reuses its block, so
fp64 rewards / discounts or a bool ``terminal`` end up behind one address."""
import ctypes

import numpy as np
import pytest
import torch

from pfrl_b200 import _lib
from pfrl_b200.ops import losses, ppo


class _FakeLib:
    """Records each call; ``expect[name]`` = {arg index: expected array} is checked
    while the call is in progress, i.e. while the wrapper still holds its copies."""

    def __init__(self):
        self.expect = {}
        self.calls = []

    def __getattr__(self, name):
        if not name.startswith("b2rl_"):
            raise AttributeError(name)

        def entry(*args):
            vals = [a.value if isinstance(a, ctypes.c_void_p) else a for a in args]
            checks = self.expect[name]
            ptrs = [vals[i] for i in checks]
            assert all(p is not None for p in ptrs), (name, ptrs)
            assert len(set(ptrs)) == len(ptrs), "%s: aliased input pointers %s" % (name, ptrs)
            for i, want in checks.items():
                got = np.frombuffer(ctypes.string_at(vals[i], want.nbytes), dtype=want.dtype)
                np.testing.assert_array_equal(got, want.reshape(-1), err_msg="%s arg %d" % (name, i))
            self.calls.append(name)
            return 0

        return entry


@pytest.fixture
def fake(monkeypatch):
    lib = _FakeLib()
    monkeypatch.setattr(_lib, "load", lambda: lib)
    monkeypatch.setattr(_lib, "check", lambda status: None)
    monkeypatch.setattr(losses, "_stream", lambda: None)
    monkeypatch.setattr(ppo, "_stream", lambda: None)
    return lib


def _f32(x):
    return np.ascontiguousarray(x.detach().numpy().astype(np.float32))


def _wide(g, *shape, dtype=torch.float64):
    """A column of a wider tensor: non-contiguous, stride 3 along the last axis."""
    return torch.randn(*shape, 3, generator=g, dtype=dtype)[..., 1]


def test_td_loss_inputs(fake):
    g = torch.Generator().manual_seed(0)
    B, nA = 37, 5
    q = torch.randn(nA, B, generator=g).t()                   # fp32, transposed
    action = torch.randint(0, nA, (2 * B,), generator=g)[::2]  # int64, strided
    next_q = _wide(g, B)
    reward = torch.randn(B, generator=g, dtype=torch.float64)
    discount = torch.full((2 * B,), 0.99, dtype=torch.float64)[::2]
    terminal = torch.rand(B, generator=g) < 0.3               # bool
    weights = torch.rand(B, generator=g, dtype=torch.float64)
    fake.expect["b2rl_td_loss_fwd"] = {
        0: _f32(q), 1: action.numpy().astype(np.int64), 2: _f32(next_q), 3: _f32(reward),
        4: _f32(discount), 5: terminal.numpy().astype(np.float32), 6: _f32(weights)}
    losses.td_loss(q, action, next_q, reward, discount, terminal, weights)
    assert fake.calls == ["b2rl_td_loss_fwd"]


def test_c51_loss_inputs(fake):
    g = torch.Generator().manual_seed(1)
    B, n = 13, 11
    y = torch.rand(n, B, generator=g, dtype=torch.float64).t()  # fp64, transposed
    next_p = torch.rand(B, 2 * n, generator=g)[:, ::2]           # fp32, strided rows
    reward = _wide(g, B)
    discount = torch.full((B,), 0.99, dtype=torch.float64)
    terminal = (torch.rand(B, generator=g) < 0.3).to(torch.uint8)
    weights = _wide(g, B, dtype=torch.float16)
    z = torch.linspace(-10, 10, n, dtype=torch.float64)
    fake.expect["b2rl_c51_loss_fwd"] = {
        0: _f32(y), 1: _f32(next_p), 2: _f32(reward), 3: _f32(discount),
        4: terminal.numpy().astype(np.float32), 5: _f32(weights), 6: _f32(z)}
    losses.c51_loss(y, next_p, reward, discount, terminal, weights, z=z)
    assert fake.calls == ["b2rl_c51_loss_fwd"]


def test_quantile_huber_inputs(fake):
    g = torch.Generator().manual_seed(2)
    B, N, Np = 6, 8, 5
    y = _wide(g, B, N)
    t = torch.randn(Np, B, generator=g, dtype=torch.float64).t()
    taus = torch.rand(B, 2 * N, generator=g)[:, 1::2]
    weights = torch.rand(B, generator=g, dtype=torch.float64)
    fake.expect["b2rl_quantile_huber_fwd"] = {
        0: _f32(y), 1: _f32(t), 2: _f32(taus), 3: _f32(weights)}
    losses.quantile_huber_loss(y, t, taus, weights)
    assert fake.calls == ["b2rl_quantile_huber_fwd"]


def test_gae_inputs(fake):
    g = torch.Generator().manual_seed(3)
    T, E = 9, 4
    reward = torch.randn(T, E, generator=g, dtype=torch.float64)
    nonterminal = (torch.rand(T, E, generator=g) > 0.2).to(torch.float64)
    v = torch.randn(E, T, generator=g).t()
    v_next = _wide(g, T, E)
    cut = torch.rand(T, E, generator=g) < 0.2                 # bool
    valid = (torch.rand(T, E, generator=g) < 0.9).t().contiguous().t()  # bool, transposed
    fake.expect["b2rl_gae"] = {
        0: _f32(reward), 1: _f32(nonterminal), 2: _f32(v), 3: _f32(v_next),
        4: cut.numpy().astype(np.uint8), 5: np.ascontiguousarray(valid.numpy()).astype(np.uint8)}
    ppo.gae(reward, nonterminal, v, v_next, cut, 0.99, 0.95, valid=valid)
    assert fake.calls == ["b2rl_gae"]


@pytest.mark.parametrize("clip_vf", [None, 0.2])
def test_ppo_loss_inputs(fake, clip_vf):
    g = torch.Generator().manual_seed(4)
    M = 21
    lp = _wide(g, M)
    ent = torch.rand(M, generator=g, dtype=torch.float64)
    v = torch.randn(M, 1, generator=g, dtype=torch.float64)
    lp_old = torch.randn(2 * M, generator=g)[1::2]
    v_old = _wide(g, M, 1)
    adv = torch.randn(M, generator=g, dtype=torch.float64)
    vt = torch.randn(1, M, generator=g).t()
    stats = torch.tensor([0.1, 1.3], dtype=torch.float64)
    want = {0: _f32(lp), 1: _f32(ent), 2: _f32(v), 3: _f32(lp_old), 5: _f32(adv), 6: _f32(vt),
            7: _f32(stats)}
    if clip_vf is not None:
        want[4] = _f32(v_old)
    fake.expect["b2rl_ppo_loss"] = want
    ppo.ppo_loss(lp, ent, v, lp_old, v_old if clip_vf is not None else None, adv, vt, stats,
                 0.2, clip_vf, 0.5, 0.01)
    assert fake.calls == ["b2rl_ppo_loss"]
