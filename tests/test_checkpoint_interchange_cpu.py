"""Model checkpoints written by the reference load into this package's
classes: parameter names and shapes of every model class we mirror equal the
reference's (tests/golden/ref_state_dict_layouts.json), and a real
``Agent.save`` directory of a small Rainbow agent (tests/golden/
ref_ckpt_rainbow/, pfrl/agent.py:81-106) loads with ``agent.load`` and
reproduces the reference's outputs.  Fixtures: oracle/gen_golden.py:
gen_state_dict_layouts."""
import json
import os

import numpy as np
import torch
from torch import nn

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _models():
    import pfrl_b200 as lib

    noisy = lib.q_functions.DistributionalDuelingDQN(18, 51, -10, 10)
    lib.nn.to_factorized_noisy(noisy, sigma_scale=0.5)
    return {
        "LargeAtariCNN": lib.nn.LargeAtariCNN(),
        "SmallAtariCNN": lib.nn.SmallAtariCNN(),
        "MLP(7,3,(16,8))": lib.nn.MLP(7, 3, (16, 8)),
        "EmpiricalNormalization(6)": lib.nn.EmpiricalNormalization(6),
        "FCStateQFunctionWithDiscreteAction(5,3,16,2)":
            lib.q_functions.FCStateQFunctionWithDiscreteAction(5, 3, 16, 2),
        "DistributionalFCStateQFunctionWithDiscreteAction(5,3,11,-1,1,16,2)":
            lib.q_functions.DistributionalFCStateQFunctionWithDiscreteAction(5, 3, 11, -1, 1, 16, 2),
        "DuelingDQN(6)": lib.q_functions.DuelingDQN(6),
        "DistributionalDuelingDQN(18,51,-10,10)":
            lib.q_functions.DistributionalDuelingDQN(18, 51, -10, 10),
        "DistributionalDuelingDQN(18,51,-10,10)+noisy": noisy,
        "GaussianHeadWithStateIndependentCovariance(3,diagonal)":
            lib.policies.GaussianHeadWithStateIndependentCovariance(3, var_type="diagonal"),
        "Branched(Linear(4,2),Linear(4,1))": lib.nn.Branched(nn.Linear(4, 2), nn.Linear(4, 1)),
    }


def test_state_dict_layouts_equal_the_reference():
    with open(os.path.join(GOLD, "ref_state_dict_layouts.json")) as f:
        want = json.load(f)
    models = _models()
    assert sorted(models) == sorted(want)
    for name, m in models.items():
        got = {k: list(v.shape) for k, v in m.state_dict().items()}
        assert got == want[name], name


def test_reference_agent_checkpoint_loads_and_reproduces_outputs():
    import pfrl_b200 as lib
    from pfrl_b200.replay_buffers import HostReplayBuffer
    from pfrl_b200.utils import evaluating

    exp = np.load(os.path.join(GOLD, "ref_ckpt_rainbow_expected.npz"))
    q = lib.q_functions.DistributionalFCStateQFunctionWithDiscreteAction(5, 2, 11, -1, 2, 16, 2)
    lib.nn.to_factorized_noisy(q, sigma_scale=0.5)
    agent = lib.agents.CategoricalDoubleDQN(
        q, torch.optim.Adam(q.parameters(), lr=1e-3), HostReplayBuffer(100, num_steps=2), 0.9,
        lib.explorers.Greedy(), replay_start_size=20, minibatch_size=8,
        target_update_interval=10, phi=lambda x: x.astype(np.float32, copy=False))
    agent.load(os.path.join(GOLD, "ref_ckpt_rainbow"))
    torch.manual_seed(123)  # the noisy layers draw fresh noise at every forward
    with torch.no_grad(), evaluating(agent.model):
        out = agent.model(torch.tensor(exp["probe"]))
    np.testing.assert_allclose(out.q_dist.numpy(), exp["q_dist"], rtol=1e-6, atol=1e-7)
    np.testing.assert_allclose(out.q_values.numpy(), exp["q_values"], rtol=1e-6, atol=1e-7)
    # Adam moments came along: one step per update the reference had made
    steps = {int(st["step"]) for st in agent.optimizer.state_dict()["state"].values()}
    assert steps == {int(exp["optim_steps"])}
    # target net differs from the online net (it was last synchronised some updates ago)
    assert any(not torch.equal(a, b) for a, b in zip(agent.model.parameters(),
                                                     agent.target_model.parameters()))


def test_same_torch_seed_gives_the_reference_initial_weights():
    """Constructors consume torch's global generator in the reference's order
    (tests/golden/ref_seeded_init.npz, oracle/gen_golden.py:gen_seeded_init), so a
    script that only sets the seed starts from the same network."""
    import pfrl_b200 as lib
    from oracle.digest import assert_exact

    g = np.load(os.path.join(GOLD, "ref_seeded_init.npz"))

    def noisy():
        q = lib.q_functions.DistributionalFCStateQFunctionWithDiscreteAction(5, 2, 11, -1.0, 2.0, 16, 2)
        lib.nn.to_factorized_noisy(q, sigma_scale=0.5)
        return q

    makers = {
        "FCQ": lambda: lib.q_functions.FCStateQFunctionWithDiscreteAction(5, 2, 32, 2),
        "DistFCQ": lambda: lib.q_functions.DistributionalFCStateQFunctionWithDiscreteAction(
            5, 2, 21, -1.0, 2.0, 32, 2),
        "MLP": lambda: lib.nn.MLP(7, 3, (16, 8)),
        "SmallAtariCNN": lambda: lib.nn.SmallAtariCNN(),
        "NoisyDistFCQ": noisy,
    }
    for name, make in makers.items():
        torch.manual_seed(11)
        for k, v in make().state_dict().items():
            assert_exact(g, name + "__" + k, v.numpy())
