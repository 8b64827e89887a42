"""The reference-shaped agents (alphazero_gym_b200/agent/agents.py): constructed from the reference's Hydra-style configs with the
`_target_`s of this repo's config/*/*.yaml, they must reproduce the UNMODIFIED reference agents' `update` steps -- the golden vectors
of oracle/gen_train_golden.py (same configs with the reference's `_target_`s, same seeded replay batches)."""
import json
import os

import numpy as np
import pytest
import torch
import yaml

from alphazero_gym_b200.agent.agents import ContinuousAgent, DiscreteAgent

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")

CONT_POLICY = dict(_target_="alphazero_gym_b200.network.make_policy", representation_dim=3, action_dim=1, action_bound=2.0,
                   distribution="normal", num_components=2, hidden_dimensions=[128, 128, 128], nonlinearity="elu", layernorm=False,
                   log_param_min=-5, log_param_max=2)
DISC_POLICY = dict(_target_="alphazero_gym_b200.network.make_policy", representation_dim=4, num_actions=2, action_dim=1,
                   distribution="discrete", hidden_dimensions=[128, 128], nonlinearity="relu", layernorm=False)
MCTS_C = dict(_target_="alphazero_gym_b200.search.mcts.MCTSContinuous", n_rollouts=25, c_uct=0.05, c_pw=1, kappa=0.5, gamma=1, epsilon=0,
              V_target_policy="off_policy", device="cpu", root_state=None)
MCTS_D = dict(_target_="alphazero_gym_b200.search.mcts.MCTSDiscrete", num_actions=2, n_rollouts=8, c_uct=1.5, gamma=1, epsilon=0.1,
              V_target_policy="off_policy", device="cpu", root_state=None)
RMSPROP = dict(_target_="torch.optim.RMSprop", lr=0.001, momentum=0, weight_decay=0, alpha=0.9, eps=1e-10)
ADAM = dict(_target_="torch.optim.Adam", lr=0.001, betas=[0.9, 0.99], weight_decay=0, eps=1e-07, amsgrad=False)
L = "alphazero_gym_b200.agent.losses."
CASES = {
    "train_a0c_tuned_rmsprop": (ContinuousAgent, CONT_POLICY, MCTS_C, dict(_target_=L + "A0CLossTuned", action_dim=1, alpha_init=1, lr=0.001, tau=0.1,
                                policy_coeff=0.1, value_coeff=1, reduction="mean", grad_clip=0, device="cpu"), RMSPROP, 0.0, dict(epsilon=0)),
    "train_a0c_adam_clip": (ContinuousAgent, CONT_POLICY, MCTS_C, dict(_target_=L + "A0CLoss", tau=0.1, policy_coeff=1, alpha=1, value_coeff=1,
                            reduction="mean"), ADAM, 0.5, dict(epsilon=0)),
    "train_a0c_discrete_rmsprop": (DiscreteAgent, DISC_POLICY, MCTS_D, dict(_target_=L + "A0CLoss", tau=0.1, policy_coeff=1, alpha=1, value_coeff=1,
                                   reduction="mean"), RMSPROP, 0.0, dict(temperature=1.0)),
}


@pytest.mark.parametrize("name", sorted(CASES))
def test_reference_shaped_agent_reproduces_reference_updates(name):
    cls, policy, mcts, loss, opt, clip, extra = CASES[name]
    g = np.load(os.path.join(GOLD, name + ".npz"))
    torch.set_num_threads(1)
    agent = cls(policy_cfg=policy, mcts_cfg=mcts, loss_cfg=loss, optimizer_cfg=opt, final_selection="max_visit", train_epochs=1,
                grad_clip=clip, device="cpu", **extra)
    agent.nn.load_flat(g["w0"])
    assert agent.n_rollouts == mcts["n_rollouts"] and agent.c_uct == mcts["c_uct"] and agent.gamma == 1 and agent.learning_rate == 0.001
    for s in range(3):
        info = agent.update(tuple(g[f"{k}_{s}"] for k in ("states", "actions", "counts", "Q", "V")))
        for k, v in info.items():
            ref = float(g[f"info_{k}_{s}"])
            assert abs(v - ref) <= 1e-5 * abs(ref) + 1e-7, (s, k, v, ref)
    sd = agent.nn.state_dict()
    keys = [k for k in sd if k.startswith("trunk.")] + ["value_head.weight", "value_head.bias", "dist_head.weight", "dist_head.bias"]
    w = np.concatenate([sd[k].numpy().ravel() for k in keys])
    assert np.abs(w - g["w_3"]).max() <= 2e-6


def test_agent_yaml_dropins_have_the_reference_keys():
    """config/agent|loss|policy|mcts/*.yaml: the reference's keys and values, only `_target_` changed.  The reference's values
    (config/<group>/<name>.yaml of timoklein/alphazero-gym, `_target_` left out) are recorded in tests/golden/reference_config.json,
    as the reference is not part of this repository."""
    with open(os.path.join(GOLD, "reference_config.json")) as fh:
        golden = json.load(fh)
    for grp in ("agent", "loss", "policy", "mcts"):
        for f in os.listdir(os.path.join(ROOT, "config", grp)):
            mine = yaml.safe_load(open(os.path.join(ROOT, "config", grp, f)))
            assert f"{grp}/{f}" in golden, (grp, f)
            ref = golden[f"{grp}/{f}"]
            if grp == "agent":
                mine = mine["agent"]
            assert set(mine) == set(ref) | {"_target_"}, (grp, f)
            for k in ref:
                if k != "_target_":
                    assert mine[k] == ref[k], (grp, f, k)
            assert mine["_target_"].startswith("alphazero_gym_b200."), (grp, f)
