"""MountainCar-v0 on the CPU: the CPU reference's env (tests/mc_oracle.c) against gym's step() restated in plain Python, its discrete
search over three actions through ties, epsilon picks, terminal nodes and visit counts past 255, and the host-side plumbing that selects
the env (no GPU needed)."""
import math
import re

import numpy as np
import pytest

from oracle import azo
import mc_oracle as M
from mc_oracle import MountainCarEnv, det_cos


def edge_cases():
    """(state, action) pairs: random states in the box with all three actions, the left wall with negative velocity, velocities
    crossing +-0.07, the goal line with velocity +0 / -0 / -eps, signed zeros and NaN in the state."""
    rng = np.random.default_rng(8)
    out = [((p, v), int(a)) for p, v, a in zip(rng.uniform(-1.2, 0.6, 300), rng.uniform(-0.07, 0.07, 300), rng.integers(0, 3, 300))]
    for v in (-0.07, -0.05, -1e-3, -1e-300, -0.0):  # the left wall: position clamps to -1.2 and a negative velocity becomes +0
        out += [((-1.19, v), 0), ((-1.2, v), 1), ((-1.2, v), 2)]
    for v in (0.069999, -0.069999, 0.07, -0.07, 0.0699999999999):  # both speed clips
        out += [((0.0, v), 2), ((-0.52, v), 0), ((0.3, v), 1)]
    for v in (0.0, -0.0, -5e-324, 5e-324):  # the goal line
        out += [((0.5, v), 1), ((0.5, v), 2), ((0.4999999999, v), 2), ((0.49, v), 1)]
    out += [((0.6, 0.07), 2), ((0.59, 0.07), 2), ((-0.0, 0.0), 1), ((0.0, -0.0), 1), ((-0.5235987755982988, -0.0), 1),
            ((np.nan, 0.0), 1), ((-0.5, np.nan), 0), ((np.nan, np.nan), 2)]
    return out


def _bits(x):
    return np.asarray(x, np.float64).view(np.uint64)


@pytest.mark.parametrize("math_mode", [azo.MATH_LIBM, azo.MATH_DET])
def test_env_step_equals_gym_restatement(math_mode):
    """mc_oracle.env_step == MountainCarEnv.step bit for bit (state, reward, done, observation) with the same cosine."""
    cfg = M.config()
    cfg.math_mode = math_mode
    cos = math.cos if math_mode == azo.MATH_LIBM else det_cos
    n_done = n_wall = 0
    for s, a in edge_cases():
        nxt, r, term, obs = M.env_step(cfg, np.array(s, np.float64), a)
        gs, gr, gdone, _ = MountainCarEnv(s, cos=cos).step(a)
        gs = np.asarray(gs, np.float64)
        assert np.array_equal(_bits(nxt), _bits(gs)), (s, a, nxt, gs)
        assert _bits(r) == _bits(gr) and r == -1.0, (s, a, r, gr)
        assert term == gdone, (s, a)
        assert np.array_equal(obs.view(np.uint32), gs.astype(np.float32).view(np.uint32))
        n_done += term
        n_wall += gs[0] == -1.2
    assert n_done >= 8 and n_wall >= 6


def test_env_step_edges():
    cfg = M.config()
    # the left wall: velocity becomes +0.0 (the int 0)
    s, _, _, _ = M.env_step(cfg, np.array([-1.2, -0.03]), 0)
    assert s[0] == -1.2 and _bits(s[1]) == _bits(0.0)
    # action 1 applies zero force: the velocity change is the gravity term alone
    s, _, _, _ = M.env_step(cfg, np.array([-0.5, 0.01]), 1)
    assert s[1] == 0.01 + (0.0 + det_cos(3 * -0.5) * -0.0025)
    # pushing left / right differ by exactly 2 * force before rounding
    s0, _, _, _ = M.env_step(cfg, np.array([-0.5, 0.0]), 0)
    s2, _, _, _ = M.env_step(cfg, np.array([-0.5, 0.0]), 2)
    assert s0[1] < s2[1]
    # the goal line: done with velocity +0 and -0, not with a negative velocity, nor for a NaN state
    for v, want in ((0.0, True), (-0.0, True), (-1e-300, False)):
        env = MountainCarEnv((0.5, v))
        env.state = (0.5, v)
        assert bool(0.5 >= env.goal_position and v >= env.goal_velocity) == want
    _, r, term, _ = M.env_step(cfg, np.array([0.499, 0.07]), 2)
    assert term and r == -1.0
    s, _, term, _ = M.env_step(cfg, np.array([np.nan, 0.0]), 1)
    assert np.isnan(s).all() and not term
    # both speed clips
    s, _, _, _ = M.env_step(cfg, np.array([0.55, 0.07]), 2)  # cos(1.65) < 0: gravity pushes right too
    assert s[1] == 0.07
    s, _, _, _ = M.env_step(cfg, np.array([0.0, -0.07]), 0)
    assert s[1] == -0.07


def roots(kind, B, seed=3):
    rng = np.random.default_rng(seed)
    if kind == "goal":
        return np.stack([rng.uniform(0.42, 0.5, B), rng.uniform(0.0, 0.07, B)], 1)
    return np.stack([rng.uniform(-0.6, -0.4, B), np.zeros(B)], 1)  # Env.reset's distribution


def weights(cfg, seed=34):
    from alphazero_gym_b200.network import init_policy_weights
    return init_policy_weights(seed, cfg.state_dim, cfg.hidden, cfg.n_hidden, cfg.head_dim)


def zero_head(cfg, w):
    """All head weights and biases zero: uniform priors and V = 0 at every node, so the three scores tie at every fresh node."""
    w = w.copy()
    w[-(1 + cfg.hidden + cfg.head_dim * cfg.hidden + cfg.head_dim):] = 0.0
    return w


def test_oracle_search_ties_and_terminals():
    """Near the goal: terminal expansions (V = 0, r = -1), traces that end on an existing terminal node (counters[6]), and three-way
    ties resolved by the random pick among the winners (all three actions taken first at some fresh node)."""
    cfg = M.config(n_rollouts=50, epsilon=0.0)
    w = zero_head(cfg, weights(cfg))
    out = M.search(cfg, w, roots("goal", 64), n_threads=4)
    assert out["counters"][6] > 0
    term = out["terminal"].astype(bool)
    assert term.any() and not term[:, 0].any()
    assert (out["V"][term] == 0).all() and (out["r"][term] == -1.0).all()
    assert (out["prior"][:, 0] == np.float32(1 / 3)).all()
    first = out["paction"][:, 1]  # the action of the first simulation: a uniform pick among three tied scores
    assert set(first.tolist()) == {0, 1, 2}
    assert (out["counters"][2] == 3 * out["counters"][1])
    # the root and every non-terminal node take the env's reward, unscaled
    live = np.arange(out["r"].shape[1])[None, :] < out["n_nodes"][:, None]
    live[:, 0] = False
    assert (out["r"][live] == -1.0).all()


def test_oracle_search_epsilon_and_deep_counts():
    """epsilon = 0.25 makes random picks of every action; N = 300 pushes the root's visit count past 255."""
    cfg = M.config(n_rollouts=300, epsilon=0.25, V_target_policy="on_policy", gamma=0.99)
    out = M.search(cfg, weights(cfg), roots("valley", 8), n_threads=4)
    assert out["counts"].sum() == 8 * 300 and out["node_n"][:, 0].max() == 300
    assert (out["en"][:, 0, 2] > 0).all() and out["counters"][5] == 2 * out["counters"][1]
    tot = out["counts"].sum(1).astype(np.float64)
    v = np.zeros(8)
    for a in range(3):
        v = v + (out["counts"][:, a] / tot) * out["Q"][:, a]
    assert np.array_equal(v, out["V_target"])


def test_oracle_selfplay_reset_and_reuse():
    from oracle import selfplay as SP
    cfg = M.config(n_rollouts=10)
    r0 = roots("goal", 8)
    steps = M.selfplay_run(cfg, weights(cfg), r0, steps=3, max_episode_length=2, seed=5)
    for k, rec in enumerate(steps):
        key = SP.step_seed(5, k)
        for t in np.nonzero(rec["done"])[0]:
            u = SP._unit(azo.rng_u32(key, t, 3, int(rec["episode"][t]), 0, 0))
            assert rec["env_state"][t, 0] == -0.6 + (-0.4 - -0.6) * u and _bits(rec["env_state"][t, 1]) == _bits(0.0)
    assert any(r["done"].any() for r in steps) and steps[0]["obs"].shape == (8, 2)
    assert set(np.concatenate([r["action_taken"] for r in steps]).tolist()) <= {0.0, 1.0, 2.0}
    assert steps[0]["root_n"][steps[0]["done"] == 0].min() > 0  # tree reuse carries the chosen child's visit count


def test_engine_config_and_env_recognition():
    from alphazero_gym_b200 import _cabi
    from alphazero_gym_b200._cabi import CONTINUOUS, DISCRETE
    from alphazero_gym_b200.engine import CARTPOLE, MOUNTAIN_CAR, EngineConfig
    from alphazero_gym_b200.search.mcts import discrete_env, env_hidden_state, reward_model
    from alphazero_gym_b200.selfplay import initial_states
    from mcc_oracle import Continuous_MountainCarEnv

    c = EngineConfig(variant=DISCRETE, num_actions=3, state_dim=2, env=MOUNTAIN_CAR)
    assert c.c().flags & _cabi.FLAG_ENV_MOUNTAIN_CAR and _cabi.FLAG_ENV_MOUNTAIN_CAR == 32 and c.is_fused()
    assert not c.c().flags & _cabi.FLAG_ENV_MOUNTAIN_CAR_CONTINUOUS
    assert not EngineConfig(variant=DISCRETE, state_dim=4, num_actions=3, env=MOUNTAIN_CAR).is_fused()
    assert not EngineConfig(variant=DISCRETE).c().flags & _cabi.FLAG_ENV_MOUNTAIN_CAR
    with pytest.raises(ValueError):
        EngineConfig(variant=CONTINUOUS, env=MOUNTAIN_CAR).c()

    class TimeLimit:
        def __init__(self, env):
            self.env = env

    class ScaleRewardWrapper(TimeLimit):
        pass

    env = MountainCarEnv((-0.5, 0.0))
    assert discrete_env(TimeLimit(env)) == MOUNTAIN_CAR and discrete_env(object()) == CARTPOLE
    assert np.array_equal(env_hidden_state(TimeLimit(env), DISCRETE, env_id=MOUNTAIN_CAR), [-0.5, 0.0])
    for variant in (DISCRETE, CONTINUOUS):  # the two-argument form keeps refusing it
        with pytest.raises(TypeError):
            env_hidden_state(env, variant)
    with pytest.raises(TypeError):
        env_hidden_state(Continuous_MountainCarEnv((-0.5, 0.0)), DISCRETE, env_id=MOUNTAIN_CAR)
    assert reward_model(TimeLimit(env), DISCRETE) == (1.0, 1.0)
    with pytest.raises(NotImplementedError):
        reward_model(ScaleRewardWrapper(env), DISCRETE)
    s = initial_states(DISCRETE, 6, seed=9, tree_id0=2, total=10, env=MOUNTAIN_CAR)
    rng = np.random.default_rng(9)
    assert np.array_equal(s, np.stack([rng.uniform(-0.6, -0.4, 10), np.zeros(10)], 1)[2:8])


def test_dropin_refusals_without_gpu():
    """MCTSDiscrete: MountainCar with num_actions other than 3 and the continuous env raise before any engine exists."""
    from alphazero_gym_b200.search.mcts import MCTSContinuous, MCTSDiscrete
    from mcc_oracle import Continuous_MountainCarEnv
    m = MCTSDiscrete(model=None, num_actions=2, n_rollouts=8, c_uct=1.5, gamma=1.0, epsilon=0.0, V_target_policy="off_policy",
                     device="cuda:0", root_state=None)
    with pytest.raises(ValueError):
        m.search(MountainCarEnv((-0.5, 0.0)))
    with pytest.raises(TypeError):
        m.search(Continuous_MountainCarEnv((-0.5, 0.0)))
    c = MCTSContinuous(model=None, n_rollouts=8, c_uct=0.05, c_pw=1.0, kappa=0.5, gamma=1.0, epsilon=0.0, V_target_policy="off_policy",
                       device="cuda:0", root_state=None)
    with pytest.raises(TypeError):
        c.search(MountainCarEnv((-0.5, 0.0)))


def test_dispatch_tables_have_gpu_cases():
    """Every MountainCar instantiation in engine.cu's dispatch tables runs in tests/test_mountain_car_discrete_gpu.py."""
    import os
    import test_mountain_car_discrete_gpu as G
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = open(os.path.join(root, "alphazero_gym_b200", "csrc", "engine.cu")).read()

    def table(macro):
        return {tuple(int(v) for v in c) for c in re.findall(r"\b" + macro + r"\((\d+), (\d+)\)", src)}

    assert table("FUSED_MC_CASE") == table("QMLP_MC_CASE") == set(G.Q8_SHAPES)
    assert table("MLP_MCC_CASE") == set(G.FP32_SHAPES)  # k_mlp<H, 2, ACT> serves both MountainCar envs
