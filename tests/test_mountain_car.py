"""MountainCarContinuous-v0 on the CPU: the CPU reference's env (tests/mcc_oracle.c) against gym's step() restated in plain Python,
its continuous search through the env's terminal paths, and the host-side plumbing that selects the env (no GPU needed)."""
import math
import re

import numpy as np
import pytest

from oracle import azo
import mcc_oracle as M
from mcc_oracle import Continuous_MountainCarEnv, R_SCALE, det_cos


def edge_cases():
    """(state, action) pairs: random states in the box with random actions, actions beyond +-1 / +-0 / NaN / inf, the left wall
    with negative velocity, velocities crossing +-0.07, the goal line with velocity +0 / -0 / -eps."""
    rng = np.random.default_rng(7)
    out = [((p, v), a) for p, v, a in zip(rng.uniform(-1.2, 0.6, 400), rng.uniform(-0.07, 0.07, 400),
                                          rng.uniform(-1.5, 1.5, 400).astype(np.float32))]
    for a in (1.0, -1.0, 1.0000001, -1.0000001, 3.5, -7.25, 0.0, -0.0, np.nan, np.inf, -np.inf, 1e-30, -1e-45):
        out += [((-0.5, 0.0), np.float32(a)), ((0.44, 0.02), np.float32(a))]
    for v in (-0.07, -0.05, -1e-3, -1e-300):  # the left wall: position clamps to -1.2 and a negative velocity becomes +0
        out += [((-1.19, v), np.float32(-1.0)), ((-1.2, v), np.float32(0.0)), ((-1.2, v), np.float32(1.0))]
    for v in (0.069999, -0.069999, 0.07, -0.07, 0.0699999999999):
        out += [((0.0, v), np.float32(1.0)), ((-0.52, v), np.float32(-1.0)), ((0.3, v), np.float32(0.5))]
    # the goal line, with velocity +0, -0 and +-eps
    for v in (0.0, -0.0, -5e-324, 5e-324):
        out += [((0.45, v), np.float32(0.0)), ((0.45, v), np.float32(1.0)), ((0.4499999999, v), np.float32(1.0))]
    out += [((0.6, 0.07), np.float32(1.0)), ((0.59, 0.07), np.float32(1.0)), ((np.nan, 0.0), np.float32(0.0))]
    return out


def _bits(x):
    return np.asarray(x, np.float64).view(np.uint64)


@pytest.mark.parametrize("math_mode", [azo.MATH_LIBM, azo.MATH_DET])
def test_env_step_equals_gym_restatement(math_mode):
    """mcc_oracle.env_step == Continuous_MountainCarEnv.step bit for bit (state, reward, done, observation) with the same cosine."""
    cfg = M.config()
    cfg.math_mode = math_mode
    cos = math.cos if math_mode == azo.MATH_LIBM else det_cos
    n_done = n_wall = 0
    for s, a in edge_cases():
        nxt, r, term, obs = M.env_step(cfg, np.array(s, np.float64), float(a))
        env = Continuous_MountainCarEnv(s, cos=cos)
        gs, gr, gdone, _ = env.step(np.array([a], np.float32))
        assert np.array_equal(_bits(nxt), _bits(gs)), (s, a, nxt, gs)
        assert _bits(r) == _bits(gr), (s, a, r, gr)
        assert term == gdone, (s, a)
        assert np.array_equal(obs.view(np.uint32), gs.astype(np.float32).view(np.uint32))
        n_done += term
        n_wall += gs[0] == -1.2
    assert n_done >= 10 and n_wall >= 6


def test_env_step_signed_zeros_and_reward():
    cfg = M.config()
    # a zero action pays +0.0 (0 - 0.0 with the int 0), not -0.0
    _, r, term, _ = M.env_step(cfg, np.array([-0.5, 0.0]), 0.0)
    assert not term and _bits(r) == _bits(0.0)
    _, r, _, _ = M.env_step(cfg, np.array([-0.5, 0.0]), -0.0)
    assert _bits(r) == _bits(0.0)
    # the reward uses the unclipped action: pow(a, 2) * 0.1 of an f32 is exact in f64 before the * 0.1
    _, r, _, _ = M.env_step(cfg, np.array([-0.5, 0.0]), 3.0)
    assert r == -(9.0 * 0.1)
    # the left wall: velocity becomes +0.0
    s, _, _, _ = M.env_step(cfg, np.array([-1.2, -0.03]), -1.0)
    assert s[0] == -1.2 and _bits(s[1]) == _bits(0.0)
    # the goal: done, reward 100 - 0.1 a^2
    s, r, term, _ = M.env_step(cfg, np.array([0.449, 0.07]), 0.5)
    assert term and s[0] >= 0.45 and r == 100.0 - (0.5 * 0.5) * 0.1
    # velocity -0.0 at the goal line counts as >= goal_velocity (0)
    env = Continuous_MountainCarEnv((0.45, -0.0))
    assert bool(-0.0 >= env.goal_velocity)


def test_env_step_nan_action_passes_the_clip():
    """max(nan, -1.0) is nan in Python: a NaN action makes the velocity NaN (and the done test False), in both restatements."""
    cfg = M.config()
    s, r, term, _ = M.env_step(cfg, np.array([-0.5, 0.01]), float("nan"))
    gs, gr, gdone, _ = Continuous_MountainCarEnv((-0.5, 0.01)).step(np.array([np.nan], np.float32))
    assert np.isnan(s).all() and np.isnan(gs).all() and np.isnan(r) and np.isnan(gr) and not term and not gdone


def near_goal_roots(B, seed=3):
    rng = np.random.default_rng(seed)
    return np.stack([rng.uniform(0.40, 0.45, B), rng.uniform(0.0, 0.07, B)], 1)


def valley_roots(B, seed=4):
    rng = np.random.default_rng(seed)
    return np.stack([rng.uniform(-0.6, -0.4, B), np.zeros(B)], 1)


def mcc_config(**kw):
    d = dict(n_rollouts=100, num_components=2, n_hidden=2, activation=azo.ACT_RELU)
    d.update(kw)
    return M.config(**d)


def mcc_weights(cfg, seed=34):
    from alphazero_gym_b200.network import init_policy_weights
    return init_policy_weights(seed, cfg.state_dim, cfg.hidden, cfg.n_hidden, cfg.head_dim)


def test_oracle_search_terminal_paths():
    """Near the goal the search expands terminal nodes (V = 0, r = (100 - 0.1 a^2) / 16.2736044), and later simulations that
    select an existing terminal node back it up again (counters[6]) with the same return: W of a terminal edge is its r added
    n times, in order."""
    cfg = mcc_config()
    w = mcc_weights(cfg)
    roots = near_goal_roots(64)
    out = M.search(cfg, w, roots, n_threads=4)
    assert out["counters"][6] > 0
    term = out["terminal"].astype(bool)
    assert term.sum() > 0 and not term[:, 0].any()  # the root is never terminal, even at the goal
    a = out["action"][term].astype(np.float64)
    assert np.array_equal(out["V"][term], np.zeros(term.sum(), np.float32))
    assert np.array_equal(out["r"][term], (100.0 - (a * a) * 0.1) / R_SCALE)
    assert (out["state"][term][:, 0] >= 0.45).all() and (out["state"][term][:, 1] >= 0).all()
    revisited = term & (out["en"] > 1)
    assert revisited.any()
    for b, row in zip(*np.nonzero(revisited)):
        W = 0.0
        for _ in range(out["en"][b, row]):
            W = W + out["r"][b, row]
        assert out["eW"][b, row] == W
    # non-terminal expanded rows: the raw reward is -0.1 a^2
    live = (out["expanded"] == 1) & ~term
    live[:, 0] = False
    a = out["action"][live].astype(np.float64)
    assert np.array_equal(out["r"][live], (0.0 - (a * a) * 0.1) / R_SCALE)


def test_oracle_search_valley_roots_and_state_dim():
    cfg = mcc_config(n_rollouts=50)
    out = M.search(cfg, mcc_weights(cfg), valley_roots(16), n_threads=4)
    assert out["counts"].sum() == 16 * 50
    assert (out["state"][:, 0] == valley_roots(16)).all()
    with pytest.raises(ValueError):  # the env needs state_dim 2
        M.search(mcc_config(state_dim=3), mcc_weights(mcc_config(state_dim=3)), valley_roots(2))


def test_oracle_selfplay_reset():
    """Env.reset of the oracle's self-play loop: position -0.6 + (-0.4 - -0.6) u from Philox stream 3, velocity +0."""
    from oracle import selfplay as SP
    cfg = mcc_config(n_rollouts=10)
    roots = near_goal_roots(8)
    steps = M.selfplay_run(cfg, mcc_weights(cfg), roots, steps=3, max_episode_length=2, seed=5)
    for k, rec in enumerate(steps):
        key = SP.step_seed(5, k)
        for t in np.nonzero(rec["done"])[0]:
            u = SP._unit(azo.rng_u32(key, t, 3, int(rec["episode"][t]), 0, 0))
            assert rec["env_state"][t, 0] == -0.6 + (-0.4 - -0.6) * u and _bits(rec["env_state"][t, 1]) == _bits(0.0)
            assert -0.6 <= rec["env_state"][t, 0] <= -0.4
    assert any(r["done"].any() for r in steps)
    assert steps[0]["obs"].shape == (8, 2) and np.array_equal(steps[0]["obs"], roots.astype(np.float32))


def test_engine_config_and_env_recognition():
    from alphazero_gym_b200 import _cabi
    from alphazero_gym_b200._cabi import CONTINUOUS, DISCRETE
    from alphazero_gym_b200.engine import MOUNTAIN_CAR_CONTINUOUS, PENDULUM, EngineConfig
    from alphazero_gym_b200.search.mcts import continuous_env, env_hidden_state, reward_model
    from alphazero_gym_b200.selfplay import initial_states

    c = EngineConfig(variant=CONTINUOUS, state_dim=2, num_components=1, env=MOUNTAIN_CAR_CONTINUOUS, action_bound=1.0)
    assert c.c().flags & _cabi.FLAG_ENV_MOUNTAIN_CAR_CONTINUOUS and c.is_fused()
    p = EngineConfig(variant=CONTINUOUS, state_dim=3)
    assert not p.c().flags & _cabi.FLAG_ENV_MOUNTAIN_CAR_CONTINUOUS and p.env_name() == PENDULUM and p.is_fused()
    assert not EngineConfig(variant=CONTINUOUS, state_dim=3, env=MOUNTAIN_CAR_CONTINUOUS).is_fused()
    with pytest.raises(ValueError):
        EngineConfig(variant=CONTINUOUS, env="MountainCar-v0").c()

    class TimeLimit:
        def __init__(self, env):
            self.env = env

    class ReparametrizeWrapper(TimeLimit):
        pass

    class MountainCarEnv:  # gym's discrete MountainCar-v0: 3 actions, not served
        state = np.zeros(2)

    env = Continuous_MountainCarEnv((-0.5, 0.0))
    assert np.array_equal(env_hidden_state(TimeLimit(env), CONTINUOUS), [-0.5, 0.0])
    assert continuous_env(TimeLimit(env)) == MOUNTAIN_CAR_CONTINUOUS
    assert reward_model(TimeLimit(env), CONTINUOUS) == (1.0, 1.0)
    with pytest.raises(NotImplementedError):
        reward_model(ReparametrizeWrapper(env), CONTINUOUS)
    with pytest.raises(TypeError):
        env_hidden_state(env, DISCRETE)
    for variant in (DISCRETE, CONTINUOUS):
        with pytest.raises(TypeError):
            env_hidden_state(MountainCarEnv(), variant)
    s = initial_states(CONTINUOUS, 6, seed=9, tree_id0=2, total=10, env=MOUNTAIN_CAR_CONTINUOUS)
    rng = np.random.default_rng(9)
    assert np.array_equal(s, np.stack([rng.uniform(-0.6, -0.4, 10), np.zeros(10)], 1)[2:8])


def test_mountain_car_dispatch_tables_have_gpu_cases():
    """Every MountainCarContinuous instantiation in engine.cu's dispatch tables runs in tests/test_mountain_car_gpu.py."""
    import os
    import test_mountain_car_gpu as G
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = open(os.path.join(root, "alphazero_gym_b200", "csrc", "engine.cu")).read()

    def table(macro):
        return {tuple(int(v) for v in c) for c in re.findall(r"\b" + macro + r"\((\d+), (\d+)\)", src)}

    assert table("FUSED_MCC_CASE") == table("QMLP_MCC_CASE") == set(G.Q8_SHAPES)
    assert table("MLP_MCC_CASE") == set(G.FP32_SHAPES)
