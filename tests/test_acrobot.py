"""Acrobot-v1 on the CPU: the CPU reference's env (tests/acrobot_oracle.c) against gym's step() restated in plain Python, the wrap
cap, its discrete search over three actions through ties, epsilon picks, terminal nodes and visit counts past 255, the self-play
reset and observation rows, and the host-side plumbing that selects the env (no GPU needed)."""
import itertools
import math
import re

import numpy as np
import pytest

from oracle import azo
import acrobot_oracle as M
from acrobot_oracle import AcrobotEnv, WrapCapReached, det_cos, det_sin

PI = np.pi


def edge_cases():
    """(state, action) pairs: random states in gym's box with all three actions, wraps in each direction and over several turns, angles
    landing on +-pi, both velocity bounds hit and exceeded, states on both sides of the terminal line, signed zeros and NaN."""
    rng = np.random.default_rng(8)
    n = 300
    box = np.stack([rng.uniform(-PI, PI, n), rng.uniform(-PI, PI, n), rng.uniform(-4 * PI, 4 * PI, n), rng.uniform(-9 * PI, 9 * PI, n)], 1)
    out = [(tuple(s), int(a)) for s, a in zip(box, rng.integers(0, 3, n))]
    for s in itertools.product((-PI, 0.0, PI), (-PI, PI), (-4 * PI, 4 * PI), (-9 * PI, 9 * PI)):  # the box's corners
        out += [(s, a) for a in range(3)]
    out += [((3.0, 3.0, 12.0, 28.0), 2), ((-3.0, -3.0, -12.0, -28.0), 0)]          # wraps in each direction
    out += [((300.0, -300.0, 0.0, 0.0), 1), ((20.0, -20.0, 5.0, -5.0), 1)]         # several turns (300 rad: 48 turns)
    out += [((PI, -PI, 0.0, 0.0), 1), ((-PI, PI, -0.0, 0.0), 1), ((PI, PI, 0.0, -0.0), 1)]
    out += [((0.0, 0.0, 13.0, 0.0), 1), ((0.0, 0.0, -13.0, 0.0), 1), ((0.0, 0.0, 0.0, 29.0), 1), ((0.0, 0.0, 0.0, -29.0), 1),
            ((0.0, 0.0, 4 * PI, 9 * PI), 1), ((0.0, 0.0, -4 * PI, -9 * PI), 1)]
    out += [((PI - 0.2, 0.0, 0.0, 0.0), a) for a in range(3)]                       # near the top: terminal or just short of it
    out += [((2.3, 0.2, 0.1, 0.0), 1), ((2.2, 0.1, 0.2, 0.1), 2), ((-2.25, -0.15, -0.1, 0.0), 0)]
    out += [((0.0, 0.0, 0.0, 0.0), a) for a in range(3)] + [((-0.0, -0.0, -0.0, -0.0), 1)]
    out += [((np.nan, 0.0, 0.0, 0.0), 1), ((0.0, np.nan, 0.0, 0.0), 0), ((0.0, 0.0, np.nan, 0.0), 2), ((0.0, 0.0, 0.0, np.nan), 1)]
    return out


def _bits(x):
    return np.asarray(x, np.float64).view(np.uint64)


def same(a, b):
    """Bit for bit, except that any NaN equals any NaN (the sign and payload of a NaN differ between x86, the GPU and numpy)."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    nan = np.isnan(a)
    return bool(np.array_equal(nan, np.isnan(b)) and np.array_equal(_bits(a[~nan]), _bits(b[~nan])))


def same32(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    nan = np.isnan(a)
    return bool(np.array_equal(nan, np.isnan(b)) and np.array_equal(a[~nan].view(np.uint32), b[~nan].view(np.uint32)))


def terminal_line(s):
    return -math.cos(s[0]) - math.cos(s[1] + s[0])


@pytest.mark.parametrize("math_mode", [azo.MATH_LIBM, azo.MATH_DET])
def test_env_step_equals_gym_restatement(math_mode):
    """acrobot_oracle.env_step == AcrobotEnv.step bit for bit (state, reward, done, observation) with the same sin / cos."""
    cfg = M.config()
    cfg.math_mode = math_mode
    sin, cos = (math.sin, math.cos) if math_mode == azo.MATH_LIBM else (det_sin, det_cos)
    n_done = n_wrap = n_bound = n_nan = 0
    for s, a in edge_cases():
        nxt, r, term, obs = M.env_step(cfg, np.array(s, np.float64), a)
        env = AcrobotEnv(s, sin=sin, cos=cos)
        gob, gr, gdone, _ = env.step(a)
        assert same(nxt, env.state), (s, a, nxt, env.state)
        assert _bits(r) == _bits(gr) and r == (0.0 if gdone else -1.0), (s, a)
        assert term == gdone, (s, a)
        assert same32(obs, gob.astype(np.float32)), (s, a)
        n_done += term
        n_bound += abs(env.state[2]) == 4 * PI or abs(env.state[3]) == 9 * PI
        n_nan += bool(np.isnan(env.state).any())
        pre = np.asarray(s[:2])
        n_wrap += bool(np.isfinite(pre).all() and (np.abs(pre) > 2.5).any())
    assert n_done >= 5 and n_bound >= 8 and n_nan == 4 and n_wrap >= 10


def test_wrap_bound_and_terminal_edges():
    # wrap: gym's loops, each direction and several turns; +-pi stay; NaN passes
    assert M.wrap(PI + 0.5, -PI, PI) == (PI + 0.5) - 2 * PI and M.wrap(-PI - 0.5, -PI, PI) == (-PI - 0.5) + 2 * PI
    x = 40.0
    while x > PI:
        x = x - (PI - -PI)
    assert M.wrap(40.0, -PI, PI) == x and M.wrap(PI, -PI, PI) == PI and M.wrap(-PI, -PI, PI) == -PI
    assert np.isnan(M.wrap(np.nan, -PI, PI))
    # bound: both limits, exactly and beyond; -0 stays -0; NaN passes
    assert M.bound(13.0, -4 * PI, 4 * PI) == 4 * PI and M.bound(-13.0, -4 * PI, 4 * PI) == -4 * PI
    assert M.bound(4 * PI, -4 * PI, 4 * PI) == 4 * PI and _bits(M.bound(-0.0, -1.0, 1.0)) == _bits(-0.0)
    assert np.isnan(M.bound(np.nan, -1.0, 1.0))
    # the engine's restatement agrees at those points (through a step whose velocities are large)
    cfg = M.config()
    s, _, _, _ = M.env_step(cfg, np.array([0.0, 0.0, 20.0, -40.0]), 1)
    assert s[2] == 4 * PI and s[3] == -9 * PI
    # the terminal line `> 1.`: approached from both sides by bisection on theta1 with theta2 = 0 (-2 cos(theta1) = 1 at 2 pi / 3)
    lo, hi = 2.0, 2.2
    for _ in range(60):
        mid = (lo + hi) / 2
        ns = AcrobotEnv((mid, 0.0, 0.0, 0.0), sin=det_sin, cos=det_cos)
        ns.step(1)
        if ns._terminal():
            hi = mid
        else:
            lo = mid
    for th, want in ((lo, False), (hi, True)):
        _, r, term, _ = M.env_step(cfg, np.array([th, 0.0, 0.0, 0.0]), 1)
        assert term == want and r == (0.0 if want else -1.0)


def test_wrap_cap():
    """A huge finite angle reaches the cap in the C reference and in the restatement; the in-box maximum is far below it."""
    cfg = M.config()
    for s in ((1e6, 0.0, 0.0, 0.0), (0.0, -1e6, 0.0, 0.0), (0.0, 1e12, 0.0, 0.0)):
        with pytest.raises(WrapCapReached):
            M.env_step(cfg, np.array(s), 1)
        with pytest.raises(WrapCapReached):
            AcrobotEnv(s, sin=det_sin, cos=det_cos).step(1)
    # 63 turns pass, the pre-wrap angle at 64 turns + pi does not
    assert M.wrap(PI + 63.5 * (2 * PI), -PI, PI) < PI
    with pytest.raises(WrapCapReached):
        M.wrap(PI + 64.5 * (2 * PI), -PI, PI)
    # the measurement DESIGN.md records: pre-wrap |angle| over gym's box (random states and the corners, all three torques)
    env = AcrobotEnv(sin=np.sin, cos=np.cos)
    rng = np.random.default_rng(0)
    n = 200000
    S = np.stack([rng.uniform(-PI, PI, n), rng.uniform(-PI, PI, n), rng.uniform(-4 * PI, 4 * PI, n), rng.uniform(-9 * PI, 9 * PI, n)])
    corners = np.array(list(itertools.product((-PI, 0.0, PI), (-PI, 0.0, PI), (-4 * PI, 4 * PI), (-9 * PI, 9 * PI)))).T
    S = np.concatenate([S, corners], 1)
    f = lambda y: np.array(env._dsdt(y, 0)[:4] + (np.zeros(y.shape[1]),))  # noqa: E731
    worst = 0.0
    for a in (-1.0, 0.0, 1.0):
        y0 = np.concatenate([S, np.full((1, S.shape[1]), a)])
        k1 = f(y0); k2 = f(y0 + 0.1 * k1); k3 = f(y0 + 0.1 * k2); k4 = f(y0 + 0.2 * k3)  # noqa: E702
        worst = max(worst, float(np.abs((y0 + 0.2 / 6.0 * (k1 + 2 * k2 + 2 * k3 + k4))[:2]).max()))
    assert 20.0 < worst < PI + 5 * 2 * PI  # 26.26 rad measured: under 5 turns, the cap is 64


def roots(kind, B, seed=3):
    rng = np.random.default_rng(seed)
    if kind == "goal":  # near the terminal line: theta1 around 2 pi / 3 .. pi, swinging up
        return np.stack([rng.uniform(1.9, 2.6, B), rng.uniform(-0.3, 0.3, B), rng.uniform(0.0, 1.0, B), rng.uniform(-0.5, 0.5, B)], 1)
    return rng.uniform(-0.1, 0.1, (B, 4))  # Env.reset's distribution


def weights(cfg, seed=34):
    from alphazero_gym_b200.network import init_policy_weights
    return init_policy_weights(seed, cfg.state_dim, cfg.hidden, cfg.n_hidden, cfg.head_dim)


def zero_head(cfg, w):
    """All head weights and biases zero: uniform priors and V = 0 at every node, so the three scores tie at every fresh node."""
    w = w.copy()
    w[-(1 + cfg.hidden + cfg.head_dim * cfg.hidden + cfg.head_dim):] = 0.0
    return w


def test_oracle_search_ties_and_terminals():
    """Near the goal: terminal expansions (V = 0, r = 0), traces that end on an existing terminal node (counters[6]), and three-way
    ties resolved by the random pick among the winners."""
    cfg = M.config(n_rollouts=50, epsilon=0.0)
    w = zero_head(cfg, weights(cfg))
    out = M.search(cfg, w, roots("goal", 64), n_threads=4)
    assert out["counters"][6] > 0
    term = out["terminal"].astype(bool)
    assert term.any() and not term[:, 0].any()
    assert (out["V"][term] == 0).all() and (out["r"][term] == 0.0).all()
    assert (out["prior"][:, 0] == np.float32(1 / 3)).all()
    assert set(out["paction"][:, 1].tolist()) == {0, 1, 2}
    assert out["counters"][2] == 3 * out["counters"][1]
    live = np.arange(out["r"].shape[1])[None, :] < out["n_nodes"][:, None]
    live[:, 0] = False
    assert (out["r"][live & ~term] == -1.0).all()
    # the dump keeps the hidden state: the root's is the root, a child's is one step of it
    rs = roots("goal", 64)
    assert np.array_equal(out["state"][:, 0], rs)
    a = int(out["paction"][0, 1])
    assert np.array_equal(out["state"][0, 1], M.env_step(cfg, rs[0], a)[0])


def test_oracle_search_epsilon_and_deep_counts():
    """epsilon = 0.25 makes random picks of every action; N = 300 pushes the root's visit count past 255."""
    cfg = M.config(n_rollouts=300, epsilon=0.25, V_target_policy="on_policy", gamma=0.99)
    out = M.search(cfg, weights(cfg), roots("reset", 8), n_threads=4)
    assert out["counts"].sum() == 8 * 300 and out["node_n"][:, 0].max() == 300
    assert (out["en"][:, 0] > 0).all() and out["counters"][5] == 2 * out["counters"][1]
    tot = out["counts"].sum(1).astype(np.float64)
    v = np.zeros(8)
    for a in range(3):
        v = v + (out["counts"][:, a] / tot) * out["Q"][:, a]
    assert np.array_equal(v, out["V_target"])


def test_oracle_search_wrap_cap():
    cfg = M.config(n_rollouts=10)
    rs = roots("reset", 4)
    rs[2, 0] = 1e6
    with pytest.raises(WrapCapReached):
        M.search(cfg, weights(cfg), rs)


def test_oracle_selfplay_reset_and_obs_rows():
    from oracle import selfplay as SP
    cfg = M.config(n_rollouts=10)
    cfg.math_mode = azo.MATH_DET
    r0 = roots("goal", 8)
    steps = M.selfplay_run(cfg, weights(cfg), r0, steps=3, max_episode_length=2, seed=5)
    for k, rec in enumerate(steps):
        key = SP.step_seed(5, k)
        for t in np.nonzero(rec["done"])[0]:
            want = [-0.1 + (0.1 - -0.1) * SP._unit(azo.rng_u32(key, t, 3, int(rec["episode"][t]), 0, w)) for w in range(4)]
            assert np.array_equal(rec["env_state"][t], want)
    assert any(r["done"].any() for r in steps) and steps[0]["obs"].shape == (8, 6)
    start = r0[0]
    want = np.array([det_cos(start[0]), det_sin(start[0]), det_cos(start[1]), det_sin(start[1]), start[2], start[3]]).astype(np.float32)
    assert np.array_equal(steps[0]["obs"][0], want)
    assert np.array_equal(steps[1]["obs"], M.observe(cfg, steps[0]["env_state"]))
    assert set(np.concatenate([r["action_taken"] for r in steps]).tolist()) <= {0.0, 1.0, 2.0}


def test_engine_config_and_env_recognition():
    from alphazero_gym_b200 import _cabi
    from alphazero_gym_b200._cabi import CONTINUOUS, DISCRETE
    from alphazero_gym_b200.engine import ACROBOT, CARTPOLE, EngineConfig
    from alphazero_gym_b200.search.mcts import acrobot_obs, discrete_env, env_hidden_state, reward_model
    from alphazero_gym_b200.selfplay import initial_states
    from mc_oracle import MountainCarEnv

    c = EngineConfig(variant=DISCRETE, num_actions=3, state_dim=6, env=ACROBOT)
    assert c.c().flags & _cabi.FLAG_ENV_ACROBOT and _cabi.FLAG_ENV_ACROBOT == 64 and c.is_fused()
    assert not c.c().flags & (_cabi.FLAG_ENV_MOUNTAIN_CAR | _cabi.FLAG_ENV_MOUNTAIN_CAR_CONTINUOUS)
    assert not EngineConfig(variant=DISCRETE, state_dim=4, num_actions=3, env=ACROBOT).is_fused()
    assert not EngineConfig(variant=DISCRETE).c().flags & _cabi.FLAG_ENV_ACROBOT
    assert _cabi.AZG_EWRAP == -6
    with pytest.raises(ValueError):
        EngineConfig(variant=CONTINUOUS, env=ACROBOT).c()

    class TimeLimit:
        def __init__(self, env):
            self.env = env

    class ScaleRewardWrapper(TimeLimit):
        pass

    env = AcrobotEnv((0.05, -0.02, 0.01, 0.03))
    assert discrete_env(TimeLimit(env)) == ACROBOT and discrete_env(object()) == CARTPOLE
    assert np.array_equal(env_hidden_state(TimeLimit(env), DISCRETE, env_id=ACROBOT), [0.05, -0.02, 0.01, 0.03])
    assert np.array_equal(acrobot_obs(env.state), [np.cos(0.05), np.sin(0.05), np.cos(-0.02), np.sin(-0.02), 0.01, 0.03])
    with pytest.raises(TypeError):
        env_hidden_state(env, CONTINUOUS)
    with pytest.raises(TypeError):
        env_hidden_state(MountainCarEnv((-0.5, 0.0)), DISCRETE, env_id=ACROBOT)
    with pytest.raises(TypeError):
        env_hidden_state(env, CONTINUOUS, env_id=ACROBOT)
    assert reward_model(TimeLimit(env), DISCRETE) == (1.0, 1.0)
    with pytest.raises(NotImplementedError):
        reward_model(ScaleRewardWrapper(env), DISCRETE)
    s = initial_states(DISCRETE, 6, seed=9, tree_id0=2, total=10, env=ACROBOT)
    assert np.array_equal(s, np.random.default_rng(9).uniform(-0.1, 0.1, size=(10, 4))[2:8])


def test_dropin_refusals_without_gpu():
    """MCTSDiscrete: Acrobot with num_actions other than 3 raises before any engine exists."""
    from alphazero_gym_b200.search.mcts import MCTSDiscrete
    for na in (2, 4):
        m = MCTSDiscrete(model=None, num_actions=na, n_rollouts=8, c_uct=1.5, gamma=1.0, epsilon=0.0, V_target_policy="off_policy",
                         device="cuda:0", root_state=None)
        with pytest.raises(ValueError):
            m.search(AcrobotEnv())


def test_dispatch_tables_have_gpu_cases():
    """Every Acrobot instantiation in engine.cu's dispatch tables runs in tests/test_acrobot_gpu.py."""
    import os
    import test_acrobot_gpu as G
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = open(os.path.join(root, "alphazero_gym_b200", "csrc", "engine.cu")).read()

    def table(macro):
        return {tuple(int(v) for v in c) for c in re.findall(r"\b" + macro + r"\((\d+), (\d+)\)", src)}

    assert table("FUSED_AC_CASE") == table("QMLP_AC_CASE") == set(G.Q8_SHAPES)
    assert table("MLP_AC_CASE") == set(G.FP32_SHAPES)
