"""Acrobot-v1 search on the GPU (AZG_FLAG_ENV_ACROBOT) against its CPU reference (tests/acrobot_oracle.py: the CPU oracle's discrete
search with this env): the env step, every search schedule (one launch per simulation with FP32 and tensor-core evaluation, the
two-phase and the warpgroup whole-search kernels), the MT19937 and tape modes, sharding, the wrap cap, self-play and the drop-in
classes.  Everything bit for bit on the tree dump, the root results and counters[:7]: same Philox streams, same deterministic sine
and cosine, same RK4, same 6-input evaluation arithmetic, same three-way selection and tie-break."""
import numpy as np
import pytest

from oracle import azo
import acrobot_oracle as M
from acrobot_oracle import AcrobotEnv
from parity import assert_tree_equal

SMS = 148  # B200

# the Acrobot instantiations of engine.cu (tests/test_acrobot.py checks the tables against these)
FP32_SHAPES = [(H, a) for H in (128, 64) for a in range(6)]                      # k_mlp<H, 6, ACT>: MLP_AC_CASE(H, ACT)
Q8_SHAPES = [(a, nl) for a in (azo.ACT_RELU, azo.ACT_ELU) for nl in (1, 2)]   # k_qmlp2 / k_search_wg: *_AC_CASE(ACT, NL)


def roots(kind, B, seed=3):
    rng = np.random.default_rng(seed)
    if kind == "goal":  # near the terminal line
        return np.stack([rng.uniform(1.9, 2.6, B), rng.uniform(-0.3, 0.3, B), rng.uniform(0.0, 1.0, B), rng.uniform(-0.5, 0.5, B)], 1)
    return rng.uniform(-0.1, 0.1, (B, 4))  # Env.reset's distribution


def ac_config(act=azo.ACT_RELU, L=2, N=50, q8=False, hidden=128, **kw):
    d = dict(n_rollouts=N, n_hidden=L, activation=act, hidden=hidden, epsilon=0.0)
    d.update(kw)
    cfg = M.config(**d)
    cfg.math_mode, cfg.eval_mode = azo.MATH_DET, (azo.EVAL_Q8 if q8 else azo.EVAL_FP32)
    return cfg


def weights(cfg, seed=34):
    from alphazero_gym_b200.network import init_policy_weights
    return init_policy_weights(seed, cfg.state_dim, cfg.hidden, cfg.n_hidden, cfg.head_dim)


def zero_head(cfg, w):
    w = w.copy()
    w[-(1 + cfg.hidden + cfg.head_dim * cfg.hidden + cfg.head_dim):] = 0.0
    return w


def run(cfg, w, rs, **kw):
    import enginelib as E
    from alphazero_gym_b200.engine import ACROBOT
    return E.run_engine(cfg, w, rs, env=ACROBOT, kernel=True, **kw)


def take(out, lo, hi):
    return {k: (v[lo:hi] if isinstance(v, np.ndarray) and v.ndim >= 1 and k != "counters" else v) for k, v in out.items()}


def check_full(cfg, w, rs, out, root_n=None):
    ref = M.search(cfg, w, rs, root_n, n_threads=8)
    assert_tree_equal(out, ref, discrete=True)
    assert np.array_equal(out["counters"][:7], ref["counters"][:7]), (out["counters"], ref["counters"])
    return ref


def check_slices(cfg, w, rs, out, n=256):
    B = rs.shape[0]
    for lo, hi in ((0, n), (B - n, B)):
        ref = M.search(cfg, w, rs[lo:hi], tree_id0=lo, n_threads=8)
        assert_tree_equal(take(out, lo, hi), ref, discrete=True)


# ------------------------------------------------------------------------------------------------------------------ env step

@pytest.mark.gpu
def test_env_step_equals_oracle_and_gym():
    import test_acrobot as T
    from alphazero_gym_b200.engine import ACROBOT, EngineConfig, SearchEngine
    from alphazero_gym_b200._cabi import DISCRETE, AzgError
    cases = T.edge_cases()
    s = np.array([c[0] for c in cases], np.float64)
    a = np.array([c[1] for c in cases], np.float32)
    eng = SearchEngine(EngineConfig(variant=DISCRETE, num_actions=3, state_dim=6, env=ACROBOT, max_trees=1))
    try:
        nxt, rew, term, obs = eng.env_step(s, a)
        eng.status()
        with pytest.raises(AzgError):  # a huge finite angle reaches the wrap cap
            eng.env_step(np.array([[1e6, 0.0, 0.0, 0.0]]), np.array([1], np.float32))
            eng.status()
        eng.status()
    finally:
        eng.close()
    cfg = ac_config()
    assert obs.shape == (len(cases), 6) and nxt.shape == (len(cases), 4)
    for i in range(len(cases)):
        rn, rr, rt, ro = M.env_step(cfg, s[i], int(a[i]))
        env = AcrobotEnv(s[i], sin=M.det_sin, cos=M.det_cos)
        gob, gr, gd, _ = env.step(int(a[i]))
        for ref_s, ref_r, ref_t in ((rn, rr, rt), (env.state, gr, gd)):
            assert T.same(nxt[i], ref_s), (s[i], a[i])
            assert rew[i] == ref_r and bool(term[i]) == bool(ref_t)
        assert T.same32(obs[i], ro) and T.same32(obs[i], gob.astype(np.float32))
    assert term.sum() >= 5


# ------------------------------------------------------------------------------------------------------------------ searches

@pytest.mark.gpu
@pytest.mark.parametrize("H,act", FP32_SHAPES)
def test_fp32_per_simulation(H, act):
    """Every k_mlp<H, 6, ACT> instantiation inside a search, one launch per simulation."""
    cfg = ac_config(act, 2, 50, hidden=H)
    w = weights(cfg, seed=H + act)
    rs = roots(("goal", "reset")[act % 2], 40, seed=H + act)
    out = run(cfg, w, rs, fused=False)
    assert out["kernel"] == "none" and out["counters"][7] > 50
    check_full(cfg, w, rs, out)


@pytest.mark.gpu
@pytest.mark.parametrize("act,nl", Q8_SHAPES)
@pytest.mark.parametrize("kind,N", [("goal", 50), ("reset", 300)])
def test_q8_per_simulation(act, nl, kind, N):
    cfg = ac_config(act, nl + 1, N, q8=True)
    w = weights(cfg, seed=act + 10 * nl)
    rs = roots(kind, 32, seed=N + act)
    out = run(cfg, w, rs, fused=False)
    assert out["kernel"] == "none"
    ref = check_full(cfg, w, rs, out)
    if kind == "goal":
        assert ref["terminal"].any() and ref["counters"][6] > 0
    if N == 300:
        assert ref["node_n"][:, 0].max() == 300


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["ties", "eps_onpolicy_gamma"])
@pytest.mark.parametrize("fused", [False, True])
def test_search_options(case, fused):
    """Forced three-way ties (all-zero head), epsilon = 0.25 with the on-policy target and gamma < 1."""
    kw = {"ties": dict(), "eps_onpolicy_gamma": dict(epsilon=0.25, V_target_policy="on_policy", gamma=0.97)}[case]
    cfg = ac_config(azo.ACT_RELU, 2, 100, q8=True, **kw)
    w = weights(cfg)
    if case == "ties":
        w = zero_head(cfg, w)
    rs = roots("goal", 64, seed=5)
    out = run(cfg, w, rs, fused=fused)
    assert out["kernel"] == ("two_phase" if fused else "none")
    ref = check_full(cfg, w, rs, out)
    if case == "ties":
        assert set(ref["paction"][:, 1].tolist()) == {0, 1, 2}


@pytest.mark.gpu
@pytest.mark.parametrize("act,nl", Q8_SHAPES)
def test_two_phase_search(act, nl):
    """4096 trees: the two-phase kernel (kind 1); shared-memory trees are not built for three-action rows."""
    kind, N = ("goal", "reset")[nl - 1], (50, 100)[act]
    cfg = ac_config(act, nl + 1, N, q8=True, epsilon=0.1)
    w = weights(cfg, seed=nl)
    rs = roots(kind, 4096, seed=act + nl)
    out = run(cfg, w, rs)
    assert out["kernel"] == "two_phase" and out["counters"][7] == 1
    check_slices(cfg, w, rs, out)


@pytest.mark.gpu
@pytest.mark.parametrize("act,nl", Q8_SHAPES)
def test_warpgroup_search(act, nl):
    kind, N = ("goal", "reset")[(act + nl) % 2], (100, 50)[act]
    cfg = ac_config(act, nl + 1, N, q8=True)
    w = weights(cfg, seed=nl + 5)
    B = 65536
    assert B >= 3 * 128 * SMS
    rs = roots(kind, B, seed=act + nl)
    out = run(cfg, w, rs)
    assert out["kernel"] == "warpgroups" and out["counters"][7] == 1
    check_slices(cfg, w, rs, out)


@pytest.mark.gpu
@pytest.mark.parametrize("fused", [False, True])
def test_mt19937_mode(fused):
    cfg = ac_config(azo.ACT_ELU, 3, 100, q8=True, rng_mode=azo.RNG_MT19937, epsilon=0.25)
    w = weights(cfg)
    rs = roots("goal", 48, seed=11)
    out = run(cfg, w, rs, rng_mt19937=True, fused=fused)
    assert out["kernel"] == ("two_phase" if fused else "none")
    check_full(cfg, w, rs, out)


@pytest.mark.gpu
def test_tape_mode():
    cfg = ac_config(azo.ACT_RELU, 2, 100, use_eval_tape=1, epsilon=0.1)
    B = 48
    rng = np.random.default_rng(5)
    p = rng.uniform(0.01, 1.0, (B, cfg.rows, 3)).astype(np.float32)
    tapes = {"V": rng.uniform(-30, 0, (B, cfg.rows)).astype(np.float32), "prior": p / p.sum(-1, keepdims=True)}
    rs = roots("goal", B, seed=12)
    import enginelib as E
    from alphazero_gym_b200.engine import ACROBOT
    out = E.run_engine(cfg, None, rs, tapes=tapes, env=ACROBOT)
    ref = M.search(cfg, None, rs, tapes=tapes, n_threads=8)
    assert_tree_equal(out, ref, discrete=True)
    assert np.array_equal(out["counters"][:4], ref["counters"][:4]) and out["counters"][6] == ref["counters"][6] > 0


@pytest.mark.gpu
def test_shard_offset_and_root_n():
    cfg = ac_config(azo.ACT_ELU, 3, 100, q8=True, epsilon=0.1)
    w = weights(cfg)
    rs = roots("reset", 1024, seed=13)
    rn = np.random.default_rng(1).integers(0, 40, 1024).astype(np.int32)
    full = run(cfg, w, rs, root_n_init=rn)
    lo, hi = 300, 812
    part = run(cfg, w, rs[lo:hi], root_n_init=rn[lo:hi], tree_id0=lo)
    assert_tree_equal(take(full, lo, hi), part, discrete=True)
    ref = M.search(cfg, w, rs[lo:lo + 64], rn[lo:lo + 64], tree_id0=lo, n_threads=8)
    assert_tree_equal(take(full, lo, lo + 64), ref, discrete=True)


@pytest.mark.gpu
def test_nan_weights_raise():
    from alphazero_gym_b200._cabi import AzgError
    cfg = ac_config(azo.ACT_RELU, 2, 20)
    w = weights(cfg)
    w[:] = np.nan
    with pytest.raises(AzgError):
        run(cfg, w, roots("reset", 8), fused=False)


@pytest.mark.gpu
@pytest.mark.parametrize("fused", [False, True])
def test_wrap_cap_raises(fused):
    """A large finite root angle: the first expansion from the root reaches the wrap cap, and the search fails with AZG_EWRAP."""
    from alphazero_gym_b200._cabi import AZG_EWRAP, AzgError
    cfg = ac_config(azo.ACT_RELU, 2, 20, q8=True)
    rs = roots("reset", 8)
    rs[3, 1] = -1e6
    with pytest.raises(AzgError) as ei:
        run(cfg, weights(cfg), rs, fused=fused)
    assert ei.value.code == AZG_EWRAP
    with pytest.raises(M.WrapCapReached):
        M.search(cfg, weights(cfg), rs)


# ------------------------------------------------------------------------------------------------------------------ self-play

@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["det", "t1", "value"])
def test_selfplay_equals_oracle(mode):
    import enginelib as E
    from alphazero_gym_b200.engine import ACROBOT
    from alphazero_gym_b200.selfplay import SelfPlayDriver
    det, by_value, temp = mode == "det", mode == "value", {"value": 2.0}.get(mode, 1.0)
    cfg = ac_config(azo.ACT_RELU, 2, 30, q8=True)
    w = weights(cfg)
    B, steps, max_len = 64, 8, 4
    states0 = roots("goal", B, seed=21)
    ref = M.selfplay_run(cfg, w, states0, steps, max_len, seed=cfg.seed, tree_id0=7, deterministic=det, by_value=by_value,
                         temperature=temp)
    eng = E.SearchEngine(E.engine_config(cfg, B, env=ACROBOT))
    try:
        eng.set_weights(w)
        drv = SelfPlayDriver(eng, B, cfg.n_rollouts, max_episode_length=max_len, tree_id0=7, seed=cfg.seed, deterministic=det,
                             final_selection="max_value" if by_value else "max_visit", temperature=temp)
        drv.set_states(states0)
        for s in range(steps):
            t = drv.step()
            eng.status()
            r = ref[s]
            for k in ("obs", "actions", "counts", "Q", "V_target", "n_children", "action_taken", "reward", "done", "ep_step", "episode",
                      "root_n"):
                assert np.array_equal(t[k].cpu().numpy(), r[k]), f"step {s}: {k} differs"
            assert np.array_equal(drv.env_state.cpu().numpy(), r["env_state"]), f"step {s}: env_state differs"
    finally:
        eng.close()
    done = np.array([r["done"] for r in ref], bool)
    before = np.array([np.zeros(B, np.int32)] + [r["ep_step"] for r in ref[:-1]])  # episode step at the start of each step
    assert (done & (before + 1 < max_len)).any()     # episodes that end at the goal
    assert (done & (before + 1 == max_len)).any()    # and at max_episode_length
    assert (np.array([r["root_n"] for r in ref]) > 0).any()  # tree reuse
    assert ref[0]["obs"].shape == (B, 6)


# ------------------------------------------------------------------------------------------------------------------ drop-in

class TimeLimit:
    def __init__(self, env):
        self.env = env

    @property
    def unwrapped(self):
        return self.env


@pytest.mark.gpu
def test_dropin_search_agent_and_trainer():
    import torch
    from alphazero_gym_b200.agent.agents import DiscreteAgent
    from alphazero_gym_b200.network import PolicyNet
    from alphazero_gym_b200.search.mcts import MCTSDiscrete, acrobot_obs
    from alphazero_gym_b200.train import LossConfig, Trainer
    cfg = ac_config(azo.ACT_RELU, 2, 50, q8=True)
    w = weights(cfg)
    model = PolicyNet(6, cfg.hidden, cfg.n_hidden, 3, "relu", num_actions=3).load_flat(w).cuda()
    root = roots("goal", 2, seed=31)
    mcts = MCTSDiscrete(model=model, num_actions=3, n_rollouts=50, c_uct=cfg.c_uct, gamma=cfg.gamma, epsilon=0.0,
                        V_target_policy="off_policy", device="cuda:0", root_state=None, seed=cfg.seed)
    mcts.search(Env=TimeLimit(AcrobotEnv(root[0])))
    state, actions, counts, Q, V = mcts.return_results("max_visit")
    ref = M.search(cfg, w, root[:1], tree_id0=0)
    assert state.shape == (6,) and np.array_equal(state, acrobot_obs(root[0])) and np.array_equal(actions, [0, 1, 2])
    assert np.array_equal(counts, ref["counts"][0]) and np.array_equal(Q, ref["Q"][0]) and V == ref["V_target"][0]
    a = int(counts.argmax())
    env = AcrobotEnv(root[0], sin=np.sin, cos=np.cos)
    ob, _, _, _ = env.step(a)
    mcts.forward(a, ob)  # the agent passes the 6-wide observation
    assert mcts.root_node is not None and mcts.root_node.n == ref["node_n"][0, ref["echild"][0, 0, a]]
    assert np.array_equal(mcts.root_node.state, ob)
    agent = DiscreteAgent.from_modules(model, MCTSDiscrete(model=model, num_actions=3, n_rollouts=50, c_uct=cfg.c_uct, gamma=cfg.gamma,
                                                           epsilon=0.0, V_target_policy="off_policy", device="cuda:0",
                                                           root_state=None, seed=cfg.seed))
    action, s2, acts, cnts, Qs, V2 = agent.act(TimeLimit(AcrobotEnv(root[1])))
    ref2 = M.search(cfg, w, root[1:2], tree_id0=0)
    assert np.array_equal(cnts, ref2["counts"][0]) and np.array_equal(Qs, ref2["Q"][0]) and 0 <= int(action) < 3
    assert np.asarray(s2).shape == (6,)
    batch = {"obs": torch.tensor(np.stack([state, s2]), dtype=torch.float32, device="cuda"),
             "actions": torch.tensor(np.stack([actions, acts]), dtype=torch.float32, device="cuda"),
             "counts": torch.tensor(np.stack([counts, cnts]), dtype=torch.int32, device="cuda"),
             "V_target": torch.tensor([V, V2], dtype=torch.float64, device="cuda")}
    tr = Trainer(model, LossConfig(tuned=False), optimizer="adam")
    before = tr.flat_weights().clone()
    losses = tr.update(batch)
    assert all(torch.isfinite(v).all() for v in losses.values()) and not torch.equal(before, tr.flat_weights())
    mcts.close()


@pytest.mark.gpu
def test_flag_refusals():
    from alphazero_gym_b200 import _cabi
    from alphazero_gym_b200._cabi import DISCRETE, AzgError
    from alphazero_gym_b200.engine import ACROBOT, EngineConfig, SearchEngine
    for bad in (EngineConfig(variant=DISCRETE, num_actions=2, state_dim=6, env=ACROBOT),
                EngineConfig(variant=DISCRETE, num_actions=3, state_dim=4, env=ACROBOT),
                EngineConfig(variant=DISCRETE, num_actions=3, state_dim=6),          # 6 inputs without the flag
                EngineConfig(variant=DISCRETE, num_actions=3, state_dim=6, env=ACROBOT, max_rollouts=16383)):
        with pytest.raises(AzgError):
            SearchEngine(bad)
    import ctypes as C
    lib = _cabi.load()
    for other in (_cabi.FLAG_ENV_MOUNTAIN_CAR, _cabi.FLAG_ENV_MOUNTAIN_CAR_CONTINUOUS):  # the flag combinations no EngineConfig makes
        raw = EngineConfig(variant=DISCRETE, num_actions=3, state_dim=6, env=ACROBOT).c()
        raw.flags |= other
        h = C.c_void_p()
        assert lib.azg_create(C.byref(raw), C.byref(h)) == _cabi.AZG_EINVAL and not h.value
    eng = SearchEngine(EngineConfig(variant=DISCRETE, num_actions=3, state_dim=6, env=ACROBOT, max_rollouts=16382))
    try:
        with pytest.raises(AzgError):
            eng.set_reward_model(0.005, -1.0)
        eng.set_reward_model(1.0, 1.0)
    finally:
        eng.close()
