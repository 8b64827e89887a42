"""MountainCar-v0 search on the GPU (AZG_FLAG_ENV_MOUNTAIN_CAR) against the CPU oracle's
discrete search with this env: the env step, every search schedule (one launch per simulation with FP32 and tensor-core evaluation,
the two-phase and the warpgroup whole-search kernels), the MT19937 and tape modes, sharding, self-play and the drop-in classes.
Everything bit for bit on the tree dump, the root results and counters[:7]: same Philox streams, same deterministic cosine, same
evaluation arithmetic, same three-way selection and tie-break."""
import numpy as np
import pytest

from oracle import azo
from oracle import selfplay as osp
from classic_control import MountainCarEnv, det_cos
from parity import assert_tree_equal

SMS = 148  # B200

# the MountainCar instantiations of engine.cu (tests/test_mountain_car_discrete.py checks the tables against these)
FP32_SHAPES = [(H, a) for H in (128, 64) for a in range(6)]                      # k_mlp<H, 2, ACT>: MLP_MCC_CASE(H, ACT)
Q8_SHAPES = [(a, nl) for a in (azo.ACT_RELU, azo.ACT_ELU) for nl in (1, 2)]   # k_qmlp2 / k_search_wg: *_MC_CASE(ACT, NL)


def roots(kind, B, seed=3):
    rng = np.random.default_rng(seed)
    if kind == "goal":
        return np.stack([rng.uniform(0.42, 0.5, B), rng.uniform(0.0, 0.07, B)], 1)
    return np.stack([rng.uniform(-0.6, -0.4, B), np.zeros(B)], 1)  # Env.reset's distribution


def mc_config(act=azo.ACT_RELU, L=2, N=50, q8=False, hidden=128, **kw):
    d = dict(n_rollouts=N, n_hidden=L, activation=act, hidden=hidden, epsilon=0.0)
    d.update(kw)
    cfg = azo.discrete_config(azo.MOUNTAIN_CAR, **d)
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
    return E.run_engine(cfg, w, rs, kernel=True, **kw)


def take(out, lo, hi):
    return {k: (v[lo:hi] if isinstance(v, np.ndarray) and v.ndim >= 1 and k != "counters" else v) for k, v in out.items()}


def check_full(cfg, w, rs, out, root_n=None):
    ref = azo.search(cfg, w, rs, root_n, n_threads=8)
    assert_tree_equal(out, ref, discrete=True)
    assert np.array_equal(out["counters"][:7], ref["counters"][:7]), (out["counters"], ref["counters"])
    return ref


def check_slices(cfg, w, rs, out, n=256):
    B = rs.shape[0]
    for lo, hi in ((0, n), (B - n, B)):
        ref = azo.search(cfg, w, rs[lo:hi], tree_id0=lo, n_threads=8)
        assert_tree_equal(take(out, lo, hi), ref, discrete=True)


# ------------------------------------------------------------------------------------------------------------------ env step

@pytest.mark.gpu
def test_env_step_equals_oracle_and_gym():
    import test_mountain_car_discrete as T
    from alphazero_gym_b200.engine import MOUNTAIN_CAR, EngineConfig, SearchEngine
    from alphazero_gym_b200._cabi import DISCRETE
    cases = T.edge_cases()
    s = np.array([c[0] for c in cases], np.float64)
    a = np.array([c[1] for c in cases], np.float32)
    eng = SearchEngine(EngineConfig(variant=DISCRETE, num_actions=3, state_dim=2, env=MOUNTAIN_CAR, max_trees=1))
    try:
        nxt, rew, term, obs = eng.env_step(s, a)
    finally:
        eng.close()
    cfg = mc_config()
    assert obs.shape == (len(cases), 2) and nxt.shape == (len(cases), 2)
    for i in range(len(cases)):
        rn, rr, rt, ro = azo.env_step(cfg, s[i], int(a[i]))
        gs, gr, gd, _ = MountainCarEnv(s[i], cos=det_cos).step(int(a[i]))
        for ref_s, ref_r, ref_t in ((rn, rr, rt), (gs, gr, gd)):
            assert np.array_equal(nxt[i].view(np.uint64), np.asarray(ref_s, np.float64).view(np.uint64)), (s[i], a[i])
            assert rew[i] == ref_r == -1.0 and bool(term[i]) == bool(ref_t)
        assert np.array_equal(obs[i].view(np.uint32), ro.view(np.uint32))
    assert term.sum() >= 8


# ------------------------------------------------------------------------------------------------------------------ searches

@pytest.mark.gpu
@pytest.mark.parametrize("H,act", FP32_SHAPES)
def test_fp32_per_simulation(H, act):
    """Every k_mlp<H, 2, ACT> instantiation inside a search, one launch per simulation."""
    cfg = mc_config(act, 2, 50, hidden=H)
    w = weights(cfg, seed=H + act)
    rs = roots(("goal", "valley")[act % 2], 40, seed=H + act)
    out = run(cfg, w, rs, fused=False)
    assert out["kernel"] == "none" and out["counters"][7] > 50
    check_full(cfg, w, rs, out)


@pytest.mark.gpu
@pytest.mark.parametrize("act,nl", Q8_SHAPES)
@pytest.mark.parametrize("kind,N", [("goal", 50), ("valley", 200), ("goal", 300)])
def test_q8_per_simulation(act, nl, kind, N):
    cfg = mc_config(act, nl + 1, N, q8=True)
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
@pytest.mark.parametrize("case", ["ties", "eps_onpolicy_gamma", "greedy"])
@pytest.mark.parametrize("fused", [False, True])
def test_search_options(case, fused):
    """Forced three-way ties (all-zero head), epsilon = 0.25 with the on-policy target and gamma < 1, the greedy target."""
    kw = {"ties": dict(), "eps_onpolicy_gamma": dict(epsilon=0.25, V_target_policy="on_policy", gamma=0.97),
          "greedy": dict(V_target_policy="greedy", epsilon=0.1)}[case]
    cfg = mc_config(azo.ACT_RELU, 2, 100, q8=True, **kw)
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
    kind, N = ("goal", "valley")[nl - 1], (50, 100)[act]
    cfg = mc_config(act, nl + 1, N, q8=True, epsilon=0.1)
    w = weights(cfg, seed=nl)
    rs = roots(kind, 4096, seed=act + nl)
    out = run(cfg, w, rs)
    assert out["kernel"] == "two_phase" and out["counters"][7] == 1
    check_slices(cfg, w, rs, out)


@pytest.mark.gpu
@pytest.mark.parametrize("act,nl", Q8_SHAPES)
def test_warpgroup_search(act, nl):
    kind, N = ("goal", "valley")[(act + nl) % 2], (100, 50)[act]
    cfg = mc_config(act, nl + 1, N, q8=True)
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
    cfg = mc_config(azo.ACT_ELU, 3, 100, q8=True, rng_mode=azo.RNG_MT19937, epsilon=0.25)
    w = weights(cfg)
    rs = roots("goal", 48, seed=11)
    out = run(cfg, w, rs, rng_mt19937=True, fused=fused)
    assert out["kernel"] == ("two_phase" if fused else "none")
    check_full(cfg, w, rs, out)


@pytest.mark.gpu
def test_tape_mode():
    cfg = mc_config(azo.ACT_RELU, 2, 100, use_eval_tape=1, epsilon=0.1)
    B = 48
    rng = np.random.default_rng(5)
    p = rng.uniform(0.01, 1.0, (B, cfg.rows, 3)).astype(np.float32)
    tapes = {"V": rng.uniform(-30, 0, (B, cfg.rows)).astype(np.float32), "prior": p / p.sum(-1, keepdims=True)}
    rs = roots("goal", B, seed=12)
    import enginelib as E
    out = E.run_engine(cfg, None, rs, tapes=tapes)
    ref = azo.search(cfg, None, rs, tapes=tapes, n_threads=8)
    assert_tree_equal(out, ref, discrete=True)
    assert np.array_equal(out["counters"][:4], ref["counters"][:4]) and out["counters"][6] == ref["counters"][6] > 0


@pytest.mark.gpu
def test_shard_offset_and_root_n():
    cfg = mc_config(azo.ACT_ELU, 3, 100, q8=True, epsilon=0.1)
    w = weights(cfg)
    rs = roots("valley", 1024, seed=13)
    rn = np.random.default_rng(1).integers(0, 40, 1024).astype(np.int32)
    full = run(cfg, w, rs, root_n_init=rn)
    lo, hi = 300, 812
    part = run(cfg, w, rs[lo:hi], root_n_init=rn[lo:hi], tree_id0=lo)
    assert_tree_equal(take(full, lo, hi), part, discrete=True)
    halves = [run(cfg, w, rs[a:b], root_n_init=rn[a:b], tree_id0=a) for a, b in ((0, 512), (512, 1024))]
    for k in ("counts", "Q", "V_target", "eW", "en", "node_n"):
        assert np.array_equal(np.concatenate([h[k] for h in halves]), full[k]), k
    ref = azo.search(cfg, w, rs[lo:lo + 64], rn[lo:lo + 64], tree_id0=lo, n_threads=8)
    assert_tree_equal(take(full, lo, lo + 64), ref, discrete=True)


@pytest.mark.gpu
def test_nan_weights_raise():
    from alphazero_gym_b200._cabi import AzgError
    cfg = mc_config(azo.ACT_RELU, 2, 20)
    w = weights(cfg)
    w[:] = np.nan
    with pytest.raises(AzgError):
        run(cfg, w, roots("valley", 8), fused=False)


# ------------------------------------------------------------------------------------------------------------------ self-play

@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["det", "t05", "t1", "t2", "value"])
def test_selfplay_equals_oracle(mode):
    import enginelib as E
    from alphazero_gym_b200.selfplay import SelfPlayDriver
    det, by_value, temp = mode == "det", mode == "value", {"t05": 0.5, "t2": 2.0, "value": 2.0}.get(mode, 1.0)
    cfg = mc_config(azo.ACT_RELU, 2, 30, q8=True)
    w = weights(cfg)
    B, steps, max_len = 64, 8, 4
    states0 = roots("goal", B, seed=21)
    ref = osp.run(cfg, w, states0, steps, max_len, seed=cfg.seed, tree_id0=7, deterministic=det, by_value=by_value,
                         temperature=temp)
    eng = E.SearchEngine(E.engine_config(cfg, B))
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
    from alphazero_gym_b200.search.mcts import MCTSDiscrete
    from alphazero_gym_b200.train import LossConfig, Trainer
    cfg = mc_config(azo.ACT_RELU, 2, 50, q8=True)
    w = weights(cfg)
    model = PolicyNet(2, cfg.hidden, cfg.n_hidden, 3, "relu", num_actions=3).load_flat(w).cuda()
    root = roots("goal", 2, seed=31)
    mcts = MCTSDiscrete(model=model, num_actions=3, n_rollouts=50, c_uct=cfg.c_uct, gamma=cfg.gamma, epsilon=0.0,
                        V_target_policy="off_policy", device="cuda:0", root_state=None, seed=cfg.seed)
    mcts.search(Env=TimeLimit(MountainCarEnv(root[0])))
    state, actions, counts, Q, V = mcts.return_results("max_visit")
    ref = azo.search(cfg, w, root[:1], tree_id0=0)
    assert np.array_equal(state, root[0]) and np.array_equal(actions, [0, 1, 2])
    assert np.array_equal(counts, ref["counts"][0]) and np.array_equal(Q, ref["Q"][0]) and V == ref["V_target"][0]
    a = int(counts.argmax())
    nxt, _, _, _ = azo.env_step(cfg, root[0], a)
    mcts.forward(a, nxt)
    assert mcts.root_node is not None and mcts.root_node.n == ref["node_n"][0, ref["echild"][0, 0, a]]
    agent = DiscreteAgent.from_modules(model, MCTSDiscrete(model=model, num_actions=3, n_rollouts=50, c_uct=cfg.c_uct, gamma=cfg.gamma,
                                                           epsilon=0.0, V_target_policy="off_policy", device="cuda:0",
                                                           root_state=None, seed=cfg.seed))
    action, s2, acts, cnts, Qs, V2 = agent.act(TimeLimit(MountainCarEnv(root[1])))
    ref2 = azo.search(cfg, w, root[1:2], tree_id0=0)
    assert np.array_equal(cnts, ref2["counts"][0]) and np.array_equal(Qs, ref2["Q"][0]) and 0 <= int(action) < 3
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
    from alphazero_gym_b200._cabi import CONTINUOUS, DISCRETE, AzgError
    from alphazero_gym_b200.engine import MOUNTAIN_CAR, EngineConfig, SearchEngine
    for bad in (EngineConfig(variant=DISCRETE, num_actions=2, state_dim=2, env=MOUNTAIN_CAR),
                EngineConfig(variant=DISCRETE, num_actions=3, state_dim=4, env=MOUNTAIN_CAR),
                EngineConfig(variant=DISCRETE, num_actions=3, state_dim=2),          # 3 actions without the flag
                EngineConfig(variant=DISCRETE, num_actions=3, state_dim=2, env=MOUNTAIN_CAR, max_rollouts=16383)):
        with pytest.raises(AzgError):
            SearchEngine(bad)
    eng = SearchEngine(EngineConfig(variant=DISCRETE, num_actions=3, state_dim=2, env=MOUNTAIN_CAR, max_rollouts=16382))
    try:
        with pytest.raises(AzgError):
            eng.set_reward_model(0.005, -1.0)
        eng.set_reward_model(1.0, 1.0)
    finally:
        eng.close()
