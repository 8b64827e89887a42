"""MountainCarContinuous-v0 search on the GPU (AZG_FLAG_ENV_MOUNTAIN_CAR_CONTINUOUS) against the CPU oracle's
search with this env: the env step, every
search schedule (one launch per simulation with FP32 and tensor-core evaluation, the two-phase and the warpgroup whole-search
kernels), the MT19937 and tape modes, sharding, self-play and the drop-in classes.  Everything bit for bit: same Philox streams,
same deterministic cosine, same evaluation arithmetic.  Roots near the goal make the search expand terminal nodes (V = 0) and
back up existing ones again, the continuous tree's terminal paths that Pendulum never reaches."""
import numpy as np
import pytest

from oracle import azo
from oracle import selfplay as osp
from classic_control import Continuous_MountainCarEnv, det_cos
from parity import assert_tree_equal

SMS = 148  # B200

# the MountainCarContinuous instantiations of engine.cu (tests/test_mountain_car.py checks the tables against these)
FP32_SHAPES = [(H, a) for H in (128, 64) for a in range(6)]                      # k_mlp<H, 2, ACT>: MLP_MCC_CASE(H, ACT)
Q8_SHAPES = [(a, nl) for a in (azo.ACT_RELU, azo.ACT_ELU) for nl in (1, 2)]   # k_qmlp2 / k_search_wg: *_MCC_CASE(ACT, NL)

# (K, activation, n_hidden) x (roots, N) for the per-simulation schedules; N = 200 reaches the root fan-out of 15
SHAPES = [(K, a, L) for K in (1, 2, 3) for a in (azo.ACT_RELU, azo.ACT_ELU) for L in (2, 3)]
ROOTS_N = [("valley", 100), ("goal", 100), ("goal", 200), ("valley", 200)]
PER_SIM = [s + r for s in SHAPES for r in ROOTS_N[:3]] + [SHAPES[5] + ROOTS_N[3]]
# the whole-search kernels, one case per (K, activation, n_hidden), roots and N alternating
FUSED = [s + ROOTS_N[i % 4] for i, s in enumerate(SHAPES)]


def roots(kind, B, seed=3):
    rng = np.random.default_rng(seed)
    if kind == "goal":
        return np.stack([rng.uniform(0.40, 0.45, B), rng.uniform(0.0, 0.07, B)], 1)
    return np.stack([rng.uniform(-0.6, -0.4, B), np.zeros(B)], 1)  # Env.reset's distribution


def mcc_config(K=2, act=azo.ACT_RELU, L=2, N=100, q8=False, hidden=128, **kw):
    cfg = azo.continuous_config(azo.MOUNTAIN_CAR_CONTINUOUS, n_rollouts=N, num_components=K, n_hidden=L, activation=act, hidden=hidden, **kw)
    cfg.math_mode, cfg.eval_mode = azo.MATH_DET, (azo.EVAL_Q8 if q8 else azo.EVAL_FP32)
    return cfg


def weights(cfg, seed=34):
    from alphazero_gym_b200.network import init_policy_weights
    return init_policy_weights(seed, cfg.state_dim, cfg.hidden, cfg.n_hidden, cfg.head_dim)


def run(cfg, w, rs, **kw):
    import enginelib as E
    return E.run_engine(cfg, w, rs, kernel=True, **kw)


def oracle_slice(cfg, w, rs, lo, hi, **kw):
    return azo.search(cfg, w, rs[lo:hi], tree_id0=lo, n_threads=8, **kw)


def take(out, lo, hi):
    return {k: (v[lo:hi] if isinstance(v, np.ndarray) and v.ndim >= 1 and k != "counters" else v) for k, v in out.items()}


def fit(out, ref):
    import enginelib as E
    for k in ("actions", "counts", "Q"):
        out[k] = E.fit_columns(out[k], ref[k].shape[1])
    return out


def check_full(cfg, w, rs, out):
    """dump + results + counters[:7] of the whole batch bit for bit."""
    ref = azo.search(cfg, w, rs, n_threads=8)
    assert_tree_equal(fit(out, ref), ref, discrete=False)
    assert np.array_equal(out["counters"][:7], ref["counters"][:7]), (out["counters"], ref["counters"])
    return ref


def check_slices(cfg, w, rs, out, n=256):
    """A large batch: the first and the last n trees (dump + results) bit for bit against the oracle run on those trees alone."""
    B = rs.shape[0]
    for lo, hi in ((0, n), (B - n, B)):
        ref = oracle_slice(cfg, w, rs, lo, hi)
        assert_tree_equal(fit(take(out, lo, hi), ref), ref, discrete=False)


# ------------------------------------------------------------------------------------------------------------------ env step

@pytest.mark.gpu
def test_env_step_equals_oracle_and_gym():
    import test_mountain_car as T
    from alphazero_gym_b200.engine import MOUNTAIN_CAR_CONTINUOUS, EngineConfig, SearchEngine
    from alphazero_gym_b200._cabi import CONTINUOUS
    cases = T.edge_cases()
    s = np.array([c[0] for c in cases], np.float64)
    a = np.array([c[1] for c in cases], np.float32)
    eng = SearchEngine(EngineConfig(variant=CONTINUOUS, state_dim=2, num_components=1, env=MOUNTAIN_CAR_CONTINUOUS, action_bound=1.0,
                                    max_trees=1))
    try:
        nxt, rew, term, obs = eng.env_step(s, a)
    finally:
        eng.close()
    cfg = mcc_config()
    assert obs.shape == (len(cases), 2)
    for i in range(len(cases)):
        rn, rr, rt, ro = azo.env_step(cfg, s[i], float(a[i]))
        gs, gr, gd, _ = Continuous_MountainCarEnv(s[i], cos=det_cos).step(a[i:i + 1])
        for ref_s, ref_r, ref_t in ((rn, rr, rt), (gs, gr, gd)):
            assert np.array_equal(nxt[i].view(np.uint64), np.asarray(ref_s, np.float64).view(np.uint64)), (s[i], a[i])
            assert rew[i:i + 1].view(np.uint64)[0] == np.float64(ref_r).view(np.uint64), (s[i], a[i], rew[i], ref_r)
            assert bool(term[i]) == bool(ref_t)
        assert np.array_equal(obs[i].view(np.uint32), ro.view(np.uint32))
    assert term.sum() >= 10
    # under math.cos instead of the deterministic cosine, gym differs by at most rounding
    for i in range(len(cases)):
        gs, gr, _, _ = Continuous_MountainCarEnv(s[i]).step(a[i:i + 1])
        assert np.allclose(nxt[i], gs, rtol=1e-13, atol=1e-16, equal_nan=True)


# ------------------------------------------------------------------------------------------------------------------ searches

@pytest.mark.gpu
@pytest.mark.parametrize("K,act,L,kind,N", PER_SIM)
@pytest.mark.parametrize("q8", [False, True])
def test_per_simulation_search(K, act, L, kind, N, q8):
    cfg = mcc_config(K, act, L, N, q8)
    w = weights(cfg, seed=K + 10 * L)
    rs = roots(kind, 48, seed=N + K)
    out = run(cfg, w, rs, fused=False)
    assert out["kernel"] == "none" and out["counters"][7] > N
    ref = check_full(cfg, w, rs, out)
    if kind == "goal":
        assert ref["terminal"].any() and ref["counters"][6] > 0
    if N == 200:
        assert ref["n_children"].max() == 15


@pytest.mark.gpu
@pytest.mark.parametrize("H,act", FP32_SHAPES)
def test_fp32_evaluation_shapes(H, act):
    """Every k_mlp<H, 2, ACT> instantiation inside a search (one launch per simulation)."""
    cfg = mcc_config(1, act, 2, 50, hidden=H)
    w = weights(cfg)
    rs = roots("goal", 40, seed=H + act)
    out = run(cfg, w, rs)
    assert out["kernel"] == "none"
    check_full(cfg, w, rs, out)


@pytest.mark.gpu
@pytest.mark.parametrize("K,act,L,kind,N", FUSED)
def test_two_phase_search(K, act, L, kind, N):
    cfg = mcc_config(K, act, L, N, q8=True)
    w = weights(cfg, seed=K)
    rs = roots(kind, 4096, seed=K + N)
    out = run(cfg, w, rs)
    assert out["kernel"] == "two_phase" and out["counters"][7] == 1
    check_slices(cfg, w, rs, out)


@pytest.mark.gpu
@pytest.mark.parametrize("act,nl", Q8_SHAPES)
def test_warpgroup_search(act, nl):
    K, kind, N = 1 + (act + 2 * nl) % 3, ("goal", "valley")[nl - 1], (100, 200)[act]
    cfg = mcc_config(K, act, nl + 1, N, q8=True)
    w = weights(cfg, seed=nl)
    B = 65536
    assert B >= 3 * 128 * SMS  # at least three full tiles per SM: the warpgroup kernel's range
    rs = roots(kind, B, seed=act + nl)
    out = run(cfg, w, rs)
    assert out["kernel"] == "warpgroups" and out["counters"][7] == 1
    check_slices(cfg, w, rs, out)
    if kind == "goal":
        assert out["terminal"].any() and out["counters"][6] > 0


@pytest.mark.gpu
def test_mt19937_mode():
    cfg = mcc_config(2, azo.ACT_ELU, 3, 100, rng_mode=azo.RNG_MT19937, epsilon=0.1)
    w = weights(cfg)
    rs = roots("goal", 48, seed=11)
    out = run(cfg, w, rs, rng_mt19937=True)
    assert out["kernel"] == "none"
    check_full(cfg, w, rs, out)


@pytest.mark.gpu
def test_tape_mode():
    cfg = mcc_config(2, azo.ACT_RELU, 2, 100, use_eval_tape=1)
    B = 48
    rng = np.random.default_rng(5)
    tapes = {"V": rng.uniform(-1, 1, (B, cfg.rows)).astype(np.float32), "action": rng.uniform(-1.2, 1.2, (B, cfg.rows)).astype(np.float32)}
    rs = roots("goal", B, seed=12)
    import enginelib as E
    out = E.run_engine(cfg, None, rs, tapes=tapes)
    ref = azo.search(cfg, None, rs, tapes=tapes, n_threads=8)
    assert_tree_equal(fit(out, ref), ref, discrete=False, skip=("head",))
    assert np.array_equal(out["counters"][:4], ref["counters"][:4]) and out["counters"][6] == ref["counters"][6] > 0


@pytest.mark.gpu
def test_shard_with_offset_tree_ids():
    cfg = mcc_config(2, azo.ACT_ELU, 3, 100, q8=True)
    w = weights(cfg)
    rs = roots("goal", 1024, seed=13)
    full = run(cfg, w, rs)
    lo, hi = 300, 812
    part = run(cfg, w, rs[lo:hi], tree_id0=lo)
    assert_tree_equal(take(full, lo, hi), part, discrete=False)


# ------------------------------------------------------------------------------------------------------------------ self-play

@pytest.mark.gpu
@pytest.mark.parametrize("by_value", [False, True])
def test_selfplay_equals_oracle(by_value):
    import enginelib as E
    from alphazero_gym_b200.selfplay import SelfPlayDriver
    cfg = mcc_config(2, azo.ACT_ELU, 3, 30, q8=True)
    w = weights(cfg)
    B, steps, max_len = 64, 8, 4
    states0 = roots("goal", B, seed=21)
    ref = osp.run(cfg, w, states0, steps, max_len, seed=cfg.seed, tree_id0=7, by_value=by_value)
    eng = E.SearchEngine(E.engine_config(cfg, B))
    try:
        eng.set_weights(w)
        drv = SelfPlayDriver(eng, B, cfg.n_rollouts, max_episode_length=max_len, tree_id0=7, seed=cfg.seed,
                             final_selection="max_value" if by_value else "max_visit")
        drv.set_states(states0)
        for s in range(steps):
            t = drv.step()
            eng.status()
            r = ref[s]
            for k in ("obs", "actions", "counts", "Q", "V_target", "n_children", "action_taken", "reward", "done", "ep_step", "episode"):
                a, b = t[k].cpu().numpy(), r[k]
                if a.ndim == 2 and a.shape[1] != b.shape[1]:
                    m = min(a.shape[1], b.shape[1])
                    assert not a[:, m:].any() and not b[:, m:].any()
                    a, b = a[:, :m], b[:, :m]
                assert np.array_equal(a, b), f"step {s}: {k} differs"
            assert np.array_equal(drv.env_state.cpu().numpy(), r["env_state"]), f"step {s}: env_state differs"
    finally:
        eng.close()
    done = np.array([r["done"] for r in ref], bool)
    reward = np.array([r["reward"] for r in ref])
    assert (done & (reward > 50)).any()                 # episodes that end at the goal
    assert (done & (reward < 50)).any()                 # and at max_episode_length
    assert ref[0]["obs"].shape == (B, 2)


# ------------------------------------------------------------------------------------------------------------------ drop-in

def _model(cfg, w):
    from alphazero_gym_b200.network import PolicyNet
    hd = 3 * cfg.num_components if cfg.num_components > 1 else 2
    act = {azo.ACT_RELU: "relu", azo.ACT_ELU: "elu"}[cfg.activation]
    return PolicyNet(2, cfg.hidden, cfg.n_hidden, hd, act, num_components=cfg.num_components, action_bound=1.0).load_flat(w)


@pytest.mark.gpu
def test_dropin_search_agent_and_trainer():
    import torch
    from alphazero_gym_b200.agent.agents import ContinuousAgent
    from alphazero_gym_b200.search.mcts import MCTSContinuous
    from alphazero_gym_b200.train import LossConfig, Trainer
    cfg = mcc_config(2, azo.ACT_ELU, 3, 50, q8=True)
    w = weights(cfg)
    model = _model(cfg, w).cuda()
    root = roots("goal", 2, seed=31)
    env = Continuous_MountainCarEnv(root[0])
    mcts = MCTSContinuous(model=model, n_rollouts=50, c_uct=cfg.c_uct, c_pw=cfg.c_pw, kappa=cfg.kappa, gamma=cfg.gamma, epsilon=0,
                          V_target_policy="off_policy", device="cuda:0", root_state=None, seed=cfg.seed)
    mcts.search(Env=env)
    state, actions, counts, Q, V = mcts.return_results("max_visit")
    ref = azo.search(cfg, w, root[:1], tree_id0=0)
    C = int(ref["n_children"][0])
    assert np.array_equal(state, root[0]) and actions.shape == (C,)
    assert np.array_equal(counts, ref["counts"][0, :C]) and np.array_equal(Q, ref["Q"][0, :C]) and V == ref["V_target"][0]
    assert np.array_equal(actions, ref["actions"][0, :C])
    # the agent: actions[counts.argmax()] of its search (the second search of this object: tree id 1)
    agent = ContinuousAgent.from_modules(model, mcts)
    env2 = Continuous_MountainCarEnv(root[1])
    action, s2, acts, cnts, Qs, V2 = agent.act(env2)
    ref2 = azo.search(cfg, w, root[1:2], tree_id0=1)
    C2 = int(ref2["n_children"][0])
    assert np.array_equal(cnts, ref2["counts"][0, :C2]) and np.array_equal(Qs, ref2["Q"][0, :C2])
    assert action[0] == acts[cnts.argmax()] and np.array_equal(s2, root[1])
    # one Trainer.update on those rows, then the new weights reach the engine
    batch = {"obs": torch.tensor(np.stack([state, s2]), dtype=torch.float32, device="cuda"),
             "actions": torch.tensor(np.stack([actions[:min(C, C2)], acts[:min(C, C2)]]), dtype=torch.float32, device="cuda"),
             "counts": torch.tensor(np.stack([counts[:min(C, C2)], cnts[:min(C, C2)]]), dtype=torch.int32, device="cuda"),
             "V_target": torch.tensor([V, V2], dtype=torch.float64, device="cuda")}
    tr = Trainer(model, LossConfig(tuned=False), optimizer="adam")
    before = tr.flat_weights().clone()
    losses = tr.update(batch)
    assert all(torch.isfinite(v).all() for v in losses.values())
    after = tr.flat_weights()
    assert not torch.equal(before, after)
    eng = mcts._engine(1)
    tr.push_weights(eng, broadcast=False)
    eng.search(torch.from_numpy(root[:1]).cuda(), 50)
    eng.status()
    got = eng.root_results()
    ref3 = azo.search(cfg, after.cpu().numpy(), root[:1], tree_id0=0)
    assert np.array_equal(got["counts"].cpu().numpy()[0, :ref3["counts"].shape[1]], ref3["counts"][0])
    mcts.close()


# ------------------------------------------------------------------------------------------------------------------ refusals

@pytest.mark.gpu
def test_flag_refusals():
    from alphazero_gym_b200._cabi import CONTINUOUS, DISCRETE, AzgError
    from alphazero_gym_b200.engine import MOUNTAIN_CAR_CONTINUOUS, EngineConfig, SearchEngine
    for bad in (EngineConfig(variant=DISCRETE, state_dim=4, env=MOUNTAIN_CAR_CONTINUOUS),
                EngineConfig(variant=DISCRETE, state_dim=2, env=MOUNTAIN_CAR_CONTINUOUS),
                EngineConfig(variant=CONTINUOUS, state_dim=3, env=MOUNTAIN_CAR_CONTINUOUS),
                EngineConfig(variant=CONTINUOUS, state_dim=4, env=MOUNTAIN_CAR_CONTINUOUS),
                EngineConfig(variant=CONTINUOUS, state_dim=2)):  # state_dim 2 without the flag: Pendulum needs 3
        with pytest.raises(AzgError):
            SearchEngine(bad)
