"""Hidden widths other than 64 / 128 on the GPU: the streamed FP32 evaluation kernel k_mlp_stream<S, ACT> (mlp_stream.cuh) against
the CPU oracle (bit for bit) and the f64 evaluation (f64ref.py), then through every layer above it: searches of every env with the
full tree dump compared, the MT19937 mode, batches of several passes per CTA, self-play, the drop-in classes with a make_policy
model, and the widths and flags azg_create refuses.

The case tables (STREAM_SHAPES, ENVS) are torch-free: test_wide_trunk.py checks them against engine.cu on machines without a GPU.
"""
import numpy as np
import pytest

from oracle import azo
import f64ref as F
import test_kernel_matrix_gpu as M

SMS = 148  # B200
SMEM_OPTIN = 232448  # B200: dynamic shared memory a block may opt in to
ACTS = M.ACTS
WIDTHS = (32, 96, 160, 192, 224, 256)  # every streamed width the tests cover (64 and 128 run k_mlp)

# k_mlp_stream<S, ACT>: every instantiation of engine.cu MLP_STREAM_CASE (S = 2 both MountainCars, 3 Pendulum, 4 CartPole, 6 Acrobot)
STREAM_SHAPES = [(S, a) for S in (4, 3, 2, 6) for a in ACTS]
# the envs by input width, with their head sizes (discrete: A; continuous: the mixture components K)
ENVS = {"CartPole-v0": (4, (0,)), "Pendulum-v0": (3, tuple(range(1, 9))), "MountainCar-v0": (2, (0,)),
        "MountainCarContinuous-v0": (2, tuple(range(1, 9))), "Acrobot-v1": (6, (0,))}
DISCRETE_ENVS = ("CartPole-v0", "MountainCar-v0", "Acrobot-v1")


def make_cfg(env, act, n_hidden, K=0, hidden=256, **kw):
    """Oracle config of `env` with the FP32 evaluation and the deterministic math of the engine."""
    name = None if env in ("CartPole-v0", "Pendulum-v0") else env
    if env in DISCRETE_ENVS:
        cfg = azo.discrete_config(name, hidden=hidden, n_hidden=n_hidden, activation=act, **kw)
    else:
        cfg = azo.continuous_config(name, hidden=hidden, n_hidden=n_hidden, activation=act, num_components=K, **kw)
    cfg.eval_mode, cfg.math_mode = azo.EVAL_FP32, azo.MATH_DET
    return cfg


def observations(cfg, n, seed=0):
    """Observations in the env's range, then M.observations' edge rows (zero, +-big, 1e-30)."""
    if cfg.env is None:
        return M.observations(cfg, n, seed)
    rng = np.random.default_rng(seed)
    if cfg.state_dim == 2:  # position, velocity of both MountainCars
        x = np.stack([rng.uniform(-1.2, 0.6, n), rng.uniform(-0.07, 0.07, n)], 1)
    else:  # Acrobot: cos, sin of both angles, both velocities
        t1, t2 = rng.uniform(-np.pi, np.pi, n), rng.uniform(-np.pi, np.pi, n)
        x = np.stack([np.cos(t1), np.sin(t1), np.cos(t2), np.sin(t2), rng.uniform(-4 * np.pi, 4 * np.pi, n),
                      rng.uniform(-9 * np.pi, 9 * np.pi, n)], 1)
    x = x.astype(np.float32)
    big = 10.0 if cfg.activation == azo.ACT_HARDSWISH else 1e4
    edges = [np.zeros(cfg.state_dim), np.full(cfg.state_dim, big) * (-1) ** np.arange(cfg.state_dim), np.full(cfg.state_dim, 1e-30),
             -np.full(cfg.state_dim, big)]
    for i, e in enumerate(edges[:n]):
        x[i] = e
    return x


def stream_smem(H, S, P, RP):
    """mlp_stream.cuh mlp_stream_smem_bytes: ring of 4 slices of 8 k-rows, layer 0, heads, activations, head outputs, inputs, leaf
    words (4 B) and leafR (8 B) per row, nine mbarriers."""
    po = (1 + P + 3) // 4 * 4
    return 4 * (4 * 8 * H + S * H + H + H * po + po + H * RP + po * RP + S * RP + RP) + 8 * RP + 72


def rows_per_pass(cfg, smem_optin=SMEM_OPTIN):
    """engine.cu azg_create: up to 16 warps of 64 x 32 tiles; as many 64-row blocks per pass as shared memory holds."""
    H = cfg.hidden
    rb = max(1, 16 // (H // 32))
    while rb > 1 and stream_smem(H, cfg.state_dim, cfg.head_dim, 64 * rb) > smem_optin:
        rb -= 1
    return 64 * rb


def _forward_cases(env, act):
    """Every width x depth with the env's default head and default weights; x10 / edge / dead weights at one depth per width; the
    other head sizes of a continuous env spread over the widths."""
    S, heads = ENVS[env]
    K0 = 2 if heads != (0,) else 0
    for i, H in enumerate(WIDTHS):
        for L in (1, 2, 3, 4):
            kinds = ("default", "x10", "edge", "dead") if L == 2 + i % 3 else ("default",)
            yield H, L, K0, kinds
            for K in heads:
                if K not in (0, K0) and (K + L) % len(WIDTHS) == i:
                    yield H, L, K, ("default",)


def _sample_rows(n, R):
    """Rows compared with the oracle out of n: the first and last two passes' worth (CTA boundaries, the ragged last pass) and a
    stride through the rest."""
    idx = np.concatenate([np.arange(min(n, 2 * R + 2)), np.arange(max(0, n - 2 * R - 2), n), np.arange(0, n, 97)])
    return np.unique(idx)


def check_forward(cfg, weight_sets):
    """azg_mlp_forward at the row counts 1, 31, 32, 33, R - 1, R, R + 1 and 148 R + 5 (R = rows per pass): V and the post-processed
    head bit-identical to the oracle on the sampled rows; the first 64 rows inside the f64 bound."""
    import enginelib as E
    R = rows_per_pass(cfg)
    counts = (1, 31, 32, 33, R - 1, R, R + 1, SMS * R + 5)
    x = observations(cfg, counts[-1], seed=cfg.hidden + cfg.n_hidden + cfg.num_components)
    eng = E.SearchEngine(E.engine_config(cfg, 4, eval_q8=False, fused=False))
    try:
        for kind, w in weight_sets:
            eng.set_weights(w)
            runs = {n: eng.mlp_forward(x[:n]) for n in counts}
            rows = _sample_rows(counts[-1], R)
            Vo, raw = azo.mlp_forward(cfg, w, x[rows])
            post = np.stack([azo.head_post(cfg, r) for r in raw])
            name = f"{cfg.env} H={cfg.hidden} act={cfg.activation} L={cfg.n_hidden} K={cfg.num_components} {kind}"
            for n, (V, head) in runs.items():
                sel = rows < n
                assert np.array_equal(V[rows[sel]], Vo[sel]), f"{name} n={n}: V differs from the oracle"
                assert np.array_equal(head[rows[sel]], post[sel]), f"{name} n={n}: head differs from the oracle"
            ref = F.forward(cfg, w, x[:64])
            V, head = runs[counts[-1]]
            for what, got, r, b in (("V", V[:64], ref["V"], ref["bV"]), ("head", head[:64], ref["post"], ref["bpost"])):
                ok, ratio = F.within(got, r, b)
                assert ok, f"{name}: {what} outside the f64 bound (worst |err| / bound = {ratio:.3g})"
    finally:
        eng.close()


@pytest.mark.gpu
@pytest.mark.parametrize("S,act", STREAM_SHAPES)
def test_streamed_evaluation_kernel_matrix(S, act):
    """k_mlp_stream<S, ACT> for every streamed width, n_hidden 1-4 and every head size of the envs with S inputs."""
    n = 0
    for env in (e for e, (s, _) in ENVS.items() if s == S):
        for H, L, K, kinds in _forward_cases(env, act):
            cfg = make_cfg(env, act, L, K, hidden=H)
            check_forward(cfg, [(k, M.weights(cfg, k)) for k in kinds])
            n += 1
    assert n >= 24


# ------------------------------------------------------------------------------------------------------------------ searches


def _roots(env, B, seed=34):
    if env in ("CartPole-v0", "Pendulum-v0"):
        return M.roots_for(make_cfg(env, 0, 2, 1), B, seed)
    rng = np.random.default_rng(seed)
    if env == "Acrobot-v1":
        return rng.uniform(-0.1, 0.1, (B, 4))
    return np.stack([rng.uniform(-0.6, -0.4, B), rng.uniform(-0.02, 0.02, B)], 1)  # both MountainCars, near Env.reset


SEARCHES = {  # id: (env, activation, n_hidden, K, hidden, trees, n_rollouts, extra config)
    "cartpole_eps_reuse": ("CartPole-v0", azo.ACT_RELU, 2, 0, 256, 64, 60, dict(epsilon=0.1)),
    "mountain_car": ("MountainCar-v0", azo.ACT_RELU, 2, 0, 256, 48, 50, {}),
    "acrobot": ("Acrobot-v1", azo.ACT_ELU, 2, 0, 256, 40, 50, {}),
    "pendulum_k1": ("Pendulum-v0", azo.ACT_ELU, 3, 1, 256, 48, 40, {}),
    "pendulum_k2": ("Pendulum-v0", azo.ACT_ELU, 3, 2, 256, 48, 40, {}),
    "pendulum_k3": ("Pendulum-v0", azo.ACT_SILU, 2, 3, 256, 48, 40, {}),
    "pendulum_k4": ("Pendulum-v0", azo.ACT_ELU, 4, 4, 256, 48, 40, {}),
    "mountain_car_continuous": ("MountainCarContinuous-v0", azo.ACT_RELU, 2, 2, 256, 48, 40, {}),
    "cartpole_192": ("CartPole-v0", azo.ACT_LEAKYRELU, 3, 0, 192, 64, 40, dict(epsilon=0.1)),
    "cartpole_mt19937": ("CartPole-v0", azo.ACT_RELU, 2, 0, 256, 40, 40, dict(epsilon=0.25, rng_mode=azo.RNG_MT19937)),
    "pendulum_mt19937": ("Pendulum-v0", azo.ACT_ELU, 3, 2, 256, 40, 30, dict(rng_mode=azo.RNG_MT19937)),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(SEARCHES))
def test_search_at_wide_trunk(case):
    """One launch per simulation with the streamed evaluation: tree dump, root results and counters bit-identical to the oracle,
    the stored evaluations inside the f64 bound (CartPole, Pendulum)."""
    env, act, L, K, H, B, N, kw = SEARCHES[case]
    cfg = make_cfg(env, act, L, K, hidden=H, n_rollouts=N, **kw)
    w = M.weights(cfg, "x10" if case == "pendulum_k3" else "default", seed=L + K)
    roots = _roots(env, B, seed=len(case))
    rn = None
    if case == "cartpole_eps_reuse":  # a tree carried over by forward(): the root keeps its visit count
        rn = np.random.default_rng(2).integers(0, 30, B).astype(np.int32)
    out, _ = M.run_search(cfg, w, roots, "per_simulation", rn)
    assert out["counters"][7] > N
    if env in ("CartPole-v0", "Pendulum-v0"):
        M.check_stored_evaluation(cfg, w, out)


@pytest.mark.gpu
def test_search_batch_of_several_passes():
    """More trees than one pass of every SM (148 R + 5 at hidden 192): CTAs evaluate several passes, the last one ragged; the root
    results of the whole batch and counters equal the oracle's."""
    cfg = make_cfg("Pendulum-v0", azo.ACT_ELU, 2, 2, hidden=192, n_rollouts=6)
    B = SMS * rows_per_pass(cfg) + 5
    w = M.weights(cfg)
    M.run_search(cfg, w, _roots("Pendulum-v0", B, seed=7), "per_simulation", tree_id0=5, dump=False)


# ------------------------------------------------------------------------------------------------------------------ self-play


@pytest.mark.gpu
@pytest.mark.parametrize("env", ["CartPole-v0", "Pendulum-v0"])
def test_selfplay_at_wide_trunk(env):
    """azg_selfplay_step at hidden 256 equals the oracle's episode loop, every array of every step."""
    from oracle import gen_golden as G, selfplay as osp
    import test_selfplay_gpu as SP
    if env == "CartPole-v0":
        cfg = make_cfg(env, azo.ACT_RELU, 2, hidden=256, n_rollouts=16, epsilon=0.1)
        B, steps, max_len, states0 = 48, 7, 4, G.cartpole_roots(48, seed=5)
    else:
        cfg = make_cfg(env, azo.ACT_ELU, 3, 2, hidden=256, n_rollouts=20)
        B, steps, max_len, states0 = 32, 6, 3, G.pendulum_roots(32, seed=5)
    cfg.use_eval_tape = 0
    w = M.weights(cfg)
    ref = osp.run(cfg, w, states0, steps, max_len, seed=cfg.seed, tree_id0=7)
    got, _, _ = SP._run_engine(cfg, w, states0, steps, max_len, tree_id0=7)
    SP._compare(got, ref, cfg.cmax)
    assert sum(int(r["done"].sum()) for r in ref) >= B


# ------------------------------------------------------------------------------------------------------------------ drop-in


@pytest.mark.gpu
def test_dropin_discrete_make_policy_256():
    """MCTSDiscrete and DiscreteAgent with make_policy(hidden_dimensions=[256, 256]): search, return_results, forward with the root
    count carried, act, and one Trainer.update whose weights reach the engine, each equal to the oracle."""
    import torch
    from alphazero_gym_b200.agent.agents import DiscreteAgent
    from alphazero_gym_b200.network import describe_model, make_policy
    from alphazero_gym_b200.search.mcts import MCTSDiscrete
    from alphazero_gym_b200.train import LossConfig, Trainer
    from oracle.ref_harness import CartPoleEnv
    torch.manual_seed(3)
    model = make_policy(4, 1, "discrete", [256, 256], "relu", num_actions=2)
    assert describe_model(model)["hidden"] == 256
    cfg = make_cfg("CartPole-v0", azo.ACT_RELU, 2, hidden=256, n_rollouts=30, epsilon=0.1)
    w = azo.flatten_state_dict(model.state_dict())
    root = _roots("CartPole-v0", 2, seed=11)
    env = CartPoleEnv(root[0])
    mcts = MCTSDiscrete(model=model, num_actions=2, n_rollouts=30, c_uct=cfg.c_uct, gamma=cfg.gamma, epsilon=0.1,
                        V_target_policy="off_policy", device="cuda:0", root_state=np.array(env.state), seed=cfg.seed)
    eng = mcts._engine(1)
    assert not eng.cfg.is_q8() and not eng.cfg.is_fused()
    mcts.search(Env=env)
    state, actions, counts, Q, V = mcts.return_results("max_visit")
    ref = azo.search(cfg, w, root[:1])
    assert np.array_equal(counts, ref["counts"][0]) and np.array_equal(Q, ref["Q"][0]) and V == ref["V_target"][0]
    a = int(np.argmax(counts))
    obs, _, _, _ = env.step(a)
    mcts.forward(a, obs)
    assert mcts.root_node is not None
    n0 = mcts.root_node.n
    mcts.search(Env=env)
    _, _, counts2, Q2, _ = mcts.return_results("max_visit")
    ref2 = azo.search(cfg, w, np.array(env.state)[None], np.array([n0], np.int32), tree_id0=1)
    assert np.array_equal(counts2, ref2["counts"][0]) and np.array_equal(Q2, ref2["Q"][0])
    # the agent (its search is the object's third: tree id 2)
    agent = DiscreteAgent.from_modules(model, mcts)
    agent.reset_mcts(root_state=root[1])
    env2 = CartPoleEnv(root[1])
    act_, s2, acts, cnts, Qs, V2 = agent.act(env2)
    ref3 = azo.search(cfg, w, root[1:2], tree_id0=2)
    assert np.array_equal(cnts, ref3["counts"][0]) and np.array_equal(Qs, ref3["Q"][0]) and act_ in (0, 1)
    # one Trainer.update on those rows, then the new weights reach the engine
    model.cuda()
    batch = {"obs": torch.tensor(np.stack([state, s2]), dtype=torch.float32, device="cuda"),
             "actions": torch.tensor(np.stack([actions, acts]), dtype=torch.float32, device="cuda"),
             "counts": torch.tensor(np.stack([counts, cnts]), dtype=torch.int32, device="cuda"),
             "V_target": torch.tensor([V, V2], dtype=torch.float64, device="cuda")}
    tr = Trainer(model, LossConfig(tuned=False), optimizer="adam")
    before = tr.flat_weights().clone()
    losses = tr.update(batch)
    assert all(torch.isfinite(v).all() for v in losses.values())
    after = tr.flat_weights()
    assert not torch.equal(before, after)
    eng = mcts._engine(1)
    tr.push_weights(eng, broadcast=False)
    eng.search(torch.from_numpy(root[:1]).cuda(), 30)
    eng.status()
    got = eng.root_results()
    ref4 = azo.search(cfg, after.cpu().numpy(), root[:1], tree_id0=0)
    assert np.array_equal(got["counts"].cpu().numpy()[0, :2], ref4["counts"][0])
    mcts.close()


@pytest.mark.gpu
def test_dropin_continuous_make_policy_256():
    """MCTSContinuous and ContinuousAgent with make_policy(hidden_dimensions=[256, 256, 256]) (a GMM head of 2 components):
    search, return_results and act equal the oracle."""
    import torch
    from alphazero_gym_b200.agent.agents import ContinuousAgent
    from alphazero_gym_b200.network import describe_model, make_policy
    from alphazero_gym_b200.search.mcts import MCTSContinuous
    from oracle.ref_harness import PendulumEnv
    torch.manual_seed(4)
    model = make_policy(3, 1, "normal", [256, 256, 256], "elu", num_components=2, action_bound=2.0)
    d = describe_model(model)
    assert d["hidden"] == 256 and d["n_hidden"] == 3
    cfg = make_cfg("Pendulum-v0", azo.ACT_ELU, 3, 2, hidden=256, n_rollouts=25)
    w = azo.flatten_state_dict(model.state_dict())
    root = _roots("Pendulum-v0", 2, seed=12)
    env = PendulumEnv(root[0])
    mcts = MCTSContinuous(model=model, n_rollouts=25, c_uct=cfg.c_uct, c_pw=cfg.c_pw, kappa=cfg.kappa, gamma=cfg.gamma, epsilon=0,
                          V_target_policy="off_policy", device="cuda:0", root_state=env.obs(), seed=cfg.seed)
    mcts.search(Env=env)
    state, actions, counts, Q, V = mcts.return_results("max_visit")
    ref = azo.search(cfg, w, root[:1])
    C = int(ref["n_children"][0])
    assert np.array_equal(state, env.obs()) and actions.shape == (C,)
    assert np.array_equal(counts, ref["counts"][0, :C]) and np.array_equal(Q, ref["Q"][0, :C]) and V == ref["V_target"][0]
    assert np.array_equal(actions, ref["actions"][0, :C])
    agent = ContinuousAgent.from_modules(model, mcts)
    env2 = PendulumEnv(root[1])
    agent.reset_mcts(root_state=env2.obs())
    action, _, acts, cnts, Qs, _ = agent.act(env2)
    ref2 = azo.search(cfg, w, root[1:2], tree_id0=1)
    C2 = int(ref2["n_children"][0])
    assert np.array_equal(cnts, ref2["counts"][0, :C2]) and np.array_equal(Qs, ref2["Q"][0, :C2])
    assert action[0] == acts[cnts.argmax()]
    mcts.close()


# ------------------------------------------------------------------------------------------------------------------ refusals


@pytest.mark.gpu
def test_refusals():
    """Widths that are not a multiple of 32 or exceed 256, and the tensor-core evaluation or the whole-search kernel at a streamed
    width, raise AzgError; every streamed width is accepted for both variants."""
    from alphazero_gym_b200._cabi import AzgError
    from alphazero_gym_b200.engine import EngineConfig, SearchEngine
    from alphazero_gym_b200._cabi import CONTINUOUS, DISCRETE
    for variant, sd in ((DISCRETE, 4), (CONTINUOUS, 3)):
        for H in (100, 288, 512, 16, 0):
            with pytest.raises(AzgError):
                SearchEngine(EngineConfig(variant=variant, state_dim=sd, hidden=H, eval_q8=False, fused=False))
        for kw in (dict(eval_q8=True, fused=False), dict(eval_q8=True, fused=True), dict(eval_q8=False, fused=True)):
            with pytest.raises(AzgError):
                SearchEngine(EngineConfig(variant=variant, state_dim=sd, hidden=256, **kw))
        for H in WIDTHS:
            for L in (1, 4):
                SearchEngine(EngineConfig(variant=variant, state_dim=sd, hidden=H, n_hidden=L, num_components=8)).close()
