"""Every kernel template the engine compiles, run against the CPU oracle (bit for bit) and against an f64 evaluation with a
derived error bound (f64ref.py).

* Evaluation kernels (azg_mlp_forward): every k_mlp<H, S, ACT> with n_hidden 1-4 where the network fits in shared memory and
  every head size K 1-8; every k_qmlp2<S, ACT, NL> with K 1-5 (the head sizes the tensor-core kernel accepts).
* Whole-search kernels: every (variant, activation, n_hidden) instantiation through the trees-in-shared-memory kernel, the
  two-phase kernel, the warpgroup kernel and one launch per simulation, with the full tree dump compared; the evaluation stored
  in each dump is checked against the f64 bound.
* Edges of the tilings (warpgroup rounds, idle warpgroups, 1-row tiles, CTAs with one row or none) and of the discrete search's
  lookup tables (visit counts past FUSED_TAB = 255 and AZG_TAB = 1024), and the shapes azg_create refuses.

The case tables (MLP_SHAPES, QMLP_SHAPES, SEARCH_CASES) are torch-free: test_kernel_matrix.py checks them against the dispatch
tables of engine.cu on machines without a GPU.
"""
import os

import numpy as np
import pytest

from oracle import azo
from parity import assert_tree_equal
import f64ref as F

SMS = 148               # B200
TSM = "two_phase_trees_in_shared_memory"
ACTS = (azo.ACT_RELU, azo.ACT_ELU, azo.ACT_LEAKYRELU, azo.ACT_RELU6, azo.ACT_SILU, azo.ACT_HARDSWISH)
CARTPOLE, PENDULUM = 4, 3  # state_dim of the two variants (the S template argument)

# k_mlp<H, S, ACT>: every instantiation of engine.cu MLP_CASE
MLP_SHAPES = [(H, S, a) for H in (128, 64) for S in (CARTPOLE, PENDULUM) for a in ACTS]
# k_qmlp2<S, ACT, NL> / k_search_wg<S, ACT, NL>: every instantiation of engine.cu QMLP_CASE and FUSED_CASE
QMLP_SHAPES = [(S, a, nl) for S in (CARTPOLE, PENDULUM) for a in (azo.ACT_RELU, azo.ACT_ELU) for nl in (1, 2)]
SEARCH_KERNELS = {CARTPOLE: ("tsm", "two_phase", "warpgroups", "per_simulation"),
                  PENDULUM: ("two_phase", "warpgroups", "per_simulation")}
SEARCH_CASES = [(S, a, nl, K, k) for (S, a, nl) in QMLP_SHAPES for K in ((0,) if S == CARTPOLE else (1, 2, 3, 4))
                for k in SEARCH_KERNELS[S]]
# FP32 evaluation inside the search (one launch per simulation): the narrow network, 1 and 4 hidden layers, the FP32-only heads
FP32_SEARCH_CASES = [(S, a, L, K) for S in (CARTPOLE, PENDULUM) for L in (1, 4) for K in ((0,) if S == CARTPOLE else (5, 6, 7, 8))
                     for a in (ACTS[(L + K) % 6],)]


def make_cfg(S, act, n_hidden, K=0, hidden=128, q8=False, **kw):
    if S == CARTPOLE:
        cfg = azo.discrete_config(hidden=hidden, n_hidden=n_hidden, activation=act, **kw)
    else:
        cfg = azo.continuous_config(hidden=hidden, n_hidden=n_hidden, activation=act, num_components=K, **kw)
    cfg.eval_mode, cfg.math_mode = (azo.EVAL_Q8 if q8 else azo.EVAL_FP32), azo.MATH_DET
    return cfg


def q8_accepted(cfg) -> bool:
    """engine.cu azg_create: the tensor-core evaluation serves relu / elu, hidden 128, 2 or 3 hidden layers and at most 16 padded
    outputs (value + head rounded up to a multiple of 4)."""
    po_pad = (1 + cfg.head_dim + 3) // 4 * 4
    return cfg.hidden == 128 and cfg.n_hidden in (2, 3) and po_pad <= 16 and cfg.activation in (azo.ACT_RELU, azo.ACT_ELU)


def mlp_fits(cfg, smem_optin=232448) -> bool:
    """engine.cu azg_create: the FP32 kernel stages the packed weights and four groups of 32-row operands in shared memory."""
    H, P = cfg.hidden, cfg.head_dim
    po = (1 + P + 3) // 4 * 4
    wcount = cfg.state_dim * H + H + (cfg.n_hidden - 1) * (H * H + H) + H * po + po
    return (wcount + 4 * (H + po) * 32) * 4 <= smem_optin


def weights(cfg, kind="default", seed=3):
    """default: torch default init (network.init_policy_weights); x10: trained-like (|V| >> 1); edge: hidden layer 1 with an
    all-zero weight row, a 1e-30 row and a row whose largest magnitude is an exact power of two; dead: every layer-1 unit
    negative for observations in range (a zero row into the next layer)."""
    from alphazero_gym_b200.network import init_policy_weights
    w = init_policy_weights(seed, cfg.state_dim, cfg.hidden, cfg.n_hidden, cfg.head_dim).astype(np.float32)
    H, S = cfg.hidden, cfg.state_dim
    if kind == "x10":
        w = w * np.float32(10)
    elif kind in ("edge", "dead") and cfg.n_hidden >= 2:
        o = S * H + H  # hidden layer 1 weights [H][H]
        if kind == "edge":
            w[o:o + H] = 0.0
            w[o + 5 * H:o + 6 * H] *= np.float32(1e-30)
            row = w[o + 7 * H:o + 8 * H]
            row *= np.float32(0.125) / np.abs(row).max()
            row[np.argmax(np.abs(row))] = np.float32(0.125)
        else:
            w[S * H:S * H + H] = -50.0
    return w


def observations(cfg, n, seed=0):
    """Observations in the environments' ranges, then a zero row, 1e4 and 1e-30 rows (hardswish grows quadratically: 1e4 would
    overflow f32 after three layers, so it gets 10 instead)."""
    rng = np.random.default_rng(seed)
    if cfg.variant == azo.DISCRETE:
        x = rng.uniform(-1, 1, (n, 4)) * np.array([2.4, 3.0, 0.21, 3.0])
    else:
        th = rng.uniform(-np.pi, np.pi, n)
        x = np.stack([np.cos(th), np.sin(th), rng.uniform(-8, 8, n)], 1)
    x = x.astype(np.float32)
    big = 10.0 if cfg.activation == azo.ACT_HARDSWISH else 1e4
    edges = [np.zeros(cfg.state_dim), np.full(cfg.state_dim, big) * (-1) ** np.arange(cfg.state_dim),
             np.full(cfg.state_dim, 1e-30), -np.full(cfg.state_dim, big)]
    for i, e in enumerate(edges):
        if i < n:
            x[i] = e
    return x


def _with_env(env, fn):
    """Run fn with the AZG_* variables of `env` set (None: unset) and restore them afterwards."""
    old = {k: os.environ.pop(k, None) for k in env}
    try:
        for k, v in env.items():
            if v is not None:
                os.environ[k] = v
        return fn()
    finally:
        for k, v in old.items():
            os.environ.pop(k, None)
            if v is not None:
                os.environ[k] = v


# ------------------------------------------------------------------------------------------------ evaluation kernels

ROW_COUNTS = (1, 31, 32, 33, 127, 128, 129, SMS * 128 + 5)


def _check_forward(cfg, w, x, eng_q8):
    import enginelib as E
    eng = E.SearchEngine(E.engine_config(cfg, 4, eval_q8=eng_q8, fused=False))
    try:
        eng.set_weights(w)
        runs = {n: eng.mlp_forward(x[:n]) for n in ROW_COUNTS}
    finally:
        eng.close()
    Vo, raw = azo.mlp_forward(cfg, w, x)
    post = np.stack([azo.head_post(cfg, r) for r in raw[:256]])
    ref = F.forward(cfg, w, x[:256])
    name = f"H={cfg.hidden} S={cfg.state_dim} act={cfg.activation} L={cfg.n_hidden} K={cfg.num_components} q8={eng_q8}"
    for n, (V, head) in runs.items():
        assert np.array_equal(V, Vo[:n]), f"{name} n={n}: V differs from the oracle at {np.flatnonzero(V != Vo[:n])[:4]}"
        m = min(n, 256)
        assert np.array_equal(head[:m], post[:m]), f"{name} n={n}: head differs from the oracle"
    V, head = runs[ROW_COUNTS[-1]]
    for what, got, r, b in (("V", V[:256], ref["V"], ref["bV"]), ("head", head[:256], ref["post"], ref["bpost"])):
        ok, ratio = F.within(got, r, b)
        assert ok, f"{name}: {what} outside the f64 bound (worst |err| / bound = {ratio:.3g})"


@pytest.mark.gpu
@pytest.mark.parametrize("H,S,act", MLP_SHAPES)
def test_fp32_evaluation_kernel_matrix(H, S, act):
    """k_mlp<H, S, ACT> for n_hidden 1-4 (where the weights fit) and every head size: bit-identical to the oracle, inside the bound."""
    for L in (1, 2, 3, 4):
        for K in ((0,) if S == CARTPOLE else range(1, 9)):
            cfg = make_cfg(S, act, L, K, hidden=H)
            if not mlp_fits(cfg):
                continue
            for kind in (("default", "x10", "edge", "dead") if K in (0, 2) else ("default",)):
                _check_forward(cfg, weights(cfg, kind), observations(cfg, ROW_COUNTS[-1], seed=L + K), False)


@pytest.mark.gpu
@pytest.mark.parametrize("S,act,nl", QMLP_SHAPES)
@pytest.mark.parametrize("kind", ["default", "x10", "edge", "dead"])
def test_q8_evaluation_kernel_matrix(S, act, nl, kind):
    """k_qmlp2<S, ACT, NL> (evaluation only) for every head size the tensor-core kernel accepts."""
    for K in ((0,) if S == CARTPOLE else (1, 2, 3, 4, 5)):
        cfg = make_cfg(S, act, nl + 1, K, q8=True)
        assert q8_accepted(cfg)
        _check_forward(cfg, weights(cfg, kind), observations(cfg, ROW_COUNTS[-1], seed=K), True)


# ------------------------------------------------------------------------------------------------ whole-search kernels

KERNEL_ENV = {"tsm": {}, "two_phase": {"AZG_FUSED_KERNEL": "two_phase", "AZG_NO_TSM": "1"},
              "warpgroups": {"AZG_FUSED_KERNEL": "warpgroups"}, "per_simulation": {}}
KERNEL_NAME = {"tsm": TSM, "two_phase": "two_phase", "warpgroups": "warpgroups", "per_simulation": "none"}


def roots_for(cfg, B, seed=34):
    rng = np.random.default_rng(seed)
    if cfg.variant == azo.DISCRETE:
        return rng.uniform(-0.05, 0.05, (B, 4))
    return np.stack([rng.uniform(-np.pi, np.pi, B), rng.uniform(-1, 1, B)], 1)


def run_search(cfg, w, roots, kernel, root_n_init=None, tree_id0=0, dump=True, env=None):
    """Engine and oracle on the same search; the engine's dump, results and counters must equal the oracle's bit for bit, and the
    search must have run on `kernel` (None: whichever the engine chooses)."""
    import enginelib as E
    ref = azo.search(cfg, w, roots, root_n_init, tree_id0=tree_id0, dump=dump, n_threads=os.cpu_count() or 8)
    fused = kernel != "per_simulation"
    env = dict(KERNEL_ENV.get(kernel, {}), **(env or {}))
    env = {k: env.get(k) for k in ("AZG_FUSED_KERNEL", "AZG_NO_TSM")}
    out = _with_env(env, lambda: E.run_engine(cfg, w, roots, root_n_init, tree_id0=tree_id0, dump=dump, kernel=True, fused=fused,
                                              eval_q8=cfg.eval_mode == azo.EVAL_Q8))
    for k in ("counts", "actions", "Q"):
        out[k] = E.fit_columns(out[k], ref[k].shape[1])
    if kernel is not None:
        assert out["kernel"] == KERNEL_NAME[kernel], (out["kernel"], kernel)
    assert_tree_equal(out, ref, cfg.variant == azo.DISCRETE, exact_fp=True, results_only=not dump)
    assert np.array_equal(out["counters"][:7], ref["counters"][:7]), (out["counters"], ref["counters"])
    return out, ref


def check_stored_evaluation(cfg, w, dump):
    """Every evaluated, non-terminal node of the dump: its stored V and prior / head against the f64 forward of its observation,
    rebuilt from the stored state (Pendulum: cos / sin may round one f32 ulp away from the engine's, so the bound allows it)."""
    if cfg.variant == azo.DISCRETE:
        B, R = dump["node_n"].shape
        live = (np.arange(R)[None, :] < dump["n_nodes"][:, None]) & (dump["terminal"] == 0)
        x = dump["state"][live].astype(np.float32)
        xe = None
        V, post = dump["V"][live], dump["prior"][live]
    else:
        B, R = dump["node_n"].shape
        live = (np.arange(R)[None, :] < dump["n_rows"][:, None]) & ((dump["expanded"] == 1) | (np.arange(R)[None, :] == 0))
        live &= dump["terminal"] == 0
        th, thd = dump["state"][live][:, 0], dump["state"][live][:, 1]
        x = np.stack([np.cos(th), np.sin(th), thd], 1).astype(np.float32)
        xe = np.stack([np.spacing(np.abs(x[:, 0])), np.spacing(np.abs(x[:, 1])), np.zeros(len(x), np.float32)], 1)
        V, post = dump["V"][live], dump["head"][live]
    assert len(x) > 0
    ref = F.forward(cfg, w, x, x_err=xe)
    ok, ratio = F.within(V, ref["V"], ref["bV"])
    assert ok, f"stored V outside the f64 bound (worst |err| / bound {ratio:.3g})"
    ok, ratio = F.within(post, ref["post"], ref["bpost"])
    assert ok, f"stored {'prior' if cfg.variant == azo.DISCRETE else 'head'} outside the f64 bound (worst ratio {ratio:.3g})"


@pytest.mark.gpu
@pytest.mark.parametrize("S,act,nl,K,kernel", SEARCH_CASES)
def test_search_kernel_matrix(S, act, nl, K, kernel):
    B, N = (300, 40) if S == CARTPOLE else (300, 24)
    cfg = make_cfg(S, act, nl + 1, K, q8=True, n_rollouts=N, **({"epsilon": 0.1} if S == CARTPOLE else {}))
    w = weights(cfg, "x10" if K == 3 else "default")
    out, _ = run_search(cfg, w, roots_for(cfg, B), kernel)
    if kernel == "per_simulation":
        assert out["counters"][7] > N
    else:
        assert out["counters"][7] == 1
    check_stored_evaluation(cfg, w, out)


@pytest.mark.gpu
@pytest.mark.parametrize("S,act,L,K", FP32_SEARCH_CASES)
def test_fp32_search_matrix(S, act, L, K):
    cfg = make_cfg(S, act, L, K, hidden=64, n_rollouts=30, **({"epsilon": 0.1} if S == CARTPOLE else {}))
    w = weights(cfg)
    out, _ = run_search(cfg, w, roots_for(cfg, 200), "per_simulation")
    check_stored_evaluation(cfg, w, out)


# ------------------------------------------------------------------------------------------------ tilings and tables


def wg_plan(B, sms=SMS):
    """Mirror of the warpgroup kernel's partition (engine.cu launch_fused_t, search_wg.cuh k_search_wg): per CTA of every chunk,
    (rows, rounds, rows per tile, tiles).  Returns the set of properties the batch reaches."""
    chunk = sms * 16 * 128
    seen = set()
    for lo in range(0, B, chunk):
        n = min(B, lo + chunk) - lo
        grid = max(1, min((n + 3) // 4, sms))
        per = (n + grid - 1) // grid
        for b in range(grid):
            nrows = min(b * per + per, n) - b * per
            if nrows <= 0:
                seen.add("empty_cta")
                continue
            if nrows == 1:
                seen.add("one_row_cta")
            rounds = (nrows + 511) // 512
            th = (nrows + 4 * rounds - 1) // (4 * rounds)
            if th > 32:
                th = (th + 31) & ~31
            ntiles = (nrows + th - 1) // th
            seen.add(f"rounds{rounds}")
            if ntiles < 4 * rounds:
                seen.add("idle_warpgroup")
            if th == 1 or nrows - (ntiles - 1) * th == 1:
                seen.add("one_row_tile")
            if th > 32 and th % 32 == 0 and th * 4 * rounds > nrows + 32:
                seen.add("th_rounded")
    return seen


WG_FORCED = {1: {"one_row_tile", "idle_warpgroup", "one_row_cta"}, 2: {"one_row_tile", "idle_warpgroup"}, 3: {"one_row_tile"},
             5: {"one_row_tile"}, 33: {"one_row_tile"}, 129: {"one_row_tile"}, 130: {"one_row_tile"}, 592: {"rounds1"},
             593: {"empty_cta"}, 736: {"one_row_cta"}, 14801: {"empty_cta"}}


@pytest.mark.gpu
@pytest.mark.parametrize("B", sorted(WG_FORCED))
def test_warpgroup_tiling_edges(B):
    assert WG_FORCED[B] <= wg_plan(B), (B, wg_plan(B))
    cfg = make_cfg(PENDULUM, azo.ACT_ELU, 3, 2, q8=True, n_rollouts=12)
    run_search(cfg, weights(cfg), roots_for(cfg, B, seed=B), "warpgroups", tree_id0=B, dump=B <= 1000)


@pytest.mark.gpu
@pytest.mark.parametrize("S,B,N,claims", [(PENDULUM, SMS * 513, 6, {"rounds2", "idle_warpgroup", "th_rounded"}),
                                          (PENDULUM, SMS * 1100, 4, {"rounds3"}),
                                          (CARTPOLE, 65536, 50, {"rounds1"})])
def test_warpgroups_chosen_by_batch_size(S, B, N, claims):
    assert claims <= wg_plan(B), wg_plan(B)
    cfg = make_cfg(S, azo.ACT_RELU, 2, 2, q8=True, n_rollouts=N, **({"epsilon": 0.1} if S == CARTPOLE else {}))
    run_search(cfg, weights(cfg), roots_for(cfg, B, seed=N), None, tree_id0=11, dump=False)


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 127, 128, 129, 2 * SMS * 128 + 1])
def test_two_phase_partition_edges(B):
    """One tile, a full tile and one row more, and more tiles than SMs (several tiles per CTA)."""
    cfg = make_cfg(PENDULUM, azo.ACT_RELU, 3, 3, q8=True, n_rollouts=10)
    run_search(cfg, weights(cfg), roots_for(cfg, B, seed=B), "two_phase", tree_id0=B, dump=B <= 1000)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", ["tsm", "two_phase", "warpgroups", "per_simulation"])
@pytest.mark.parametrize("N,reuse", [(300, False), (600, False), (300, True)])
def test_discrete_visit_counts_past_shared_tables(kernel, N, reuse):
    """Visit counts above FUSED_TAB (255): the whole-search kernels leave their shared-memory reciprocal / sqrt tables."""
    B = 40
    cfg = make_cfg(CARTPOLE, azo.ACT_RELU, 2, q8=True, n_rollouts=N, epsilon=0.1)
    rn = np.random.default_rng(N).integers(250, 301, B).astype(np.int32) if reuse else None
    out, _ = run_search(cfg, weights(cfg), roots_for(cfg, B, seed=N), kernel, rn, tree_id0=7)
    assert out["node_n"].max() > 255


@pytest.mark.gpu
def test_per_simulation_visit_counts_past_global_table():
    """Root visit counts above AZG_TAB (1024): one launch per simulation leaves its global-memory tables."""
    B, N = 16, 800
    cfg = make_cfg(CARTPOLE, azo.ACT_ELU, 3, q8=True, n_rollouts=N, epsilon=0.1)
    rn = np.random.default_rng(1).integers(250, 301, B).astype(np.int32)
    out, _ = run_search(cfg, weights(cfg), roots_for(cfg, B, seed=5), "per_simulation", rn, tree_id0=3)
    assert out["node_n"].max() > 1024


def _refusal_shapes():
    for S in (CARTPOLE, PENDULUM):
        for H in (64, 128):
            for L in (1, 2, 3, 4):
                for act in ACTS:
                    for K in ((0,) if S == CARTPOLE else range(1, 9)):
                        yield S, H, L, act, K


@pytest.mark.gpu
def test_refusals_agree_with_q8_supported():
    """azg_create accepts a Q8 engine exactly where EngineConfig.q8_supported() says so, and an FP32 engine exactly where its
    weights fit in shared memory; every refusal raises AzgError."""
    import enginelib as E
    from alphazero_gym_b200._cabi import AzgError
    for S, H, L, act, K in _refusal_shapes():
        cfg = make_cfg(S, act, L, K, hidden=H)
        for q8 in (False, True):
            ecfg = E.engine_config(cfg, 4, eval_q8=q8, fused=False)
            want = (ecfg.q8_supported() and mlp_fits(cfg)) if q8 else mlp_fits(cfg)
            try:
                E.SearchEngine(ecfg).close()
                ok = True
            except AzgError:
                ok = False
            assert ok == want, (S, H, L, act, K, q8)
