"""Test-side helpers: build an engine from an oracle Config, run it, and shape its output like the oracle's."""
import numpy as np
import torch

from oracle import azo
from alphazero_gym_b200.engine import EngineConfig, SearchEngine


def engine_config(cfg: azo.Config, max_trees: int, **kw) -> EngineConfig:
    d = dict(variant=cfg.variant, max_rollouts=cfg.n_rollouts, max_trees=max_trees, num_actions=cfg.num_actions,
             num_components=cfg.num_components, state_dim=cfg.state_dim, hidden=cfg.hidden, n_hidden=cfg.n_hidden,
             activation=cfg.activation, V_target_policy=cfg.V_target_policy, puct_f32=cfg.puct_f32, c_uct=cfg.c_uct,
             gamma=cfg.gamma, epsilon=cfg.epsilon, c_pw=cfg.c_pw, kappa=cfg.kappa, action_bound=cfg.action_bound,
             log_std_min=cfg.log_std_min, log_std_max=cfg.log_std_max, seed=cfg.seed,
             eval_q8=cfg.eval_mode == azo.EVAL_Q8, rng_mt19937=cfg.rng_mode == azo.RNG_MT19937, env=cfg.env)
    d.update(kw)
    return EngineConfig(**d)


def run_engine(cfg: azo.Config, weights, root_state, root_n_init=None, tree_id0=0, tapes=None, dump=True, host=False, kernel=False,
               **kw):
    """One batched search on cuda:0 through the C ABI; returns oracle-shaped dict (results [+ dump] + counters [+ kernel: the
    whole-search kernel that ran, "none" for one launch per kernel and simulation])."""
    root_state = np.ascontiguousarray(root_state, np.float64)
    B = root_state.shape[0]
    eng = SearchEngine(engine_config(cfg, B, **kw))
    try:
        if weights is not None:
            eng.set_weights(weights)
        if cfg.reward_step != 1.0 or cfg.reward_terminal != 1.0:
            eng.set_reward_model(cfg.reward_step, cfg.reward_terminal)
        if tapes is not None:
            eng.set_tapes(tapes["V"], tapes.get("prior"), tapes.get("action"))
        if host:
            out = eng.search_host(root_state, cfg.n_rollouts, root_n_init, tree_id0)
        else:
            rs = torch.from_numpy(root_state).cuda()
            rn = None if root_n_init is None else torch.from_numpy(np.ascontiguousarray(root_n_init, np.int32)).cuda()
            eng.search(rs, cfg.n_rollouts, rn, tree_id0)
            eng.status()
            out = {k: v.cpu().numpy() for k, v in eng.root_results().items()}
        # pad result columns like the oracle (cmax columns)
        if dump:
            out.update(eng.dump_tree(B))
        c = eng.counters(B)
        out["counters"] = np.array([c["sims"], c["levels"], c["children_scanned"], c["pw_inserts"], c["evals"],
                                    c["rng_draws"], c["terminal_leaf_sims"], c["launches"]], np.int64)
        if kernel:
            out["kernel"] = eng.fused_stats()["kernel"]
        return out
    finally:
        eng.close()


def fit_columns(a: np.ndarray, cols: int) -> np.ndarray:
    if a.ndim != 2 or a.shape[1] == cols:
        return a
    out = np.zeros((a.shape[0], cols), a.dtype)
    m = min(cols, a.shape[1])
    out[:, :m] = a[:, :m]
    return out
