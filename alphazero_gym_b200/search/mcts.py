"""Drop-in replacements for alphazero.search.mcts.MCTSDiscrete / MCTSContinuous.

Same constructor kwargs (reference mcts.py:316-327, :537-549), same methods and attributes the callers use
(agents.py:126-155, :291-292, :317, :521-522): `search(Env)`, `return_results(final_selection)`, `forward(action,
state)` (discrete), writable `root_node` / `root_state`, readable `n_rollouts`, `c_uct`, `gamma`.  The legacy
upstream call form `search(n_mcts, c, Env, mcts_env)` named in BASELINE.json is accepted too.

What changes underneath: the tree lives in HBM tables and the whole search -- select, env step, network
evaluation, backup -- runs in the CUDA engine (csrc/, C ABI include/azg.h).  `model` is only read for its
weights and shape; `Env` only for its hidden state (`Env.unwrapped.state`) and its class name.  Envs other than
CartPole, MountainCar and Acrobot (MCTSDiscrete), Pendulum and MountainCarContinuous (MCTSContinuous) raise: there is no CPU fallback.  Tie-break / epsilon-greedy / action-noise randomness comes from
the engine's counter-based Philox streams keyed by (`seed`, search counter) instead of Python's `random` and
torch's global generator.

Batched use (thousands of independent roots per call): `search_batch(root_states)`; or use
alphazero_gym_b200.engine.SearchEngine directly with device-resident tensors.
"""
from __future__ import annotations

from typing import Any, Dict, Optional, Tuple

import numpy as np

from .._cabi import CONTINUOUS, DISCRETE
from ..engine import ACROBOT, CARTPOLE, MOUNTAIN_CAR, MOUNTAIN_CAR_CONTINUOUS, PENDULUM, EngineConfig, SearchEngine, flatten_state_dict
from ..network import describe_model, weights_version

PENDULUM_R_SCALE = 16.2736044  # reference mcts.py:20 (applied inside the engine)


# Wrappers rl/make_game.py:71-83 puts around the env for the name suffixes -v0n / r / p / s (rl/wrappers.py:44-155) change the rewards
# or observations the search sees, while the engine steps the plain CartPole-v0 / Pendulum-v0 dynamics.  The two reward wrappers that
# are plain Python arithmetic on CartPole's reward -- ReparametrizeWrapper (-v0r) and ScaleRewardWrapper (-v0s) -- are carried into the
# engine as its reward model (azg_set_reward_model; `reward_model` below evaluates the wrappers' own expressions); the others --
# NormalizeWrapper (an sklearn scaler fitted on 10 000 random observations), PILCOWrapper (scipy's multivariate normal pdf),
# ClipRewardWrapper, ScaledObservationWrapper (Atari), and ScaleRewardWrapper around Pendulum (np.float32 rewards, whose promotion through
# the backup depends on the numpy version) -- are REFUSED: searching through them silently would not be the reference's search.
_REWARD_WRAPPERS = ("ReparametrizeWrapper", "ScaleRewardWrapper")
_REFUSED_WRAPPERS = ("NormalizeWrapper", "PILCOWrapper", "ClipRewardWrapper", "ScaledObservationWrapper")


def _wrapper_chain(env):
    """(base env, names of the reward wrappers around it, outermost first); refuses the wrappers the engine does not implement."""
    e, seen, names = env, 0, []
    while hasattr(e, "env") and e is not getattr(e, "env") and seen < 16:  # gym.Wrapper chain (rl/make_game.py:60-62)
        name = type(e).__name__
        if name in _REFUSED_WRAPPERS:
            raise NotImplementedError(f"{name} (rl/wrappers.py) changes what the search sees; the CUDA engine implements the plain "
                                      "CartPole-v0 / Pendulum-v0 envs, ReparametrizeWrapper and ScaleRewardWrapper, and has no CPU fallback")
        if name in _REWARD_WRAPPERS:
            names.append(name)
        e = e.env
        seen += 1
    return getattr(e, "unwrapped", e), names


def _unwrap(env):
    return _wrapper_chain(env)[0]


def reward_model(env, variant: int):
    """(reward_step, reward_terminal) of the env's reward wrappers, innermost applied first, each with the wrapper's own Python
    expression (rl/wrappers.py:58-105) so that the constants are the reference's bit for bit."""
    base, names = _wrapper_chain(env)
    if names and variant != DISCRETE and _is_mountain_car_continuous(base):
        raise NotImplementedError(f"{names[0]} around MountainCarContinuous-v0: the CUDA engine steps the plain env only")
    if names and variant == DISCRETE and _is_mountain_car(base):
        raise NotImplementedError(f"{names[0]} around MountainCar-v0: the CUDA engine steps the plain env only")
    if names and variant == DISCRETE and _is_acrobot(base):
        raise NotImplementedError(f"{names[0]} around Acrobot-v1: the CUDA engine steps the plain env only")
    step, terminal = 1.0, 1.0  # gym CartPole-v0 pays 1.0 for every step, the terminating one included
    for name in reversed(names):
        if name == "ReparametrizeWrapper":
            if variant == DISCRETE:  # CartPole: r = -1 if terminal else 0.005; Pendulum falls through unchanged (:88-105)
                step, terminal = 0.005, -1
        elif name == "ScaleRewardWrapper":
            if variant != DISCRETE:
                raise NotImplementedError("ScaleRewardWrapper around Pendulum returns np.float32(reward / 1000.0); how that promotes through "
                                          "the backup depends on the numpy version, and the CUDA engine does not restate it")
            step, terminal = step / 250.0, terminal / 250.0
    return float(step), float(terminal)


def _is_mountain_car_continuous(base) -> bool:
    return type(base).__name__ == "Continuous_MountainCarEnv"  # gym's class (classic_control/continuous_mountain_car.py)


def _is_mountain_car(base) -> bool:
    return type(base).__name__ == "MountainCarEnv"  # gym's class (classic_control/mountain_car.py)


def _is_acrobot(base) -> bool:
    return type(base).__name__ == "AcrobotEnv"  # gym's class (classic_control/acrobot.py)


def acrobot_obs(s: np.ndarray) -> np.ndarray:
    """AcrobotEnv._get_ob of the hidden state (theta1, theta2, dtheta1, dtheta2): what the network sees."""
    return np.array([np.cos(s[0]), np.sin(s[0]), np.cos(s[1]), np.sin(s[1]), s[2], s[3]])


def discrete_env(env) -> str:
    """The env MCTSDiscrete has the engine step for `env`: MountainCar-v0 for gym's MountainCarEnv and Acrobot-v1 for its AcrobotEnv
    (by class name, under any wrappers), CartPole-v0 otherwise (env_hidden_state refuses the envs that are none of these)."""
    base = _unwrap(env)
    return MOUNTAIN_CAR if _is_mountain_car(base) else (ACROBOT if _is_acrobot(base) else CARTPOLE)


def continuous_env(env) -> str:
    """The env MCTSContinuous has the engine step for `env`: MountainCarContinuous-v0 for gym's Continuous_MountainCarEnv (by class
    name, under any wrappers), Pendulum-v0 otherwise (env_hidden_state refuses the envs that are neither)."""
    return MOUNTAIN_CAR_CONTINUOUS if _is_mountain_car_continuous(_unwrap(env)) else PENDULUM


def env_hidden_state(env, variant: int, env_id: Optional[str] = None) -> np.ndarray:
    """Root of the search = hidden state of the gym env (replaces copy.deepcopy(Env), mcts.py:443, :680).  env_id = MOUNTAIN_CAR
    accepts gym's MountainCarEnv for the discrete variant (a 2-wide state), env_id = ACROBOT its AcrobotEnv (a 4-wide state); without
    it the search classes' original envs only."""
    base = _unwrap(env)
    if not hasattr(base, "state") or base.state is None:
        raise TypeError("Env has no hidden `.state`; only gym CartPole-v0 / MountainCar-v0 / Acrobot-v1 / Pendulum-v0 / "
                        "MountainCarContinuous-v0 style envs are supported")
    s = np.asarray(base.state, dtype=np.float64).reshape(-1)
    if env_id == MOUNTAIN_CAR:
        if variant != DISCRETE or not _is_mountain_car(base) or s.size != 2:
            raise TypeError(f"unsupported environment {type(base).__name__} for MountainCar-v0: the discrete search steps gym's "
                            "MountainCarEnv (a 2-wide state)")
        return s
    if env_id == ACROBOT:
        if variant != DISCRETE or not _is_acrobot(base) or s.size != 4:
            raise TypeError(f"unsupported environment {type(base).__name__} for Acrobot-v1: the discrete search steps gym's "
                            "AcrobotEnv (a 4-wide state)")
        return s
    name = type(base).__name__.lower()
    want = 4 if variant == DISCRETE else 2
    mcc = _is_mountain_car_continuous(base)
    if (s.size != want or ("cartpole" in name and variant != DISCRETE) or ("pendulum" in name and variant != CONTINUOUS)
            or ("mountaincar" in name and not (mcc and variant == CONTINUOUS))):
        raise TypeError(f"unsupported environment {type(base).__name__} for this search class: the CUDA engine implements "
                        "CartPole-v0 (MCTSDiscrete), Pendulum-v0 and MountainCarContinuous-v0 (MCTSContinuous) dynamics and has no "
                        "CPU fallback")
    return s


class RootNode:
    """What callers may touch of the reference's Node at the root (states.py:8-57): state, n, V, terminal."""

    def __init__(self, state: np.ndarray, n: int = 0, V: float = 0.0, terminal: bool = False, hidden: Optional[np.ndarray] = None):
        self.state, self.n, self.V, self.terminal, self.hidden = state, n, V, terminal, hidden
        self.parent_action = None


class MCTS:
    """Common part (reference mcts.py:23-307)."""

    variant = DISCRETE

    def __init__(self, model, n_rollouts: int, c_uct: float, gamma: float, epsilon: float, device: str, V_target_policy: str,
                 root_state: Optional[np.ndarray], seed: int = 34, **engine_kw: Any) -> None:
        self.device = device
        self.root_node: Optional[RootNode] = None
        self.root_state = root_state
        self.model = model
        self.n_rollouts = n_rollouts
        self.c_uct = c_uct
        self.gamma = gamma
        self.epsilon = epsilon
        self.V_target_policy = V_target_policy
        self.seed = seed
        self._engine_kw = engine_kw
        self._engines: Dict[int, SearchEngine] = {}
        self._wver: Dict[int, int] = {}
        self._searches = 0
        self._results: Optional[Dict[str, np.ndarray]] = None
        self._tree: Optional[Dict[str, np.ndarray]] = None

    # -- engine plumbing ---------------------------------------------------------------------------------
    def _cuda_index(self) -> int:
        d = str(self.device)
        return int(d.split(":")[1]) if ":" in d else 0

    def _engine_config(self, max_trees: int) -> EngineConfig:
        raise NotImplementedError

    def _engine(self, B: int) -> SearchEngine:
        cap = 1 if B == 1 else 1 << (B - 1).bit_length()
        eng = self._engines.get(cap)
        if eng is None:
            eng = SearchEngine(self._engine_config(cap))
            self._engines[cap] = eng
            self._wver[cap] = -1
        v = weights_version(self.model)
        if self._wver[cap] != v:  # the agent trains the model between searches (agents.py:157-184)
            eng.set_weights(flatten_state_dict(self.model.state_dict()))
            self._wver[cap] = v
        return eng

    def refresh_weights(self) -> None:
        """Force the next search to reload `model`'s weights (for updates the version counters cannot see, network.weights_version)."""
        for cap in self._wver:
            self._wver[cap] = -1

    def close(self) -> None:
        for e in self._engines.values():
            e.close()
        self._engines.clear()

    # -- reference API -----------------------------------------------------------------------------------------
    def search(self, *args, **kwargs) -> None:
        raise NotImplementedError

    @staticmethod
    def _env_from_args(args, kwargs):
        """Accept search(Env) / search(Env=Env) (reference) and search(n_mcts, c, Env, mcts_env) (upstream form)."""
        if "Env" in kwargs:
            return kwargs["Env"], kwargs.get("n_mcts"), kwargs.get("c")
        if len(args) == 1:
            return args[0], None, None
        if len(args) >= 3:
            return args[2], args[0], args[1]
        raise TypeError("search(Env) or search(n_mcts, c, Env, mcts_env)")

    def return_results(self, final_selection: str) -> Tuple[np.ndarray, np.ndarray, np.ndarray, np.ndarray, Any]:
        """(root state, actions.squeeze(), counts, Q, V_target) -- reference mcts.py:269-307."""
        assert self.root_node is not None
        r = self._results
        assert r is not None, "search() has not been run"
        C = int(r["n_children"][0])
        counts = r["counts"][0, :C].astype(np.int64)
        Q = r["Q"][0, :C].copy()
        if self.variant == DISCRETE:
            actions = np.arange(C)
        else:
            actions = r["actions"][0, :C].astype(np.float32)
        return self.root_node.state, actions.squeeze(), counts, Q, np.float64(r["V_target"][0])

    def search_batch(self, root_states: np.ndarray, root_n_init: Optional[np.ndarray] = None, tree_id0: int = 0) -> Dict[str, np.ndarray]:
        """Batched form: B independent roots (hidden env states) -> root results arrays with B rows."""
        root_states = np.ascontiguousarray(root_states, np.float64)
        eng = self._engine(root_states.shape[0])
        return eng.search_host(root_states, self.n_rollouts, root_n_init, tree_id0)


class MCTSDiscrete(MCTS):
    """AlphaZero search for CartPole-v0, MountainCar-v0 and Acrobot-v1 (reference mcts.py:310-526).  The env is taken from the Env
    each search() is handed (discrete_env); search_batch steps the env of the last search(), or the engine keyword `env`
    (engine.CARTPOLE by default), from hidden states.  For Acrobot-v1 the root's state (return_results) and the state forward() takes
    are the 6-wide observation (AcrobotEnv._get_ob), while the engine searches from the 4-wide hidden state."""

    variant = DISCRETE

    def __init__(self, model, num_actions: int, n_rollouts: int, c_uct: float, gamma: float, epsilon: float, V_target_policy: str,
                 device: str, root_state: Optional[np.ndarray], seed: int = 34, **engine_kw: Any):
        super().__init__(model=model, n_rollouts=n_rollouts, c_uct=c_uct, gamma=gamma, epsilon=epsilon, device=device,
                         V_target_policy=V_target_policy, root_state=root_state, seed=seed, **engine_kw)
        self.num_actions = num_actions
        self._env = self._engine_kw.pop("env", None) or CARTPOLE

    def _engine_config(self, max_trees: int) -> EngineConfig:
        d = describe_model(self.model)
        return EngineConfig(variant=DISCRETE, max_rollouts=self.n_rollouts, max_trees=max_trees, num_actions=self.num_actions,
                            state_dim=d["state_dim"], hidden=d["hidden"], n_hidden=d["n_hidden"], activation=d["activation"],
                            V_target_policy=self.V_target_policy, c_uct=self.c_uct, gamma=float(self.gamma), epsilon=self.epsilon,
                            device=self._cuda_index(), seed=self.seed, env=self._env, **self._engine_kw)

    def search(self, *args, **kwargs) -> None:
        Env, n_mcts, c = self._env_from_args(args, kwargs)
        if n_mcts is not None and (n_mcts != self.n_rollouts or c != self.c_uct):
            self.close()
            self.n_rollouts, self.c_uct = n_mcts, c
        env = discrete_env(Env)
        if env in (MOUNTAIN_CAR, ACROBOT):
            if self.num_actions != 3:
                raise ValueError(f"{env} has 3 actions, the search was built with num_actions={self.num_actions}")
            hidden = env_hidden_state(Env, DISCRETE, env_id=env)
        else:
            hidden = env_hidden_state(Env, DISCRETE)
        if env != self._env:  # the engines are built for one env
            self.close()
            self._env = env
        # initialize_search (mcts.py:364-383): new root, or continue from the node forward() selected
        if self.root_node is None:
            if self.root_state is not None:
                obs = self.root_state
            else:
                obs = acrobot_obs(hidden) if env == ACROBOT else hidden
            self.root_node = RootNode(np.asarray(obs), n=0, hidden=hidden)
        if self.root_node.terminal:
            raise ValueError("Can't do tree search from a terminal node")
        eng = self._engine(1)
        eng.set_reward_model(*reward_model(Env, DISCRETE))
        self._results = eng.search_host(hidden[None], self.n_rollouts, np.array([self.root_node.n], np.int32), tree_id0=self._searches)
        self._searches += 1
        self._tree = eng.dump_tree(1)
        self.root_node.n = int(self._tree["node_n"][0, 0])
        self.root_node.V = float(self._tree["V"][0, 0])

    def forward(self, action: int, state: np.ndarray) -> None:
        """Tree reuse (mcts.py:495-526).  As in the reference only the new root's visit count survives: its
        edges are re-created by the next search's evaluation (mcts.py:412-415; SURVEY 7-7)."""
        assert self.root_node is not None and self._tree is not None
        t = self._tree
        child = int(t["echild"][0, 0, action])
        if child < 0:
            self.root_node, self.root_state = None, state
            return
        child_state = t["state"][0, child]
        child_obs = acrobot_obs(child_state) if self._env == ACROBOT else child_state  # what the agent's `state` is
        if np.linalg.norm(child_obs - np.asarray(state, np.float64).reshape(-1)) > 0.01:
            print("Warning: this domain seems stochastic. Not re-using the subtree for next search. "
                  + "To deal with stochastic environments, implement progressive widening.")
            self.root_node, self.root_state = None, state
            return
        self.root_node = RootNode(np.asarray(state), n=int(t["node_n"][0, child]), V=float(t["V"][0, child]),
                                  terminal=bool(t["terminal"][0, child]), hidden=child_state.copy())
        self._tree = None


class MCTSContinuous(MCTS):
    """A0C search with progressive widening for Pendulum-v0 and MountainCarContinuous-v0 (reference mcts.py:529-741).  The env
    is taken from the Env each search() is handed (continuous_env); search_batch steps the env of the last search(), or the
    engine keyword `env` (engine.PENDULUM by default)."""

    variant = CONTINUOUS

    def __init__(self, model, n_rollouts: int, c_uct: float, c_pw: float, kappa: float, gamma: float, epsilon: float,
                 V_target_policy: str, device: str, root_state: Optional[np.ndarray], seed: int = 34, **engine_kw: Any):
        super().__init__(model=model, n_rollouts=n_rollouts, c_uct=c_uct, gamma=gamma, epsilon=epsilon, device=device,
                         V_target_policy=V_target_policy, root_state=root_state, seed=seed, **engine_kw)
        self.c_pw = c_pw
        self.kappa = kappa
        self._env = self._engine_kw.pop("env", None) or PENDULUM

    def _engine_config(self, max_trees: int) -> EngineConfig:
        d = describe_model(self.model)
        return EngineConfig(variant=CONTINUOUS, max_rollouts=self.n_rollouts, max_trees=max_trees,
                            num_components=d["num_components"], state_dim=d["state_dim"], hidden=d["hidden"], n_hidden=d["n_hidden"],
                            activation=d["activation"], V_target_policy=self.V_target_policy, c_uct=self.c_uct, c_pw=self.c_pw,
                            kappa=self.kappa, gamma=float(self.gamma), epsilon=self.epsilon, action_bound=d["action_bound"],
                            log_std_min=d["log_std_min"], log_std_max=d["log_std_max"], device=self._cuda_index(), seed=self.seed,
                            env=self._env, **self._engine_kw)

    def search(self, *args, **kwargs) -> None:
        Env, n_mcts, c = self._env_from_args(args, kwargs)
        if n_mcts is not None and (n_mcts != self.n_rollouts or c != self.c_uct):
            self.close()
            self.n_rollouts, self.c_uct = n_mcts, c
        hidden = env_hidden_state(Env, CONTINUOUS)
        env = continuous_env(Env)
        if env != self._env:  # the engines are built for one env
            self.close()
            self._env = env
        # initialize_search (mcts.py:589-600): always a new root; the tree is never reused
        if self.root_state is not None:
            obs = self.root_state
        elif env == MOUNTAIN_CAR_CONTINUOUS:
            obs = hidden.copy()  # the observation is the state itself
        else:
            obs = np.array([np.cos(hidden[0]), np.sin(hidden[0]), hidden[1]])
        self.root_node = RootNode(np.asarray(obs), n=0, hidden=hidden)
        eng = self._engine(1)
        eng.set_reward_model(*reward_model(Env, CONTINUOUS))
        self._results = eng.search_host(hidden[None], self.n_rollouts, None, tree_id0=self._searches)
        self._searches += 1
        self.root_node.n = self.n_rollouts
