"""ctypes binding of the CPU oracle (oracle/libazg_oracle.so).

TEST INFRASTRUCTURE ONLY.  Importable from tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs -- never from the product package `alphazero_gym_b200`.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from dataclasses import dataclass, field
from typing import Dict, Optional

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libazg_oracle.so")

DISCRETE, CONTINUOUS = 0, 1
ACT_RELU, ACT_ELU, ACT_LEAKYRELU, ACT_RELU6, ACT_SILU, ACT_HARDSWISH = 0, 1, 2, 3, 4, 5
ACT_NAMES = {0: "relu", 1: "elu", 2: "leakyrelu", 3: "relu6", 4: "silu", 5: "hardswish"}
MATH_LIBM, MATH_DET = 0, 1
EVAL_FP32, EVAL_Q8 = 0, 1
RNG_PHILOX, RNG_MT19937 = 0, 1
VT = {"off_policy": 0, "on_policy": 1, "greedy": 2}
# env names as alphazero_gym_b200.engine spells them (not imported: the oracle stays apart from the product package);
# Config.env None = the variant's own env, CartPole-v0 / Pendulum-v0
CARTPOLE, PENDULUM, MOUNTAIN_CAR_CONTINUOUS = "CartPole-v0", "Pendulum-v0", "MountainCarContinuous-v0"
MOUNTAIN_CAR, ACROBOT = "MountainCar-v0", "Acrobot-v1"
_ENV = {None: 0, MOUNTAIN_CAR_CONTINUOUS: 1, MOUNTAIN_CAR: 2, ACROBOT: 3}  # AZO_ENV_*
# the config defaults each env needs (the env's action count / observation width / action bound)
_ENV_DEFAULTS = {MOUNTAIN_CAR_CONTINUOUS: dict(state_dim=2, action_bound=1.0), MOUNTAIN_CAR: dict(num_actions=3, state_dim=2),
                 ACROBOT: dict(num_actions=3, state_dim=6)}
R_SCALE = 16.2736044  # the continuous search's reward divisor (mcts.py:20; PENDULUM_R_SCALE in azg_oracle.c)
ERR_WRAP = -4  # AZO_ERR_WRAP


class WrapCapReached(Exception):
    """Acrobot: an angle needed more than 64 iterations of a wrap loop (gym itself loops on; the engine fails with AZG_EWRAP)."""


def build(force: bool = False) -> str:
    """Compile the oracle with its Makefile (gcc only)."""
    src = os.path.join(_HERE, "azg_oracle.c")
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-s", "libazg_oracle.so"])
    return _LIB_PATH


class _Cfg(C.Structure):
    _fields_ = [
        ("variant", C.c_int32), ("n_rollouts", C.c_int32), ("num_actions", C.c_int32), ("num_components", C.c_int32),
        ("state_dim", C.c_int32), ("hidden", C.c_int32), ("n_hidden", C.c_int32), ("activation", C.c_int32),
        ("math_mode", C.c_int32), ("v_target", C.c_int32), ("puct_f32", C.c_int32), ("use_eval_tape", C.c_int32),
        ("c_uct", C.c_double), ("gamma", C.c_double), ("epsilon", C.c_double), ("c_pw", C.c_double), ("kappa", C.c_double),
        ("action_bound", C.c_float), ("log_std_min", C.c_float), ("log_std_max", C.c_float),
        ("seed", C.c_uint64), ("eval_mode", C.c_int32), ("rng_mode", C.c_int32),
        ("reward_step", C.c_double), ("reward_terminal", C.c_double), ("env", C.c_int32),
    ]


class _DumpD(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in
                ("n_nodes", "parent", "paction", "node_n", "terminal", "V", "r", "state", "prior", "eW", "en", "echild")]


class _DumpC(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in
                ("n_rows", "parent", "action", "eW", "en", "expanded", "node_n", "terminal", "V", "r", "state", "head")]


class _Res(C.Structure):
    _fields_ = [("cmax", C.c_int32), ("n_children", C.c_void_p), ("actions", C.c_void_p), ("counts", C.c_void_p),
                ("Q", C.c_void_p), ("V_target", C.c_void_p), ("counters", C.c_void_p)]


class _Tapes(C.Structure):
    _fields_ = [("V", C.c_void_p), ("prior", C.c_void_p), ("action", C.c_void_p)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            build()
        L = C.CDLL(_LIB_PATH)
        L.azo_search.restype = C.c_int
        L.azo_search.argtypes = [C.POINTER(_Cfg), C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64,
                                 C.POINTER(_Tapes), C.POINTER(_Res), C.POINTER(_DumpD), C.POINTER(_DumpC), C.c_int32]
        L.azo_num_weights.restype = C.c_int64
        L.azo_num_weights.argtypes = [C.POINTER(_Cfg)]
        L.azo_head_dim.restype = C.c_int32
        L.azo_head_dim.argtypes = [C.POINTER(_Cfg)]
        L.azo_pw_limit.restype = C.c_int32
        L.azo_pw_limit.argtypes = [C.c_double, C.c_double, C.c_int32]
        L.azo_rng_u32.restype = C.c_uint32
        L.azo_rng_u32.argtypes = [C.c_uint64, C.c_int64, C.c_int32, C.c_int64, C.c_int32, C.c_int32]
        L.azo_noise.restype = None
        L.azo_noise.argtypes = [C.c_uint64, C.c_int64, C.c_int64, C.c_int32, C.POINTER(C.c_float), C.c_void_p]
        L.azo_mlp_forward.restype = None
        L.azo_mlp_forward.argtypes = [C.POINTER(_Cfg), C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
        L.azo_head_post.restype = None
        L.azo_head_post.argtypes = [C.POINTER(_Cfg), C.c_void_p, C.c_void_p]
        L.azo_sample_action.restype = C.c_float
        L.azo_sample_action.argtypes = [C.POINTER(_Cfg), C.c_void_p, C.c_float, C.c_void_p]
        L.azo_obs.restype = None
        L.azo_obs.argtypes = [C.POINTER(_Cfg), C.c_void_p, C.c_void_p]
        L.azo_env_step.restype = C.c_int
        L.azo_env_step.argtypes = [C.POINTER(_Cfg), C.c_void_p, C.c_float, C.c_void_p, C.POINTER(C.c_double), C.c_void_p]
        for n in ("expf", "expm1f", "tanhf"):
            f = getattr(L, "azo_det_" + n)
            f.restype, f.argtypes = C.c_float, [C.c_float]
        for n in ("sin", "cos", "log"):
            f = getattr(L, "azo_det_" + n)
            f.restype, f.argtypes = C.c_double, [C.c_double]
        L.azo_det_eval.restype, L.azo_det_eval.argtypes = C.c_int, [C.c_int32, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32]
        L.azo_rng_block_batch.restype = None
        L.azo_rng_block_batch.argtypes = [C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
        L.azo_mt_seed.restype, L.azo_mt_seed.argtypes = None, [C.c_void_p, C.c_uint64]
        L.azo_mt_u32.restype, L.azo_mt_u32.argtypes = C.c_uint32, [C.c_void_p]
        L.azo_mt_random.restype, L.azo_mt_random.argtypes = C.c_double, [C.c_void_p]
        L.azo_mt_below.restype, L.azo_mt_below.argtypes = C.c_int32, [C.c_void_p, C.c_int32]
        L.azo_torch_seed.restype, L.azo_torch_seed.argtypes = None, [C.c_void_p, C.c_uint64]
        L.azo_torch_uniform.restype, L.azo_torch_uniform.argtypes = C.c_double, [C.c_void_p]
        _lib = L
    return _lib


@dataclass
class Config:
    """Search + network configuration; field names follow the reference's constructor kwargs
    (mcts.py:316-327, :537-549) and make_policy (policies.py:806-818)."""
    variant: int = DISCRETE
    n_rollouts: int = 8
    num_actions: int = 2
    num_components: int = 2
    state_dim: int = 4
    hidden: int = 128
    n_hidden: int = 2
    activation: int = ACT_RELU
    math_mode: int = MATH_DET
    V_target_policy: str = "off_policy"
    puct_f32: int = 1
    use_eval_tape: int = 0
    c_uct: float = 1.5
    gamma: float = 1.0
    epsilon: float = 0.0
    c_pw: float = 1.0
    kappa: float = 0.5
    action_bound: float = 2.0
    log_std_min: float = -5.0
    log_std_max: float = 2.0
    seed: int = 34
    eval_mode: int = 0  # EVAL_FP32 | EVAL_Q8
    rng_mode: int = 0   # RNG_PHILOX | RNG_MT19937 (discrete search: CPython's generator, seeded with seed + tree id per search)
    # reward wrappers (rl/wrappers.py) around CartPole: reward of a step / of the terminating step
    reward_step: float = 1.0
    reward_terminal: float = 1.0
    env: Optional[str] = None  # None (the variant's own env) | MOUNTAIN_CAR_CONTINUOUS | MOUNTAIN_CAR | ACROBOT

    def c(self) -> _Cfg:
        return _Cfg(self.variant, self.n_rollouts, self.num_actions, self.num_components, self.state_dim, self.hidden,
                    self.n_hidden, self.activation, self.math_mode, VT[self.V_target_policy], self.puct_f32,
                    self.use_eval_tape, self.c_uct, self.gamma, self.epsilon, self.c_pw, self.kappa,
                    self.action_bound, self.log_std_min, self.log_std_max, self.seed, self.eval_mode, self.rng_mode,
                    self.reward_step, self.reward_terminal, _ENV[self.env])

    @property
    def rows(self) -> int:
        return self.n_rollouts + 2

    @property
    def hidden_dim(self) -> int:
        """Width of the env's hidden state (the search's root states and the dump's state rows)."""
        if self.env is None:
            return 4 if self.variant == DISCRETE else 2
        return 4 if self.env == ACROBOT else 2

    @property
    def head_dim(self) -> int:
        return lib().azo_head_dim(C.byref(self.c()))

    @property
    def num_weights(self) -> int:
        return lib().azo_num_weights(C.byref(self.c()))

    @property
    def cmax(self) -> int:
        if self.variant == DISCRETE:
            return self.num_actions
        return max(pw_limit(self.c_pw, self.kappa, self.n_rollouts), pw_limit(self.c_pw, self.kappa, 0)) + 1


def discrete_config(env: Optional[str] = None, **kw) -> Config:
    """run_discrete.yaml / MCTSDiscrete.yaml / DiscretePolicy.yaml defaults, with the env's own (see _ENV_DEFAULTS)."""
    d = dict(variant=DISCRETE, n_rollouts=8, num_actions=2, state_dim=4, hidden=128, n_hidden=2, activation=ACT_RELU,
             c_uct=1.5, gamma=1.0, epsilon=0.1, env=env)
    d.update(_ENV_DEFAULTS.get(env, {}))
    d.update(kw)
    return Config(**d)


def continuous_config(env: Optional[str] = None, **kw) -> Config:
    """run_continuous.yaml / MCTSContinuous.yaml / ContinuousPolicy.yaml defaults, with the env's own (see _ENV_DEFAULTS)."""
    d = dict(variant=CONTINUOUS, n_rollouts=25, num_components=2, state_dim=3, hidden=128, n_hidden=3,
             activation=ACT_ELU, c_uct=0.05, c_pw=1.0, kappa=0.5, gamma=1.0, epsilon=0.0, action_bound=2.0, env=env)
    d.update(_ENV_DEFAULTS.get(env, {}))
    d.update(kw)
    return Config(**d)


def pw_limit(c_pw: float, kappa: float, n: int) -> int:
    return lib().azo_pw_limit(c_pw, kappa, n)


def _p(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def search(cfg: Config, weights: Optional[np.ndarray], root_state: np.ndarray, root_n_init: Optional[np.ndarray] = None,
           tree_id0: int = 0, tapes: Optional[Dict[str, np.ndarray]] = None, dump: bool = True,
           n_threads: int = 1) -> Dict[str, np.ndarray]:
    """Run B independent searches on the CPU oracle from hidden env states [B, HS]; returns root results (+ full tree dump).
    Raises WrapCapReached where the engine fails with AZG_EWRAP."""
    L = lib()
    HS = cfg.hidden_dim
    root_state = np.ascontiguousarray(root_state, dtype=np.float64).reshape(-1, HS)
    B, R, A, K3 = root_state.shape[0], cfg.rows, cfg.num_actions, 3 * max(cfg.num_components, 1)
    cm = cfg.cmax
    out: Dict[str, np.ndarray] = dict(
        n_children=np.zeros(B, np.int32), actions=np.zeros((B, cm), np.float32), counts=np.zeros((B, cm), np.int32),
        Q=np.zeros((B, cm), np.float64), V_target=np.zeros(B, np.float64), counters=np.zeros(8, np.int64))
    res = _Res(cm, _p(out["n_children"]), _p(out["actions"]), _p(out["counts"]), _p(out["Q"]), _p(out["V_target"]),
               _p(out["counters"]))
    dd = dc = None
    if dump and cfg.variant == DISCRETE:
        d = dict(n_nodes=np.zeros(B, np.int32), parent=np.zeros((B, R), np.int32), paction=np.zeros((B, R), np.int32),
                 node_n=np.zeros((B, R), np.int32), terminal=np.zeros((B, R), np.int32), V=np.zeros((B, R), np.float32),
                 r=np.zeros((B, R), np.float64), state=np.zeros((B, R, HS), np.float64),
                 prior=np.zeros((B, R, A), np.float32), eW=np.zeros((B, R, A), np.float64),
                 en=np.zeros((B, R, A), np.int32), echild=np.zeros((B, R, A), np.int32))
        dd = _DumpD(*[_p(d[n]) for n, _ in _DumpD._fields_])
        out.update(d)
    elif dump:
        d = dict(n_rows=np.zeros(B, np.int32), parent=np.zeros((B, R), np.int32), action=np.zeros((B, R), np.float32),
                 eW=np.zeros((B, R), np.float64), en=np.zeros((B, R), np.int32), expanded=np.zeros((B, R), np.int32),
                 node_n=np.zeros((B, R), np.int32), terminal=np.zeros((B, R), np.int32), V=np.zeros((B, R), np.float32),
                 r=np.zeros((B, R), np.float64), state=np.zeros((B, R, HS), np.float64),
                 head=np.zeros((B, R, K3), np.float32))
        dc = _DumpC(*[_p(d[n]) for n, _ in _DumpC._fields_])
        out.update(d)
    tp = None
    keep = []
    if tapes is not None:
        tv = np.ascontiguousarray(tapes["V"], np.float32); keep.append(tv)
        tpr = np.ascontiguousarray(tapes["prior"], np.float32) if "prior" in tapes else None; keep.append(tpr)
        ta = np.ascontiguousarray(tapes["action"], np.float32) if "action" in tapes else None; keep.append(ta)
        assert tv.shape == (B, R), (tv.shape, (B, R))
        tp = _Tapes(_p(tv), _p(tpr), _p(ta))
    w = None
    if weights is not None:
        w = np.ascontiguousarray(weights, np.float32)
        assert w.size == cfg.num_weights, (w.size, cfg.num_weights)
    rn = None if root_n_init is None else np.ascontiguousarray(root_n_init, np.int32)
    rc = L.azo_search(C.byref(cfg.c()), _p(w), 0 if w is None else w.size, B, _p(root_state), _p(rn), tree_id0,
                      None if tp is None else C.byref(tp), C.byref(res), None if dd is None else C.byref(dd),
                      None if dc is None else C.byref(dc), n_threads)
    if rc == ERR_WRAP:
        raise WrapCapReached("an angle reached the wrap cap")
    if rc != 0:
        raise ValueError({-1: "Can't do tree search from a terminal node", -2: "bad oracle config",
                          -3: "NaN in UCT"}.get(rc, f"oracle error {rc}"))
    return out


def mlp_forward(cfg: Config, weights: np.ndarray, x: np.ndarray):
    x = np.ascontiguousarray(x, np.float32).reshape(-1, cfg.state_dim)
    w = np.ascontiguousarray(weights, np.float32)
    V = np.zeros(x.shape[0], np.float32)
    head = np.zeros((x.shape[0], cfg.head_dim), np.float32)
    lib().azo_mlp_forward(C.byref(cfg.c()), _p(w), x.shape[0], _p(x), _p(V), _p(head))
    return V, head


def head_post(cfg: Config, raw: np.ndarray) -> np.ndarray:
    raw = np.ascontiguousarray(raw, np.float32)
    n = cfg.num_actions if cfg.variant == DISCRETE else 3 * cfg.num_components
    out = np.zeros(n, np.float32)
    lib().azo_head_post(C.byref(cfg.c()), _p(raw), _p(out))
    return out


def sample_action(cfg: Config, head: np.ndarray, u: float, z: np.ndarray) -> float:
    head = np.ascontiguousarray(head, np.float32)
    z = np.ascontiguousarray(z, np.float32)
    return float(lib().azo_sample_action(C.byref(cfg.c()), _p(head), C.c_float(u), _p(z)))


def env_step(cfg: Config, state: np.ndarray, action: float):
    """One step of the config's env (discrete: the action index) -> (next hidden state, reward, done, f32 observation).
    Raises WrapCapReached where the engine fails with AZG_EWRAP."""
    s = np.ascontiguousarray(state, np.float64)
    o = np.zeros(cfg.hidden_dim, np.float64)
    obs = np.zeros(cfg.state_dim, np.float32)
    r = C.c_double()
    term = lib().azo_env_step(C.byref(cfg.c()), _p(s), C.c_float(action), _p(o), C.byref(r), _p(obs))
    if term == ERR_WRAP:
        raise WrapCapReached(state)
    return o, r.value, bool(term), obs


def obs(cfg: Config, state: np.ndarray) -> np.ndarray:
    """The network input (f32 observation) of a hidden state [HS] -> [S], or of states [n, HS] -> [n, S]."""
    s = np.ascontiguousarray(state, np.float64)
    rows = s.reshape(-1, cfg.hidden_dim)
    o = np.zeros((rows.shape[0], cfg.state_dim), np.float32)
    for i in range(rows.shape[0]):
        lib().azo_obs(C.byref(cfg.c()), _p(rows[i]), _p(o[i]))
    return o if s.ndim == 2 else o[0]


def rng_u32(seed: int, tree: int, stream: int, idx: int, block: int = 0, word: int = 0) -> int:
    return int(lib().azo_rng_u32(seed, tree, stream, idx, block, word))


def rng_blocks(seed: int, tree: np.ndarray, stream: np.ndarray, idx: np.ndarray, block: np.ndarray) -> np.ndarray:
    """The four Philox words of every counter (tree[i], stream[i], idx[i], block[i]) under key `seed`: uint32 [n, 4]."""
    tree, idx = np.ascontiguousarray(tree, np.int64), np.ascontiguousarray(idx, np.int64)
    stream, block = np.ascontiguousarray(stream, np.int32), np.ascontiguousarray(block, np.int32)
    out = np.empty((tree.size, 4), np.uint32)
    lib().azo_rng_block_batch(seed, _p(tree), _p(stream), _p(idx), _p(block), tree.size, _p(out))
    return out


FN_EXPF, FN_EXPM1F, FN_TANHF, FN_SIN, FN_COS, FN_LOG, FN_ACT = 0, 1, 2, 3, 4, 5, 16
_FN = {"expf": FN_EXPF, "expm1f": FN_EXPM1F, "tanhf": FN_TANHF, "sin": FN_SIN, "cos": FN_COS, "log": FN_LOG}


def det_eval(fn, x: np.ndarray, n_threads: int = 8) -> np.ndarray:
    """Deterministic function `fn` ("expf", "expm1f", "tanhf" on float32; "sin", "cos", "log" on float64; or an ACT_* code:
    the activation in MATH_DET mode, float32) over every element of x, in threaded C."""
    code = _FN[fn] if isinstance(fn, str) else FN_ACT + int(fn)
    dt = np.float64 if code in (FN_SIN, FN_COS, FN_LOG) else np.float32
    x = np.ascontiguousarray(x, dt)
    out = np.empty_like(x)
    rc = lib().azo_det_eval(code, _p(x), _p(out), x.size, n_threads)
    if rc != 0:
        raise ValueError(f"azo_det_eval: unknown function {fn!r}")
    return out


class MT19937:
    """The oracle's MT19937 generators (AZO_RNG_MT19937): kind "python" is CPython's `random` seeded with random.seed(seed),
    kind "torch" is torch's CPU generator after torch.manual_seed(seed)."""

    def __init__(self, seed: int, kind: str = "python"):
        self.kind = kind
        self.st = np.zeros(625, np.uint32)
        (lib().azo_mt_seed if kind == "python" else lib().azo_torch_seed)(_p(self.st), seed)

    def u32(self) -> int:
        return int(lib().azo_mt_u32(_p(self.st)))

    def random(self) -> float:
        return lib().azo_mt_random(_p(self.st))

    def below(self, n: int) -> int:
        return int(lib().azo_mt_below(_p(self.st), n))

    def uniform(self) -> float:
        return lib().azo_torch_uniform(_p(self.st))


def noise(seed: int, tree: int, j: int, K: int):
    u = C.c_float()
    z = np.zeros(max(K, 1), np.float32)
    lib().azo_noise(seed, tree, j, K, C.byref(u), _p(z))
    return u.value, z


def flatten_state_dict(sd) -> np.ndarray:
    """state_dict (trunk.*, value_head.*, dist_head.*; policies.py:101-120,255-259) -> flat f32."""
    keys = [k for k in sd.keys() if k.startswith("trunk.")] + ["value_head.weight", "value_head.bias",
                                                               "dist_head.weight", "dist_head.bias"]
    return np.concatenate([np.asarray(sd[k].detach().cpu().numpy(), np.float32).ravel() for k in keys])
