"""SearchEngine: thin host wrapper over the C ABI (include/azg.h) for batches of independent trees.

PyTorch is plumbing only (device tensors, streams); all search / env / network arithmetic runs in
libazg.so's CUDA kernels.  There is no CPU path: constructing an engine without CUDA raises.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Dict, Optional

import numpy as np
import torch

from . import _cabi
from ._cabi import ACT_ELU, ACT_RELU, CONTINUOUS, DISCRETE, VT, AzgConfig, check

# the envs the engine steps (gym ids); the discrete search steps CartPole-v0 and the continuous search Pendulum-v0 unless told otherwise
CARTPOLE, PENDULUM, MOUNTAIN_CAR_CONTINUOUS = "CartPole-v0", "Pendulum-v0", "MountainCarContinuous-v0"
MOUNTAIN_CAR, ACROBOT = "MountainCar-v0", "Acrobot-v1"


@dataclass
class EngineConfig:
    """Reference constructor kwargs (alphazero/search/mcts.py:316-327, :537-549) + network shape
    (alphazero/network/policies.py:806-818) + engine capacity."""
    variant: int = DISCRETE
    max_rollouts: int = 8
    max_trees: int = 1
    num_actions: int = 2
    num_components: int = 2
    state_dim: int = 4
    hidden: int = 128
    n_hidden: int = 2
    activation: int = ACT_RELU
    V_target_policy: str = "off_policy"
    puct_f32: int = 1
    device: int = 0
    c_uct: float = 1.5
    gamma: float = 1.0
    epsilon: float = 0.0
    c_pw: float = 1.0
    kappa: float = 0.5
    action_bound: float = 2.0
    log_std_min: float = -5.0
    log_std_max: float = 2.0
    seed: int = 34
    use_graph: bool = True
    # AZG_FLAG_EVAL_Q8: hidden x hidden layers on tcgen05 as exact int8-sliced products (include/azg.h).  None = on wherever the
    # tensor-core kernel serves the network (hidden 128, 2 or 3 hidden layers, at most 15 head outputs): the drop-in classes, the
    # self-play driver and bench.py all run the same evaluation; False selects the FP32 FMA kernel (mlp.cuh).  Every other hidden
    # width (a multiple of 32 up to 256) runs the FP32 kernel that streams the hidden layers (mlp_stream.cuh), which None picks
    eval_q8: Optional[bool] = None
    rng_mt19937: bool = False  # AZG_FLAG_RNG_MT19937: CPython's generator for the discrete search's selection draws (include/azg.h)
    fused: Optional[bool] = None  # AZG_FLAG_FUSED: whole search in one persistent kernel; None = on where supported (eval_q8, so
    # hidden 128 only: the other widths run one launch per simulation)
    # the env the search steps: None = the variant's own (CartPole-v0 / Pendulum-v0); MOUNTAIN_CAR_CONTINUOUS (continuous variant,
    # state_dim 2) sets AZG_FLAG_ENV_MOUNTAIN_CAR_CONTINUOUS; MOUNTAIN_CAR (discrete variant, num_actions 3, state_dim 2) sets
    # AZG_FLAG_ENV_MOUNTAIN_CAR; ACROBOT (discrete variant, num_actions 3, state_dim 6) sets AZG_FLAG_ENV_ACROBOT
    env: Optional[str] = None

    def c(self) -> AzgConfig:
        return AzgConfig(self.variant, self.max_rollouts, self.max_trees, self.num_actions, self.num_components,
                         self.state_dim, self.hidden, self.n_hidden, self.activation, VT[self.V_target_policy],
                         self.puct_f32, self.device, self.c_uct, float(self.gamma), self.epsilon, self.c_pw, self.kappa,
                         self.action_bound, self.log_std_min, self.log_std_max,
                         (0 if self.use_graph else _cabi.FLAG_NO_GRAPH) | (_cabi.FLAG_EVAL_Q8 if self.is_q8() else 0)
                         | (_cabi.FLAG_FUSED if self.is_fused() else 0) | (_cabi.FLAG_RNG_MT19937 if self.rng_mt19937 else 0)
                         | (_cabi.FLAG_ENV_MOUNTAIN_CAR_CONTINUOUS if self.env_name() == MOUNTAIN_CAR_CONTINUOUS else 0)
                         | (_cabi.FLAG_ENV_MOUNTAIN_CAR if self.env_name() == MOUNTAIN_CAR else 0)
                         | (_cabi.FLAG_ENV_ACROBOT if self.env_name() == ACROBOT else 0), self.seed)

    def env_name(self) -> str:
        if self.env is None:
            return CARTPOLE if self.variant == DISCRETE else PENDULUM
        if self.env not in (CARTPOLE, PENDULUM, MOUNTAIN_CAR_CONTINUOUS, MOUNTAIN_CAR, ACROBOT):
            raise ValueError(f"unknown env {self.env!r}: the engine steps {CARTPOLE}, {MOUNTAIN_CAR}, {ACROBOT}, {PENDULUM} and "
                             f"{MOUNTAIN_CAR_CONTINUOUS}")
        if self.env in (MOUNTAIN_CAR, ACROBOT) and self.variant != DISCRETE:
            raise ValueError(f"{self.env} has discrete actions: it is searched by the discrete variant")
        return self.env

    def q8_supported(self) -> bool:
        head = self.num_actions if self.variant == DISCRETE else (3 * self.num_components if self.num_components > 1 else 2)
        return self.hidden == 128 and self.n_hidden in (2, 3) and 1 + head <= 16 and self.activation in (ACT_RELU, ACT_ELU)

    def is_q8(self) -> bool:
        return self.q8_supported() if self.eval_q8 is None else bool(self.eval_q8)

    def is_fused(self) -> bool:
        env_dim = {CARTPOLE: 4, PENDULUM: 3, MOUNTAIN_CAR_CONTINUOUS: 2, MOUNTAIN_CAR: 2, ACROBOT: 6}[self.env_name()]
        supported = (self.is_q8() and self.state_dim == env_dim
                     and not (self.rng_mt19937 and self.variant == CONTINUOUS))  # the torch-generator mode runs one launch per simulation
        return supported if self.fused is None else bool(self.fused)


def flatten_state_dict(sd) -> np.ndarray:
    """state_dict -> flat f32 in the order azg_set_weights expects (policies.py:101-120, :255-259, :434, :588)."""
    keys = [k for k in sd.keys() if k.startswith("trunk.")] + ["value_head.weight", "value_head.bias",
                                                               "dist_head.weight", "dist_head.bias"]
    return np.concatenate([sd[k].detach().cpu().numpy().astype(np.float32).ravel() for k in keys])


def _ptr(t) -> Optional[int]:
    if t is None:
        return None
    if isinstance(t, torch.Tensor):
        return t.data_ptr()
    return t.ctypes.data


class SearchEngine:
    def __init__(self, cfg: EngineConfig):
        self._h = None
        self._lib = _cabi.load()  # raises ImportError if libazg.so has not been built
        if not torch.cuda.is_available():
            raise RuntimeError("alphazero_gym_b200 needs a CUDA device (no CPU fallback)")
        self.cfg = cfg
        h = C.c_void_p()
        check(self._lib.azg_create(C.byref(cfg.c()), C.byref(h)))
        self._h = h
        self.device = torch.device("cuda", cfg.device)
        self.rows = self._lib.azg_rows(h)
        self.cmax = self._lib.azg_cmax(h)
        self.head_dim = self._lib.azg_head_dim(h)
        self.num_weights = self._lib.azg_num_weights(h)
        self.state_cols = 4 if cfg.variant == DISCRETE and cfg.env_name() in (CARTPOLE, ACROBOT) else 2  # hidden-state width
        self._keep = {}
        self.last_B = 0

    def close(self) -> None:
        if self._h is not None:
            self._lib.azg_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @staticmethod
    def _stream() -> int:
        return torch.cuda.current_stream().cuda_stream

    # ---- weights -------------------------------------------------------------------------------------
    def set_weights(self, flat) -> None:
        if isinstance(flat, torch.Tensor):
            flat = flat.detach().to(torch.float32).contiguous()
            n = flat.numel()
        else:
            flat = np.ascontiguousarray(flat, np.float32)
            n = flat.size
        with torch.cuda.device(self.device):
            check(self._lib.azg_set_weights(self._h, _ptr(flat), n, self._stream()))

    def set_weights_from_model(self, model) -> None:
        self.set_weights(flatten_state_dict(model.state_dict()))

    # ---- device-resident path ------------------------------------------------------------------------
    def search(self, root_state: torch.Tensor, n_rollouts: int, root_n_init: Optional[torch.Tensor] = None,
               tree_id0: int = 0) -> None:
        """Batched search; root_state is a CUDA f64 tensor [B, 4|2] (CartPole and Acrobot 4, the other envs 2).  Asynchronous on the current stream."""
        assert root_state.is_cuda and root_state.dtype == torch.float64 and root_state.is_contiguous()
        B = root_state.shape[0]
        assert root_state.shape[1] == self.state_cols
        with torch.cuda.device(self.device):
            if self.cfg.variant == DISCRETE:
                if root_n_init is not None:
                    assert root_n_init.is_cuda and root_n_init.dtype == torch.int32 and root_n_init.numel() == B
                check(self._lib.azg_search_discrete(self._h, B, _ptr(root_state), _ptr(root_n_init), n_rollouts, tree_id0,
                                                    self._stream()))
            else:
                assert root_n_init is None
                check(self._lib.azg_search_continuous(self._h, B, _ptr(root_state), n_rollouts, tree_id0, self._stream()))
        self.last_B = B

    def root_results(self, B: Optional[int] = None, out: Optional[Dict[str, torch.Tensor]] = None) -> Dict[str, torch.Tensor]:
        """return_results of every tree as device tensors; `out` (a dict from an earlier call) is overwritten in place if given."""
        B = B or self.last_B
        dev = self.device
        if out is None:
            out = dict(actions=torch.empty((B, self.cmax), dtype=torch.float32, device=dev),
                       counts=torch.empty((B, self.cmax), dtype=torch.int32, device=dev),
                       Q=torch.empty((B, self.cmax), dtype=torch.float64, device=dev),
                       V_target=torch.empty(B, dtype=torch.float64, device=dev),
                       n_children=torch.empty(B, dtype=torch.int32, device=dev))
        assert out["actions"].shape == (B, self.cmax) and out["Q"].dtype == torch.float64
        with torch.cuda.device(dev):
            check(self._lib.azg_root_results(self._h, B, _ptr(out["actions"]), _ptr(out["counts"]), _ptr(out["Q"]),
                                             _ptr(out["V_target"]), _ptr(out["n_children"]), self._stream()))
        return out

    def profile_search(self, root_state: torch.Tensor, n_rollouts: int, tree_id0: int = 0) -> Dict[str, Dict[str, float]]:
        """One search with a CUDA-event pair around every kernel launch (azg_profile_search)."""
        assert root_state.is_cuda and root_state.dtype == torch.float64 and root_state.is_contiguous()
        B = root_state.shape[0]
        ms, n = (C.c_float * 3)(), (C.c_int32 * 3)()
        with torch.cuda.device(self.device):
            check(self._lib.azg_profile_search(self._h, B, _ptr(root_state), None, n_rollouts, tree_id0, self._stream(),
                                               C.byref(ms), C.byref(n)))
        self.last_B = B
        return {k: dict(ms=float(ms[i]), launches=int(n[i])) for i, k in enumerate(("tree_step", "evaluation", "setup"))}

    def status(self) -> None:
        with torch.cuda.device(self.device):
            check(self._lib.azg_status(self._h, self._stream()))

    def set_reward_model(self, reward_step: float = 1.0, reward_terminal: float = 1.0) -> None:
        """Reward wrappers of rl/wrappers.py around the searched CartPole env (azg_set_reward_model): reward of a step / of the
        terminating step.  Defaults = the plain env."""
        check(self._lib.azg_set_reward_model(self._h, float(reward_step), float(reward_terminal)))

    # ---- host-buffer path (what MCTS*.search + return_results cost end to end) ---------------------
    def host_buffers(self, B: int) -> Dict[str, np.ndarray]:
        """Page-locked result buffers for search_host(out=...): the engine DMAs into them directly (no staging copy)."""
        t = dict(actions=torch.empty((B, self.cmax), dtype=torch.float32).pin_memory(),
                 counts=torch.empty((B, self.cmax), dtype=torch.int32).pin_memory(),
                 Q=torch.empty((B, self.cmax), dtype=torch.float64).pin_memory(),
                 V_target=torch.empty(B, dtype=torch.float64).pin_memory(),
                 n_children=torch.empty(B, dtype=torch.int32).pin_memory())
        self._keep[("host_buffers", B)] = t
        return {k: v.numpy() for k, v in t.items()}

    def search_host(self, root_state: np.ndarray, n_rollouts: int, root_n_init: Optional[np.ndarray] = None,
                    tree_id0: int = 0, out: Optional[Dict[str, np.ndarray]] = None) -> Dict[str, np.ndarray]:
        """Host buffers in, host buffers out (azg_search_host).  `out` (e.g. from host_buffers) is reused if given."""
        rs = np.ascontiguousarray(root_state, np.float64).reshape(-1, self.state_cols)
        B = rs.shape[0]
        rn = None if root_n_init is None else np.ascontiguousarray(root_n_init, np.int32)
        if out is None:
            out = dict(actions=np.empty((B, self.cmax), np.float32), counts=np.empty((B, self.cmax), np.int32),
                       Q=np.empty((B, self.cmax), np.float64), V_target=np.empty(B, np.float64),
                       n_children=np.empty(B, np.int32))
        assert out["actions"].shape == (B, self.cmax) and out["Q"].dtype == np.float64
        check(self._lib.azg_search_host(self._h, B, _ptr(rs), _ptr(rn), n_rollouts, tree_id0, _ptr(out["actions"]),
                                        _ptr(out["counts"]), _ptr(out["Q"]), _ptr(out["V_target"]), _ptr(out["n_children"])))
        self.last_B = B
        return out

    def search_host_begin(self, slot: int, root_state: np.ndarray, n_rollouts: int, out: Dict[str, np.ndarray],
                          root_n_init: Optional[np.ndarray] = None, tree_id0: int = 0) -> None:
        """Pipelined search_host (azg_search_host_begin): returns at once; `root_state`, `root_n_init` and the `out` buffers
        (host_buffers) must be page-locked and stay untouched until search_host_end(slot)."""
        B = root_state.shape[0]
        assert root_state.dtype == np.float64 and root_state.flags.c_contiguous and out["actions"].shape == (B, self.cmax)
        check(self._lib.azg_search_host_begin(self._h, slot, B, _ptr(root_state), _ptr(root_n_init), n_rollouts, tree_id0,
                                              _ptr(out["actions"]), _ptr(out["counts"]), _ptr(out["Q"]), _ptr(out["V_target"]),
                                              _ptr(out["n_children"])))
        self.last_B = B

    def search_host_end(self, slot: int) -> None:
        """Blocks until the results of `slot` are in its host buffers (azg_search_host_end)."""
        check(self._lib.azg_search_host_end(self._h, slot))

    # ---- parity hooks ----------------------------------------------------------------------------------
    def set_tapes(self, V: Optional[np.ndarray], prior: Optional[np.ndarray] = None,
                  action: Optional[np.ndarray] = None) -> None:
        """Evaluator injection: per-tree tapes indexed by node / row creation order, stride `rows`."""
        if V is None:
            self._keep.pop("tapes", None)
            check(self._lib.azg_set_tapes(self._h, None, None, None))
            return
        tv = torch.from_numpy(np.ascontiguousarray(V, np.float32)).to(self.device)
        assert tv.shape[1] == self.rows, (tv.shape, self.rows)
        tp = None if prior is None else torch.from_numpy(np.ascontiguousarray(prior, np.float32)).to(self.device)
        ta = None if action is None else torch.from_numpy(np.ascontiguousarray(action, np.float32)).to(self.device)
        self._keep["tapes"] = (tv, tp, ta)
        check(self._lib.azg_set_tapes(self._h, _ptr(tv), _ptr(tp), _ptr(ta)))

    def dump_tree(self, B: Optional[int] = None) -> Dict[str, np.ndarray]:
        B = B or self.last_B
        R, A, K3 = self.rows, self.cfg.num_actions, 3 * max(self.cfg.num_components, 1)
        if self.cfg.variant == DISCRETE:
            d = dict(n_nodes=np.zeros(B, np.int32), parent=np.zeros((B, R), np.int32), paction=np.zeros((B, R), np.int32),
                     node_n=np.zeros((B, R), np.int32), terminal=np.zeros((B, R), np.int32), V=np.zeros((B, R), np.float32),
                     r=np.zeros((B, R), np.float64), state=np.zeros((B, R, self.state_cols), np.float64),
                     prior=np.zeros((B, R, A), np.float32), eW=np.zeros((B, R, A), np.float64),
                     en=np.zeros((B, R, A), np.int32), echild=np.zeros((B, R, A), np.int32))
            s = _cabi.DumpDiscrete(*[d[n].ctypes.data for n in _cabi.DumpDiscrete.FIELDS])
            check(self._lib.azg_dump_tree_discrete(self._h, B, C.byref(s)))
        else:
            d = dict(n_rows=np.zeros(B, np.int32), parent=np.zeros((B, R), np.int32), action=np.zeros((B, R), np.float32),
                     eW=np.zeros((B, R), np.float64), en=np.zeros((B, R), np.int32), expanded=np.zeros((B, R), np.int32),
                     node_n=np.zeros((B, R), np.int32), terminal=np.zeros((B, R), np.int32), V=np.zeros((B, R), np.float32),
                     r=np.zeros((B, R), np.float64), state=np.zeros((B, R, 2), np.float64),
                     head=np.zeros((B, R, K3), np.float32))
            s = _cabi.DumpContinuous(*[d[n].ctypes.data for n in _cabi.DumpContinuous.FIELDS])
            check(self._lib.azg_dump_tree_continuous(self._h, B, C.byref(s)))
        return d

    def counters(self, B: Optional[int] = None) -> Dict[str, int]:
        B = B or self.last_B
        arr = (C.c_int64 * 8)()
        check(self._lib.azg_get_counters(self._h, B, C.byref(arr)))
        names = ("sims", "levels", "children_scanned", "pw_inserts", "evals", "rng_draws", "terminal_leaf_sims", "launches")
        return dict(zip(names, [int(v) for v in arr]))

    def fused_stats(self) -> Dict[str, float]:
        """Cycle accounting of the whole-search kernel since the last call (azg_fused_stats), as fractions of the kernel time."""
        arr = (C.c_int64 * 8)()
        check(self._lib.azg_fused_stats(self._h, C.byref(arr)))
        tot = max(1, int(arr[0]))
        kind = {1: "two_phase", 2: "warpgroups", 3: "two_phase_trees_in_shared_memory"}.get(int(arr[5]), "none")
        return {"ctas": int(arr[4]), "kernel_cycles_per_cta": tot / max(1, int(arr[4])), "tree_phase": arr[1] / tot,
                "wait_for_post_processing": arr[2] / tot, "x_wait_mma": arr[3] / tot, "kernel": kind}

    # ---- standalone kernels (known-answer tests) ---------------------------------------------------------
    def mlp_forward(self, x: np.ndarray):
        xt = torch.from_numpy(np.ascontiguousarray(x, np.float32).reshape(-1, self.cfg.state_dim)).to(self.device)
        n = xt.shape[0]
        V = torch.empty(n, dtype=torch.float32, device=self.device)
        head = torch.empty((n, self.head_dim), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            check(self._lib.azg_mlp_forward(self._h, n, _ptr(xt), _ptr(V), _ptr(head), self._stream()))
        return V.cpu().numpy(), head.cpu().numpy()

    def env_step(self, state: np.ndarray, action: np.ndarray):
        st = torch.from_numpy(np.ascontiguousarray(state, np.float64).reshape(-1, self.state_cols)).to(self.device)
        n = st.shape[0]
        a = torch.from_numpy(np.ascontiguousarray(action, np.float32).reshape(n)).to(self.device)
        nxt = torch.empty_like(st)
        rew = torch.empty(n, dtype=torch.float64, device=self.device)
        term = torch.empty(n, dtype=torch.int32, device=self.device)
        obs = torch.empty((n, self.cfg.state_dim), dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            check(self._lib.azg_env_step(self._h, n, _ptr(st), _ptr(a), _ptr(nxt), _ptr(rew), _ptr(term), _ptr(obs),
                                         self._stream()))
        return nxt.cpu().numpy(), rew.cpu().numpy(), term.cpu().numpy(), obs.cpu().numpy()
