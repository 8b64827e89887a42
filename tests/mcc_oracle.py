"""CPU reference of the MountainCarContinuous-v0 search (test infrastructure; the checker of AZG_FLAG_ENV_MOUNTAIN_CAR_CONTINUOUS).

* `Continuous_MountainCarEnv`: gym 0.17-0.19 classic_control/continuous_mountain_car.py, step() as gym writes it, in plain Python.
* `search` / `env_step`: tests/mcc_oracle.c -- the CPU oracle (oracle/azg_oracle.c, included unchanged) with this env in its continuous
  search; same configs (oracle.azo.Config), same output dicts as oracle.azo.search / env_step.
* `selfplay_run`: oracle/selfplay.py's episode loop for this env (Env.reset: position ~ U(-0.6, -0.4) from Philox stream 3, velocity 0).

The library is compiled on first use with oracle/Makefile's flags into a temporary directory (never into the tree).
"""
from __future__ import annotations

import ctypes as C
import dataclasses
import hashlib
import math
import os
import subprocess
import tempfile
from typing import Dict, List, Optional

import numpy as np

from oracle import azo
from oracle import selfplay as osp

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORACLE = os.path.join(os.path.dirname(_HERE), "oracle")
_SRC = os.path.join(_HERE, "mcc_oracle.c")
CFLAGS = ["-O2", "-ftree-vectorize", "-mavx2", "-mfma", "-ffp-contract=off", "-fno-math-errno", "-pthread", "-fPIC", "-std=gnu11"]
R_SCALE = 16.2736044  # mcts.py:20
_lib = None


class Continuous_MountainCarEnv:  # noqa: N801 -- gym's class name, which the drop-in search classes recognise
    """gym 0.17-0.19 classic_control/continuous_mountain_car.py.  The f32 action enters f64 arithmetic exactly (numpy-1.x promotion
    of the reference's pinned numpy; under NEP 50 np.float32 * float would stay f32, hence the explicit float()).  `cos` is math.cos;
    the engine's bit-exact twin is the deterministic cosine (pass cos=det_cos)."""
    min_action, max_action = -1.0, 1.0
    min_position, max_position, max_speed = -1.2, 0.6, 0.07
    goal_position, goal_velocity, power = 0.45, 0, 0.0015

    def __init__(self, state, cos=math.cos):
        self.state = np.array(state, dtype=np.float64)
        self.cos = cos

    @property
    def unwrapped(self):
        return self

    def obs(self):
        return np.array(self.state, dtype=np.float64)

    def step(self, action):
        position, velocity = float(self.state[0]), float(self.state[1])
        a = float(np.asarray(action, dtype=np.float32).ravel()[0])
        force = min(max(a, self.min_action), self.max_action)
        velocity += force * self.power - 0.0025 * self.cos(3 * position)
        if velocity > self.max_speed:
            velocity = self.max_speed
        if velocity < -self.max_speed:
            velocity = -self.max_speed
        position += velocity
        if position > self.max_position:
            position = self.max_position
        if position < self.min_position:
            position = self.min_position
        if position == self.min_position and velocity < 0:
            velocity = 0
        done = bool(position >= self.goal_position and velocity >= self.goal_velocity)
        reward = 0
        if done:
            reward = 100.0
        reward -= math.pow(a, 2) * 0.1
        self.state = np.array([position, velocity], dtype=np.float64)
        return self.obs(), reward, done, {}


def det_cos(x: float) -> float:
    return float(azo.det_eval("cos", np.array([x]), n_threads=1)[0])


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha256()
        for p in (_SRC, os.path.join(_ORACLE, "azg_oracle.c"), os.path.join(_ORACLE, "azg_oracle.h")):
            h.update(open(p, "rb").read())
        out = os.path.join(tempfile.gettempdir(), f"libmcc_oracle_{os.getuid()}_{h.hexdigest()[:16]}.so")
        if not os.path.exists(out):
            tmp = f"{out}.{os.getpid()}"
            subprocess.check_call(["gcc"] + CFLAGS + ["-shared", "-I", _ORACLE, "-o", tmp, _SRC, "-lm"])
            os.replace(tmp, out)
        L = C.CDLL(out)
        L.mcc_search.restype = C.c_int
        L.mcc_search.argtypes = [C.POINTER(azo._Cfg), C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_int64, C.POINTER(azo._Tapes),
                                 C.POINTER(azo._Res), C.POINTER(azo._DumpC), C.c_int32]
        L.mcc_env_step.restype = C.c_int
        L.mcc_env_step.argtypes = [C.POINTER(azo._Cfg), C.c_void_p, C.c_float, C.c_void_p, C.POINTER(C.c_double), C.c_void_p]
        _lib = L
    return _lib


def config(**kw) -> azo.Config:
    """ContinuousPolicy.yaml / MCTSContinuous.yaml defaults with the env's observation (2 entries) and action bound (1.0)."""
    d = dict(state_dim=2, action_bound=1.0)
    d.update(kw)
    return azo.continuous_config(**d)


def env_step(cfg: azo.Config, state: np.ndarray, action: float):
    s = np.ascontiguousarray(state, np.float64)
    o = np.zeros(2, np.float64)
    obs = np.zeros(2, np.float32)
    r = C.c_double()
    term = lib().mcc_env_step(C.byref(cfg.c()), s.ctypes.data_as(C.c_void_p), C.c_float(action), o.ctypes.data_as(C.c_void_p),
                              C.byref(r), obs.ctypes.data_as(C.c_void_p))
    return o, r.value, bool(term), obs


def search(cfg: azo.Config, weights: Optional[np.ndarray], root_state: np.ndarray, tree_id0: int = 0,
           tapes: Optional[Dict[str, np.ndarray]] = None, dump: bool = True, n_threads: int = 1) -> Dict[str, np.ndarray]:
    """B independent searches; the same dict as oracle.azo.search for the continuous variant."""
    p = azo._p
    root_state = np.ascontiguousarray(root_state, dtype=np.float64).reshape(-1, 2)
    B, R, K3, cm = root_state.shape[0], cfg.rows, 3 * max(cfg.num_components, 1), cfg.cmax
    out: Dict[str, np.ndarray] = dict(
        n_children=np.zeros(B, np.int32), actions=np.zeros((B, cm), np.float32), counts=np.zeros((B, cm), np.int32),
        Q=np.zeros((B, cm), np.float64), V_target=np.zeros(B, np.float64), counters=np.zeros(8, np.int64))
    res = azo._Res(cm, p(out["n_children"]), p(out["actions"]), p(out["counts"]), p(out["Q"]), p(out["V_target"]), p(out["counters"]))
    dc = None
    if dump:
        d = dict(n_rows=np.zeros(B, np.int32), parent=np.zeros((B, R), np.int32), action=np.zeros((B, R), np.float32),
                 eW=np.zeros((B, R), np.float64), en=np.zeros((B, R), np.int32), expanded=np.zeros((B, R), np.int32),
                 node_n=np.zeros((B, R), np.int32), terminal=np.zeros((B, R), np.int32), V=np.zeros((B, R), np.float32),
                 r=np.zeros((B, R), np.float64), state=np.zeros((B, R, 2), np.float64), head=np.zeros((B, R, K3), np.float32))
        dc = azo._DumpC(*[p(d[n]) for n, _ in azo._DumpC._fields_])
        out.update(d)
    tp, keep = None, []
    if tapes is not None:
        tv = np.ascontiguousarray(tapes["V"], np.float32)
        ta = np.ascontiguousarray(tapes["action"], np.float32)
        keep += [tv, ta]
        tp = azo._Tapes(p(tv), None, p(ta))
    w = None if weights is None else np.ascontiguousarray(weights, np.float32)
    rc = lib().mcc_search(C.byref(cfg.c()), p(w), 0 if w is None else w.size, B, p(root_state), tree_id0,
                          None if tp is None else C.byref(tp), C.byref(res), None if dc is None else C.byref(dc), n_threads)
    if rc != 0:
        raise ValueError({-2: "bad oracle config", -3: "NaN in UCT"}.get(rc, f"oracle error {rc}"))
    return out


def selfplay_run(cfg: azo.Config, weights: np.ndarray, states0: np.ndarray, steps: int, max_episode_length: int, seed: int = 34,
                 tree_id0: int = 0, by_value: bool = False, n_threads: int = 4) -> List[Dict[str, np.ndarray]]:
    """oracle/selfplay.py's loop (continuous agent: actions[counts.argmax()], or Q.argmax() by value) for this env."""
    state = np.array(states0, np.float64).copy()
    B = state.shape[0]
    ep_step, episode = np.zeros(B, np.int32), np.zeros(B, np.int32)
    out = []
    for s in range(steps):
        key = osp.step_seed(seed, s)
        c = dataclasses.replace(cfg, seed=key)
        res = search(c, weights, state, tree_id0=tree_id0, dump=False, n_threads=n_threads)
        rec = dict(obs=state.astype(np.float32), actions=res["actions"].copy(), counts=res["counts"].copy(), Q=res["Q"].copy(),
                   V_target=res["V_target"].copy(), n_children=res["n_children"].copy(), action_taken=np.zeros(B, np.float32),
                   reward=np.zeros(B, np.float64), done=np.zeros(B, np.int32))
        for t in range(B):
            nk = int(res["n_children"][t])
            a = int(np.argmax(res["Q"][t, :nk] if by_value else res["counts"][t, :nk]))
            action = float(res["actions"][t, a])
            nxt, r, term, _ = env_step(c, state[t], action)
            step = int(ep_step[t]) + 1
            done = term or step >= max_episode_length
            if done:
                episode[t] += 1
                u = osp._unit(azo.rng_u32(key, tree_id0 + t, 3, int(episode[t]), 0, 0))
                nxt = np.array([-0.6 + (-0.4 - -0.6) * u, 0.0])
            ep_step[t] = 0 if done else step
            state[t] = nxt
            rec["action_taken"][t], rec["reward"][t], rec["done"][t] = action, r, int(done)
        rec.update(env_state=state.copy(), ep_step=ep_step.copy(), episode=episode.copy())
        out.append(rec)
    return out
