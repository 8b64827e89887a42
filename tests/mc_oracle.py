"""CPU reference of the MountainCar-v0 search (test infrastructure; the checker of AZG_FLAG_ENV_MOUNTAIN_CAR).

* `MountainCarEnv`: gym 0.17-0.19 classic_control/mountain_car.py, step() as gym writes it, in plain Python.
* `search` / `env_step`: tests/mc_oracle.c -- the CPU oracle (oracle/azg_oracle.c, included unchanged) with this env in its discrete
  search; same configs (oracle.azo.Config), same output dicts as oracle.azo.search (the dump's state is 2 wide).
* `selfplay_run`: oracle/selfplay.py's episode loop for this env (Env.reset: position ~ U(-0.6, -0.4) from Philox stream 3, velocity 0)
  and three actions.

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
_SRC = os.path.join(_HERE, "mc_oracle.c")
CFLAGS = ["-O2", "-ftree-vectorize", "-mavx2", "-mfma", "-ffp-contract=off", "-fno-math-errno", "-pthread", "-fPIC", "-std=gnu11"]
_lib = None


class MountainCarEnv:  # gym's class name, which the drop-in search classes recognise
    """gym 0.17-0.19 classic_control/mountain_car.py.  `cos` is math.cos; the engine's bit-exact twin is the deterministic cosine
    (pass cos=det_cos)."""
    min_position, max_position, max_speed = -1.2, 0.6, 0.07
    goal_position, goal_velocity = 0.5, 0
    force, gravity = 0.001, 0.0025

    def __init__(self, state=(-0.5, 0.0), cos=math.cos):
        self.state = np.array(state, dtype=np.float64)
        self.cos = cos

    @property
    def unwrapped(self):
        return self

    def step(self, action):
        position, velocity = self.state
        velocity += (int(action) - 1) * self.force + self.cos(3 * position) * (-self.gravity)
        velocity = np.clip(velocity, -self.max_speed, self.max_speed)
        position += velocity
        position = np.clip(position, self.min_position, self.max_position)
        if position == self.min_position and velocity < 0:
            velocity = 0
        done = bool(position >= self.goal_position and velocity >= self.goal_velocity)
        reward = -1.0
        self.state = (position, velocity)
        return np.array(self.state), reward, done, {}


def det_cos(x: float) -> float:
    return float(azo.det_eval("cos", np.array([float(x)]), n_threads=1)[0])


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha256()
        for p in (_SRC, os.path.join(_ORACLE, "azg_oracle.c"), os.path.join(_ORACLE, "azg_oracle.h")):
            h.update(open(p, "rb").read())
        out = os.path.join(tempfile.gettempdir(), f"libmc_oracle_{os.getuid()}_{h.hexdigest()[:16]}.so")
        if not os.path.exists(out):
            tmp = f"{out}.{os.getpid()}"
            subprocess.check_call(["gcc"] + CFLAGS + ["-shared", "-I", _ORACLE, "-o", tmp, _SRC, "-lm"])
            os.replace(tmp, out)
        L = C.CDLL(out)
        L.mc_search.restype = C.c_int
        L.mc_search.argtypes = [C.POINTER(azo._Cfg), C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64,
                                C.POINTER(azo._Tapes), C.POINTER(azo._Res), C.POINTER(azo._DumpD), C.c_int32]
        L.mc_env_step.restype = C.c_int
        L.mc_env_step.argtypes = [C.POINTER(azo._Cfg), C.c_void_p, C.c_int32, C.c_void_p, C.POINTER(C.c_double), C.c_void_p]
        _lib = L
    return _lib


def config(**kw) -> azo.Config:
    """DiscretePolicy.yaml / MCTSDiscrete.yaml defaults with the env's observation (2 entries) and 3 actions."""
    d = dict(state_dim=2, num_actions=3)
    d.update(kw)
    return azo.discrete_config(**d)


def env_step(cfg: azo.Config, state: np.ndarray, action: int):
    s = np.ascontiguousarray(state, np.float64)
    o = np.zeros(2, np.float64)
    obs = np.zeros(2, np.float32)
    r = C.c_double()
    term = lib().mc_env_step(C.byref(cfg.c()), s.ctypes.data_as(C.c_void_p), int(action), o.ctypes.data_as(C.c_void_p), C.byref(r),
                             obs.ctypes.data_as(C.c_void_p))
    return o, r.value, bool(term), obs


def search(cfg: azo.Config, weights: Optional[np.ndarray], root_state: np.ndarray, root_n_init: Optional[np.ndarray] = None,
           tree_id0: int = 0, tapes: Optional[Dict[str, np.ndarray]] = None, dump: bool = True, n_threads: int = 1) -> Dict[str, np.ndarray]:
    """B independent searches; the same dict as oracle.azo.search for the discrete variant, with a 2-wide dump state."""
    p = azo._p
    root_state = np.ascontiguousarray(root_state, dtype=np.float64).reshape(-1, 2)
    B, R, A, cm = root_state.shape[0], cfg.rows, cfg.num_actions, cfg.cmax
    out: Dict[str, np.ndarray] = dict(
        n_children=np.zeros(B, np.int32), actions=np.zeros((B, cm), np.float32), counts=np.zeros((B, cm), np.int32),
        Q=np.zeros((B, cm), np.float64), V_target=np.zeros(B, np.float64), counters=np.zeros(8, np.int64))
    res = azo._Res(cm, p(out["n_children"]), p(out["actions"]), p(out["counts"]), p(out["Q"]), p(out["V_target"]), p(out["counters"]))
    dd = None
    if dump:
        d = dict(n_nodes=np.zeros(B, np.int32), parent=np.zeros((B, R), np.int32), paction=np.zeros((B, R), np.int32),
                 node_n=np.zeros((B, R), np.int32), terminal=np.zeros((B, R), np.int32), V=np.zeros((B, R), np.float32),
                 r=np.zeros((B, R), np.float64), state=np.zeros((B, R, 2), np.float64),
                 prior=np.zeros((B, R, A), np.float32), eW=np.zeros((B, R, A), np.float64),
                 en=np.zeros((B, R, A), np.int32), echild=np.zeros((B, R, A), np.int32))
        dd = azo._DumpD(*[p(d[n]) for n, _ in azo._DumpD._fields_])
        out.update(d)
    tp, keep = None, []
    if tapes is not None:
        tv = np.ascontiguousarray(tapes["V"], np.float32)
        tpr = np.ascontiguousarray(tapes["prior"], np.float32)
        keep += [tv, tpr]
        tp = azo._Tapes(p(tv), p(tpr), None)
    w = None if weights is None else np.ascontiguousarray(weights, np.float32)
    rn = None if root_n_init is None else np.ascontiguousarray(root_n_init, np.int32)
    rc = lib().mc_search(C.byref(cfg.c()), p(w), 0 if w is None else w.size, B, p(root_state), p(rn), tree_id0,
                         None if tp is None else C.byref(tp), C.byref(res), None if dd is None else C.byref(dd), n_threads)
    if rc != 0:
        raise ValueError({-2: "bad oracle config", -3: "NaN in UCT"}.get(rc, f"oracle error {rc}"))
    return out


def selfplay_run(cfg: azo.Config, weights: np.ndarray, states0: np.ndarray, steps: int, max_episode_length: int, seed: int = 34,
                 tree_id0: int = 0, deterministic: bool = False, by_value: bool = False, temperature: float = 1.0,
                 n_threads: int = 4) -> List[Dict[str, np.ndarray]]:
    """oracle/selfplay.py's loop for this env: DiscreteAgent.act over three actions (stable_normalizer, pi.argmax() or
    np.random.choice's inverse CDF), the env step, Env.reset at the goal or at max_episode_length, tree reuse of root.n."""
    state = np.array(states0, np.float64).copy()
    B = state.shape[0]
    ep_step, episode, root_n = np.zeros(B, np.int32), np.zeros(B, np.int32), np.zeros(B, np.int32)
    out = []
    for s in range(steps):
        key = osp.step_seed(seed, s)
        c = dataclasses.replace(cfg, seed=key)
        res = search(c, weights, state, root_n.copy(), tree_id0=tree_id0, n_threads=n_threads)
        rec = dict(obs=state.astype(np.float32), actions=res["actions"].copy(), counts=res["counts"].copy(), Q=res["Q"].copy(),
                   V_target=res["V_target"].copy(), n_children=res["n_children"].copy(), action_taken=np.zeros(B, np.float32),
                   reward=np.zeros(B, np.float64), done=np.zeros(B, np.int32))
        for t in range(B):
            x = res["Q"][t, :3] if by_value else res["counts"][t, :3].astype(np.float64)
            pi = osp.stable_normalizer(x, temperature)
            if deterministic:
                a = int(pi.argmax())
            else:
                u = osp._unit(azo.rng_u32(key, tree_id0 + t, 2, 0, 0, 0))
                cdf = np.cumsum(pi)
                cdf /= cdf[-1]
                a = int(np.searchsorted(cdf, u, side="right"))
            nxt, r, term, _ = env_step(c, state[t], a)
            step = int(ep_step[t]) + 1
            done = term or step >= max_episode_length
            rn = 0
            if done:
                episode[t] += 1
                u = osp._unit(azo.rng_u32(key, tree_id0 + t, 3, int(episode[t]), 0, 0))
                nxt = np.array([-0.6 + (-0.4 - -0.6) * u, 0.0])
            else:
                child = int(res["echild"][t, 0, a])
                rn = 0 if child < 0 else int(res["node_n"][t, child])
            ep_step[t] = 0 if done else step
            root_n[t] = rn
            state[t] = nxt
            rec["action_taken"][t], rec["reward"][t], rec["done"][t] = float(a), r, int(done)
        rec.update(env_state=state.copy(), ep_step=ep_step.copy(), episode=episode.copy(), root_n=root_n.copy())
        out.append(rec)
    return out
