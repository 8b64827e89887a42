"""CPU reference of the Acrobot-v1 search (test infrastructure; the checker of AZG_FLAG_ENV_ACROBOT).

* `AcrobotEnv`: gym 0.17-0.19 classic_control/acrobot.py, step() with `rk4`, `wrap` and `bound` as gym writes them, in plain Python
  with injectable `sin` / `cos` (the engine's bit-exact twins are the deterministic ones: sin=det_sin, cos=det_cos).  Two departures,
  both the engine's: the square of a float is x * x (gym's x ** 2 calls pow, which is not always correctly rounded), and wrap stops
  after WRAP_CAP iterations per loop.
* `search` / `env_step` / `observe`: tests/acrobot_oracle.c -- the CPU oracle (oracle/azg_oracle.c, included unchanged) with this env
  in its discrete search; same configs (oracle.azo.Config), same output dicts as oracle.azo.search (the dump's state is the 4-wide
  hidden state).
* `selfplay_run`: oracle/selfplay.py's episode loop for this env (Env.reset: the state ~ U(-0.1, 0.1)^4 from Philox stream 3) and
  three actions.

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
_SRC = os.path.join(_HERE, "acrobot_oracle.c")
CFLAGS = ["-O2", "-ftree-vectorize", "-mavx2", "-mfma", "-ffp-contract=off", "-fno-math-errno", "-pthread", "-fPIC", "-std=gnu11"]
WRAP_CAP = 64  # iterations per wrap loop (ACROBOT_WRAP_CAP in csrc/env.cuh, AC_WRAP_CAP in acrobot_oracle.c)
_lib = None


class WrapCapReached(Exception):
    """wrap() would loop on past WRAP_CAP iterations (gym itself loops on)."""


def wrap(x, m, M):
    """gym's wrap, with the engine's iteration cap."""
    diff = M - m
    k = 0
    while x > M:
        if k == WRAP_CAP:
            raise WrapCapReached(x)
        x = x - diff
        k += 1
    k = 0
    while x < m:
        if k == WRAP_CAP:
            raise WrapCapReached(x)
        x = x + diff
        k += 1
    return x


def bound(x, m, M=None):
    if M is None:
        M = m[1]
        m = m[0]
    return min(max(x, m), M)


def rk4(derivs, y0, t, *args, **kwargs):
    try:
        Ny = len(y0)
    except TypeError:
        yout = np.zeros((len(t),), np.float64)
    else:
        yout = np.zeros((len(t), Ny), np.float64)
    yout[0] = y0
    for i in np.arange(len(t) - 1):
        thist = t[i]
        dt = t[i + 1] - thist
        dt2 = dt / 2.0
        y0 = yout[i]
        k1 = np.asarray(derivs(y0, thist, *args, **kwargs))
        k2 = np.asarray(derivs(y0 + dt2 * k1, thist + dt2, *args, **kwargs))
        k3 = np.asarray(derivs(y0 + dt2 * k2, thist + dt2, *args, **kwargs))
        k4 = np.asarray(derivs(y0 + dt * k3, thist + dt, *args, **kwargs))
        yout[i + 1] = y0 + dt / 6.0 * (k1 + 2 * k2 + 2 * k3 + k4)
    return yout


class AcrobotEnv:  # gym's class name, which the drop-in search classes recognise
    """gym 0.17-0.19 classic_control/acrobot.py (book dynamics, no torque noise).  `sin` / `cos` default to math's (glibc)."""
    dt = .2
    LINK_LENGTH_1 = 1.
    LINK_LENGTH_2 = 1.
    LINK_MASS_1 = 1.
    LINK_MASS_2 = 1.
    LINK_COM_POS_1 = 0.5
    LINK_COM_POS_2 = 0.5
    LINK_MOI = 1.
    MAX_VEL_1 = 4 * np.pi
    MAX_VEL_2 = 9 * np.pi
    AVAIL_TORQUE = [-1., 0., +1]
    torque_noise_max = 0.
    book_or_nips = "book"

    def __init__(self, state=(0.0, 0.0, 0.0, 0.0), sin=math.sin, cos=math.cos):
        self.state = np.array(state, dtype=np.float64)
        self.sin, self.cos = sin, cos

    @property
    def unwrapped(self):
        return self

    def step(self, a):
        s = self.state
        torque = self.AVAIL_TORQUE[a]
        s_augmented = np.append(s, torque)
        ns = rk4(self._dsdt, s_augmented, [0, self.dt])
        ns = ns[-1]
        ns = ns[:4]
        ns[0] = wrap(ns[0], -np.pi, np.pi)
        ns[1] = wrap(ns[1], -np.pi, np.pi)
        ns[2] = bound(ns[2], -self.MAX_VEL_1, self.MAX_VEL_1)
        ns[3] = bound(ns[3], -self.MAX_VEL_2, self.MAX_VEL_2)
        self.state = ns
        terminal = self._terminal()
        reward = -1. if not terminal else 0.
        return (self._get_ob(), reward, terminal, {})

    def _get_ob(self):
        s = self.state
        return np.array([self.cos(s[0]), self.sin(s[0]), self.cos(s[1]), self.sin(s[1]), s[2], s[3]])

    def _terminal(self):
        s = self.state
        return bool(-self.cos(s[0]) - self.cos(s[1] + s[0]) > 1.)

    def _dsdt(self, s_augmented, t):
        sin, cos, pi = self.sin, self.cos, np.pi
        m1 = self.LINK_MASS_1
        m2 = self.LINK_MASS_2
        l1 = self.LINK_LENGTH_1
        lc1 = self.LINK_COM_POS_1
        lc2 = self.LINK_COM_POS_2
        I1 = self.LINK_MOI
        I2 = self.LINK_MOI
        g = 9.8
        a = s_augmented[-1]
        s = s_augmented[:-1]
        theta1 = s[0]
        theta2 = s[1]
        dtheta1 = s[2]
        dtheta2 = s[3]
        d1 = m1 * lc1 ** 2 + m2 * \
            (l1 ** 2 + lc2 ** 2 + 2 * l1 * lc2 * cos(theta2)) + I1 + I2
        d2 = m2 * (lc2 ** 2 + l1 * lc2 * cos(theta2)) + I2
        phi2 = m2 * lc2 * g * cos(theta1 + theta2 - pi / 2.)
        # gym writes dtheta2 ** 2, dtheta1 ** 2 and d2 ** 2: the engine's convention (DESIGN.md section 6) is the correctly rounded square
        phi1 = - m2 * l1 * lc2 * (dtheta2 * dtheta2) * sin(theta2) \
               - 2 * m2 * l1 * lc2 * dtheta2 * dtheta1 * sin(theta2)  \
            + (m1 * lc1 + m2 * l1) * g * cos(theta1 - pi / 2) + phi2
        # the "book" branch
        ddtheta2 = (a + d2 / d1 * phi1 - m2 * l1 * lc2 * (dtheta1 * dtheta1) * sin(theta2) - phi2) \
            / (m2 * lc2 ** 2 + I2 - (d2 * d2) / d1)
        ddtheta1 = -(d2 * ddtheta2 + phi1) / d1
        return (dtheta1, dtheta2, ddtheta1, ddtheta2, 0.)


def det_cos(x: float) -> float:
    return float(azo.det_eval("cos", np.array([float(x)]), n_threads=1)[0])


def det_sin(x: float) -> float:
    return float(azo.det_eval("sin", np.array([float(x)]), n_threads=1)[0])


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha256()
        for p in (_SRC, os.path.join(_ORACLE, "azg_oracle.c"), os.path.join(_ORACLE, "azg_oracle.h")):
            h.update(open(p, "rb").read())
        out = os.path.join(tempfile.gettempdir(), f"libacrobot_oracle_{os.getuid()}_{h.hexdigest()[:16]}.so")
        if not os.path.exists(out):
            tmp = f"{out}.{os.getpid()}"
            subprocess.check_call(["gcc"] + CFLAGS + ["-shared", "-I", _ORACLE, "-o", tmp, _SRC, "-lm"])
            os.replace(tmp, out)
        L = C.CDLL(out)
        L.ac_search.restype = C.c_int
        L.ac_search.argtypes = [C.POINTER(azo._Cfg), C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64,
                                C.POINTER(azo._Tapes), C.POINTER(azo._Res), C.POINTER(azo._DumpD), C.c_int32]
        L.ac_env_step.restype = C.c_int
        L.ac_env_step.argtypes = [C.POINTER(azo._Cfg), C.c_void_p, C.c_int32, C.c_void_p, C.POINTER(C.c_double), C.c_void_p]
        L.ac_observe.restype = None
        L.ac_observe.argtypes = [C.POINTER(azo._Cfg), C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


def config(**kw) -> azo.Config:
    """DiscretePolicy.yaml / MCTSDiscrete.yaml defaults with the env's observation (6 entries) and 3 actions."""
    d = dict(state_dim=6, num_actions=3)
    d.update(kw)
    return azo.discrete_config(**d)


def env_step(cfg: azo.Config, state: np.ndarray, action: int):
    """(next hidden state, reward, done, f32 observation); raises WrapCapReached where the engine fails with AZG_EWRAP."""
    s = np.ascontiguousarray(state, np.float64)
    o = np.zeros(4, np.float64)
    obs = np.zeros(6, np.float32)
    r = C.c_double()
    term = lib().ac_env_step(C.byref(cfg.c()), s.ctypes.data_as(C.c_void_p), int(action), o.ctypes.data_as(C.c_void_p), C.byref(r),
                             obs.ctypes.data_as(C.c_void_p))
    if term == -4:
        raise WrapCapReached(state)
    return o, r.value, bool(term), obs


def observe(cfg: azo.Config, state: np.ndarray) -> np.ndarray:
    """The network input of hidden states [n, 4]: _get_ob rounded to f32 per entry, [n, 6]."""
    s = np.ascontiguousarray(state, np.float64).reshape(-1, 4)
    out = np.zeros((s.shape[0], 6), np.float32)
    for i in range(s.shape[0]):
        lib().ac_observe(C.byref(cfg.c()), s[i].ctypes.data_as(C.c_void_p), out[i].ctypes.data_as(C.c_void_p))
    return out


def search(cfg: azo.Config, weights: Optional[np.ndarray], root_state: np.ndarray, root_n_init: Optional[np.ndarray] = None,
           tree_id0: int = 0, tapes: Optional[Dict[str, np.ndarray]] = None, dump: bool = True, n_threads: int = 1) -> Dict[str, np.ndarray]:
    """B independent searches from hidden states; the same dict as oracle.azo.search for the discrete variant."""
    p = azo._p
    root_state = np.ascontiguousarray(root_state, dtype=np.float64).reshape(-1, 4)
    B, R, A, cm = root_state.shape[0], cfg.rows, cfg.num_actions, cfg.cmax
    out: Dict[str, np.ndarray] = dict(
        n_children=np.zeros(B, np.int32), actions=np.zeros((B, cm), np.float32), counts=np.zeros((B, cm), np.int32),
        Q=np.zeros((B, cm), np.float64), V_target=np.zeros(B, np.float64), counters=np.zeros(8, np.int64))
    res = azo._Res(cm, p(out["n_children"]), p(out["actions"]), p(out["counts"]), p(out["Q"]), p(out["V_target"]), p(out["counters"]))
    dd = None
    if dump:
        d = dict(n_nodes=np.zeros(B, np.int32), parent=np.zeros((B, R), np.int32), paction=np.zeros((B, R), np.int32),
                 node_n=np.zeros((B, R), np.int32), terminal=np.zeros((B, R), np.int32), V=np.zeros((B, R), np.float32),
                 r=np.zeros((B, R), np.float64), state=np.zeros((B, R, 4), np.float64),
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
    rc = lib().ac_search(C.byref(cfg.c()), p(w), 0 if w is None else w.size, B, p(root_state), p(rn), tree_id0,
                         None if tp is None else C.byref(tp), C.byref(res), None if dd is None else C.byref(dd), n_threads)
    if rc == -4:
        raise WrapCapReached("an angle reached the wrap cap")
    if rc != 0:
        raise ValueError({-2: "bad oracle config", -3: "NaN in UCT"}.get(rc, f"oracle error {rc}"))
    return out


def selfplay_run(cfg: azo.Config, weights: np.ndarray, states0: np.ndarray, steps: int, max_episode_length: int, seed: int = 34,
                 tree_id0: int = 0, deterministic: bool = False, by_value: bool = False, temperature: float = 1.0,
                 n_threads: int = 4) -> List[Dict[str, np.ndarray]]:
    """oracle/selfplay.py's loop for this env: DiscreteAgent.act over three actions (stable_normalizer, pi.argmax() or
    np.random.choice's inverse CDF), the env step, Env.reset at the goal or at max_episode_length, tree reuse of root.n.  The obs
    row is the 6-wide observation of the state each search started from."""
    state = np.array(states0, np.float64).copy()
    B = state.shape[0]
    ep_step, episode, root_n = np.zeros(B, np.int32), np.zeros(B, np.int32), np.zeros(B, np.int32)
    out = []
    for s in range(steps):
        key = osp.step_seed(seed, s)
        c = dataclasses.replace(cfg, seed=key)
        res = search(c, weights, state, root_n.copy(), tree_id0=tree_id0, n_threads=n_threads)
        rec = dict(obs=observe(c, state), actions=res["actions"].copy(), counts=res["counts"].copy(), Q=res["Q"].copy(),
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
                w = [azo.rng_u32(key, tree_id0 + t, 3, int(episode[t]), 0, k) for k in range(4)]
                nxt = np.array([-0.1 + (0.1 - -0.1) * osp._unit(w[k]) for k in range(4)])
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
