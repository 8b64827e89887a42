"""CPU restatement of the reference's self-play episode loop for a batch of independent environments -- test
infrastructure (the checker of azg_selfplay_step), never a product path.

Follows, per environment and step: run_continuous.py:117-142 / run_discrete.py:100-122 (act -> store -> Env.step ->
reset or reset_mcts / mcts_forward), ContinuousAgent.act (agents.py:522-537: actions[counts.argmax()]), DiscreteAgent.act
(agents.py:292-303: stable_normalizer + pi.argmax() / np.random.choice), helpers.stable_normalizer (helpers.py:9-27),
MCTSDiscrete.forward (mcts.py:495-526; only the new root's visit count survives, SURVEY 7-7).  The searches are
oracle/azo.search.  Randomness is injected exactly as in the engine: the Philox key of step s is
seed + s * 0x9E3779B97F4A7C15 (mod 2^64); stream 2 = the discrete agent's action draw, stream 3 = Env.reset (RESETS);
a 32-bit word x maps to (x + 0.5) / 2^32.
"""
from __future__ import annotations

import dataclasses
from typing import Dict, List

import numpy as np

from . import azo

GOLDEN = 0x9E3779B97F4A7C15
MASK = (1 << 64) - 1


def step_seed(seed: int, step: int) -> int:
    return (seed + step * GOLDEN) & MASK


def _unit(x: int) -> float:
    return (float(x) + 0.5) * 2.3283064365386963e-10


def _uniform(lo: float, hi: float, w: int) -> float:
    return lo + (hi - lo) * _unit(w)


# gym's Env.reset per env, from the four words of stream 3 at the episode's index
RESETS = {
    (azo.DISCRETE, None): lambda w: [_uniform(-0.05, 0.05, w[k]) for k in range(4)],            # CartPole U(-0.05, 0.05)^4
    (azo.CONTINUOUS, None): lambda w: [_uniform(-np.pi, np.pi, w[0]), _uniform(-1.0, 1.0, w[1])],  # Pendulum th, thdot
    (azo.CONTINUOUS, azo.MOUNTAIN_CAR_CONTINUOUS): lambda w: [_uniform(-0.6, -0.4, w[0]), 0.0],  # position, velocity 0
    (azo.DISCRETE, azo.MOUNTAIN_CAR): lambda w: [_uniform(-0.6, -0.4, w[0]), 0.0],
    (azo.DISCRETE, azo.ACROBOT): lambda w: [_uniform(-0.1, 0.1, w[k]) for k in range(4)],       # U(-0.1, 0.1)^4
}


def stable_normalizer(x: np.ndarray, temp: float) -> np.ndarray:
    x = (x / np.max(x)) ** temp  # helpers.py:26
    return np.abs(x / np.sum(x))


def run(cfg: azo.Config, weights: np.ndarray, states0: np.ndarray, steps: int, max_episode_length: int, seed: int = 34,
        tree_id0: int = 0, deterministic: bool = False, by_value: bool = False, temperature: float = 1.0,
        n_threads: int = 4) -> List[Dict[str, np.ndarray]]:
    """Returns, per step, the arrays azg_selfplay_step writes (obs, actions, counts, Q, V_target, n_children,
    action_taken, reward, done) plus the carried state after the step (env_state, ep_step, episode, root_n)."""
    disc = cfg.variant == azo.DISCRETE
    state = np.array(states0, np.float64).copy()
    B = state.shape[0]
    ep_step, episode, root_n = np.zeros(B, np.int32), np.zeros(B, np.int32), np.zeros(B, np.int32)
    out = []
    for s in range(steps):
        key = step_seed(seed, s)
        c = dataclasses.replace(cfg, seed=key)
        res = azo.search(c, weights, state, root_n.copy() if disc else None, tree_id0=tree_id0, dump=disc, n_threads=n_threads)
        rec = dict(obs=azo.obs(c, state), actions=res["actions"].copy(),
                   counts=res["counts"].copy(), Q=res["Q"].copy(), V_target=res["V_target"].copy(),
                   n_children=res["n_children"].copy(), action_taken=np.zeros(B, np.float32), reward=np.zeros(B, np.float64),
                   done=np.zeros(B, np.int32))
        for t in range(B):
            nk = int(res["n_children"][t])
            if disc:
                x = (res["Q"][t, :cfg.num_actions] if by_value else res["counts"][t, :cfg.num_actions].astype(np.float64))
                pi = stable_normalizer(x, temperature)
                if deterministic:
                    a = int(pi.argmax())
                else:
                    u = _unit(azo.rng_u32(key, tree_id0 + t, 2, 0, 0, 0))
                    cdf = np.cumsum(pi)
                    cdf /= cdf[-1]
                    a = int(np.searchsorted(cdf, u, side="right"))
                action = float(a)
            else:
                vals = res["Q"][t, :nk] if by_value else res["counts"][t, :nk]
                a = int(np.argmax(vals))
                action = float(res["actions"][t, a])
            nxt, r, term, _ = azo.env_step(c, state[t], action)
            step = int(ep_step[t]) + 1
            done = term or step >= max_episode_length
            rn = 0
            if done:
                episode[t] += 1
                w = [azo.rng_u32(key, tree_id0 + t, 3, int(episode[t]), 0, k) for k in range(4)]
                nxt = np.array(RESETS[cfg.variant, cfg.env](w))
            elif disc:
                child = int(res["echild"][t, 0, a])
                rn = 0 if child < 0 else int(res["node_n"][t, child])
            ep_step[t] = 0 if done else step
            root_n[t] = rn
            state[t] = nxt
            rec["action_taken"][t], rec["reward"][t], rec["done"][t] = action, r, int(done)
        rec.update(env_state=state.copy(), ep_step=ep_step.copy(), episode=episode.copy(), root_n=root_n.copy())
        out.append(rec)
    return out
