"""Two envs of one search variant against each other in the whole-search kernels, measured in one process.

    python tools/env_bench.py ENV_A ENV_B [--out FILE] [--reps 10] [--rounds 3]

for instance `MountainCarContinuous-v0 Pendulum-v0`, `MountainCar-v0 CartPole-v0` or `Acrobot-v1 MountainCar-v0`.

Both envs run the same trunk with tensor-core evaluation and the whole search in one kernel launch, alternately, `rounds` times:
warm-up searches, then `reps` searches between two CUDA events.  The variant's network and sizes:
  discrete   (DiscretePolicy.yaml: 2 x 128 ReLU): 4096 trees x 50 simulations and 65536 x 100 (BASELINE configs 3 and 4 for CartPole).
             At 4096 trees CartPole runs its shared-memory trees and the three-action envs the two-phase kernel (three-action rows are
             not held in shared memory); at 65536 all run the warpgroup kernel.
  continuous (ContinuousPolicy.yaml: 3 x 128 ELU, K = 2): 65536 x 100 (warpgroup kernel) and 4096 x 100 (two-phase kernel).
Each env's network input is its own observation (CartPole 4, Pendulum 3, MountainCar(Continuous) 2, Acrobot 6); roots come from its
reset distribution.  The first 256 trees of every configuration are checked against the CPU oracle bit for bit.  Prints the card and
its power limit, one line per configuration, and writes JSON to --out.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from alphazero_gym_b200._cabi import ACT_ELU, ACT_RELU, DISCRETE  # noqa: E402
from alphazero_gym_b200.engine import ACROBOT, CARTPOLE, MOUNTAIN_CAR, MOUNTAIN_CAR_CONTINUOUS, PENDULUM  # noqa: E402
from alphazero_gym_b200.engine import EngineConfig, SearchEngine  # noqa: E402
from alphazero_gym_b200.network import init_policy_weights  # noqa: E402
from oracle import azo  # noqa: E402

VARIANT = {CARTPOLE: azo.DISCRETE, MOUNTAIN_CAR: azo.DISCRETE, ACROBOT: azo.DISCRETE,
           PENDULUM: azo.CONTINUOUS, MOUNTAIN_CAR_CONTINUOUS: azo.CONTINUOUS}
SIZES = {azo.DISCRETE: ((4096, 50), (65536, 100)), azo.CONTINUOUS: ((65536, 100), (4096, 100))}


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    name, power, clock = (q[0].split(", ") + ["?", "?", "?"])[:3] if q else ("?", "?", "?")
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def roots(env: str, B: int, seed: int = 5) -> np.ndarray:
    rng = np.random.default_rng(seed)
    if env in (MOUNTAIN_CAR, MOUNTAIN_CAR_CONTINUOUS):
        return np.stack([rng.uniform(-0.6, -0.4, B), np.zeros(B)], 1)
    if env == PENDULUM:
        return np.stack([rng.uniform(-np.pi, np.pi, B), rng.uniform(-1.0, 1.0, B)], 1)
    return rng.uniform(-0.05, 0.05, (B, 4)) if env == CARTPOLE else rng.uniform(-0.1, 0.1, (B, 4))


def oracle_config(env: str, N: int) -> azo.Config:
    oenv = None if env in (CARTPOLE, PENDULUM) else env
    if VARIANT[env] == azo.DISCRETE:
        ocfg = azo.discrete_config(oenv, n_rollouts=N, n_hidden=2, activation=ACT_RELU, epsilon=0.1)
    else:
        ocfg = azo.continuous_config(oenv, n_rollouts=N, num_components=2, n_hidden=3, activation=ACT_ELU)
    ocfg.math_mode, ocfg.eval_mode = azo.MATH_DET, azo.EVAL_Q8
    return ocfg


def setup(env: str, B: int, N: int):
    ocfg = oracle_config(env, N)
    ecfg = EngineConfig(variant=ocfg.variant, max_rollouts=N, max_trees=B, num_actions=ocfg.num_actions,
                        num_components=ocfg.num_components, state_dim=ocfg.state_dim, hidden=128, n_hidden=ocfg.n_hidden,
                        activation=ocfg.activation, c_uct=ocfg.c_uct, c_pw=ocfg.c_pw, kappa=ocfg.kappa, epsilon=ocfg.epsilon,
                        action_bound=ocfg.action_bound, env=env)
    assert ecfg.is_fused() and ecfg.is_q8()
    w = init_policy_weights(34, ocfg.state_dim, 128, ocfg.n_hidden, ocfg.head_dim)
    eng = SearchEngine(ecfg)
    eng.set_weights(w)
    rs = roots(env, B)
    return eng, ocfg, w, rs, torch.from_numpy(rs).cuda()


def check(eng, ocfg, w, rs, n=256) -> bool:
    got = {k: v.cpu().numpy() for k, v in eng.root_results().items()}
    ref = azo.search(ocfg, w, rs[:n], dump=False, n_threads=8)
    c = ref["counts"].shape[1]
    return bool(np.array_equal(got["counts"][:n, :c], ref["counts"]) and np.array_equal(got["Q"][:n, :c], ref["Q"])
                and np.array_equal(got["actions"][:n, :c], ref["actions"]) and np.array_equal(got["V_target"][:n], ref["V_target"]))


def time_searches(eng, rs_t, N: int, reps: int, warmup: int = 2) -> float:
    for _ in range(warmup):
        eng.search(rs_t, N)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        eng.search(rs_t, N)
    b.record()
    torch.cuda.synchronize()
    eng.status()
    return a.elapsed_time(b) / reps


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("envs", nargs=2, choices=sorted(VARIANT))
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    if VARIANT[a.envs[0]] != VARIANT[a.envs[1]]:
        ap.error(f"{a.envs[0]} and {a.envs[1]} run different search variants")
    info = card()
    print(f"card: {info['name']}, power limit {info['power_limit']}, max SM clock {info['max_sm_clock']}")
    results = []
    for B, N in SIZES[VARIANT[a.envs[0]]]:
        runs = {env: setup(env, B, N) for env in a.envs}
        ms = {env: [] for env in runs}
        for _ in range(a.rounds):
            for env, (eng, _, _, _, rs_t) in runs.items():
                ms[env].append(time_searches(eng, rs_t, N, a.reps))
        for env, (eng, ocfg, w, rs, rs_t) in runs.items():
            kernel = eng.fused_stats()["kernel"]
            eng.search(rs_t, N)
            ok = check(eng, ocfg, w, rs)
            best = min(ms[env])
            rec = {"env": env, "trees": B, "n_rollouts": N, "kernel": kernel, "ms_per_search": ms[env],
                   "m_sims_per_s_best": B * N / best / 1e3, "m_sims_per_s_median": B * N / float(np.median(ms[env])) / 1e3,
                   "oracle_first_256_trees_bit_identical": ok}
            results.append(rec)
            print(f"{env:26s} {B:6d} x {N:3d}  {kernel:34s}  ms/search {' '.join(f'{x:.3f}' for x in ms[env])}  "
                  f"best {rec['m_sims_per_s_best']:.0f} M sims/s  median {rec['m_sims_per_s_median']:.0f} M sims/s  oracle ok {ok}")
            eng.close()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump({"card": info, "results": results}, f, indent=1)
    return 0 if all(r["oracle_first_256_trees_bit_identical"] for r in results) else 1


if __name__ == "__main__":
    sys.exit(main())
