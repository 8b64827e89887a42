"""MountainCarContinuous-v0 against Pendulum-v0 in the whole-search kernels, measured in one process.

    python tools/mountain_car_bench.py [--out FILE] [--reps 10] [--rounds 3]

For each batch -- 65536 trees x 100 simulations (warpgroup kernel) and 4096 x 100 (two-phase kernel) -- both envs run the same
network (ContinuousPolicy.yaml: 3 x 128 ELU, K = 2, tensor-core evaluation), alternately, `rounds` times: warm-up searches, then
`reps` searches between two CUDA events.  Roots: MountainCarContinuous from its reset distribution (position ~ U(-0.6, -0.4),
velocity 0), Pendulum from its own (th ~ U(-pi, pi), thdot ~ U(-1, 1)).  The first 256 trees of every configuration are checked
against the CPU reference bit for bit (oracle/azo for Pendulum, tests/mcc_oracle.py for MountainCarContinuous).  Prints the card and
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
sys.path.insert(0, os.path.join(ROOT, "tests"))

from alphazero_gym_b200._cabi import ACT_ELU, CONTINUOUS  # noqa: E402
from alphazero_gym_b200.engine import MOUNTAIN_CAR_CONTINUOUS, PENDULUM, EngineConfig, SearchEngine  # noqa: E402
from alphazero_gym_b200.network import init_policy_weights  # noqa: E402
from oracle import azo  # noqa: E402
import mcc_oracle  # noqa: E402

N = 100


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    name, power, clock = (q[0].split(", ") + ["?", "?", "?"])[:3] if q else ("?", "?", "?")
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def roots(env: str, B: int, seed: int = 5) -> np.ndarray:
    rng = np.random.default_rng(seed)
    if env == MOUNTAIN_CAR_CONTINUOUS:
        return np.stack([rng.uniform(-0.6, -0.4, B), np.zeros(B)], 1)
    return np.stack([rng.uniform(-np.pi, np.pi, B), rng.uniform(-1.0, 1.0, B)], 1)


def setup(env: str, B: int):
    S = 2 if env == MOUNTAIN_CAR_CONTINUOUS else 3
    bound = 1.0 if env == MOUNTAIN_CAR_CONTINUOUS else 2.0
    ecfg = EngineConfig(variant=CONTINUOUS, max_rollouts=N, max_trees=B, num_components=2, state_dim=S, hidden=128, n_hidden=3,
                        activation=ACT_ELU, c_uct=0.05, c_pw=1.0, kappa=0.5, epsilon=0.0, action_bound=bound, env=env)
    assert ecfg.is_fused() and ecfg.is_q8()
    make = mcc_oracle.config if env == MOUNTAIN_CAR_CONTINUOUS else azo.continuous_config
    ocfg = make(n_rollouts=N, num_components=2, n_hidden=3, activation=ACT_ELU)
    ocfg.math_mode, ocfg.eval_mode = azo.MATH_DET, azo.EVAL_Q8
    w = init_policy_weights(34, S, 128, 3, 6)
    eng = SearchEngine(ecfg)
    eng.set_weights(w)
    rs = roots(env, B)
    return eng, (ocfg, env), w, rs, torch.from_numpy(rs).cuda()


def check(eng, oc, w, rs, n=256) -> bool:
    ocfg, env = oc
    got = {k: v.cpu().numpy() for k, v in eng.root_results().items()}
    if env == MOUNTAIN_CAR_CONTINUOUS:
        ref = mcc_oracle.search(ocfg, w, rs[:n], dump=False, n_threads=8)
    else:
        ref = azo.search(ocfg, w, rs[:n], dump=False, n_threads=8)
    c = ref["counts"].shape[1]
    return bool(np.array_equal(got["counts"][:n, :c], ref["counts"]) and np.array_equal(got["Q"][:n, :c], ref["Q"])
                and np.array_equal(got["actions"][:n, :c], ref["actions"]) and np.array_equal(got["V_target"][:n], ref["V_target"]))


def time_searches(eng, rs_t, reps: int, warmup: int = 2) -> float:
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
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    info = card()
    print(f"card: {info['name']}, power limit {info['power_limit']}, max SM clock {info['max_sm_clock']}")
    results = []
    for B in (65536, 4096):
        runs = {env: setup(env, B) for env in (MOUNTAIN_CAR_CONTINUOUS, PENDULUM)}
        ms = {env: [] for env in runs}
        for _ in range(a.rounds):
            for env, (eng, _, _, _, rs_t) in runs.items():
                ms[env].append(time_searches(eng, rs_t, a.reps))
        for env, (eng, ocfg, w, rs, rs_t) in runs.items():
            kernel = eng.fused_stats()["kernel"]
            eng.search(rs_t, N)
            ok = check(eng, ocfg, w, rs)
            best = min(ms[env])
            rec = {"env": env, "trees": B, "n_rollouts": N, "kernel": kernel, "ms_per_search": ms[env],
                   "m_sims_per_s_best": B * N / best / 1e3, "m_sims_per_s_median": B * N / float(np.median(ms[env])) / 1e3,
                   "oracle_first_256_trees_bit_identical": ok}
            results.append(rec)
            print(f"{env:26s} {B:6d} x {N}  {kernel:10s}  ms/search {' '.join(f'{x:.3f}' for x in ms[env])}  "
                  f"best {rec['m_sims_per_s_best']:.0f} M sims/s  median {rec['m_sims_per_s_median']:.0f} M sims/s  oracle ok {ok}")
            eng.close()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump({"card": info, "results": results}, f, indent=1)
    return 0 if all(r["oracle_first_256_trees_bit_identical"] for r in results) else 1


if __name__ == "__main__":
    sys.exit(main())
