"""Acrobot-v1 against MountainCar-v0 in the three-action discrete search, measured in one process.

    python tools/acrobot_bench.py [--out FILE] [--reps 10] [--rounds 3]

Two configurations: 4096 trees x 50 simulations (the two-phase kernel: three-action rows are not held in shared memory) and 65536 x 100
(the warpgroup kernel).  Both envs run the same trunk (DiscretePolicy.yaml: 2 x 128 ReLU, tensor-core evaluation, the whole search in
one kernel launch; Acrobot's layer 0 reads 6 inputs, MountainCar's 2), alternately, `rounds` times: warm-up searches, then `reps`
searches between two CUDA events.  The two differ in the env step (Acrobot: an RK4 step of four derivative evaluations; MountainCar:
one cosine) and the leaf input.  Roots from each env's reset distribution (Acrobot U(-0.1, 0.1)^4; MountainCar position
~ U(-0.6, -0.4), velocity 0).  The first 256 trees of every configuration are checked against the CPU reference bit for bit
(tests/acrobot_oracle.py, tests/mc_oracle.py).  Prints the card and its power limit, one line per configuration, and writes JSON to
--out.
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

from alphazero_gym_b200._cabi import ACT_RELU, DISCRETE  # noqa: E402
from alphazero_gym_b200.engine import ACROBOT, MOUNTAIN_CAR, EngineConfig, SearchEngine  # noqa: E402
from alphazero_gym_b200.network import init_policy_weights  # noqa: E402
from oracle import azo  # noqa: E402
import acrobot_oracle  # noqa: E402
import mc_oracle  # noqa: E402


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    name, power, clock = (q[0].split(", ") + ["?", "?", "?"])[:3] if q else ("?", "?", "?")
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def roots(env: str, B: int, seed: int = 5) -> np.ndarray:
    rng = np.random.default_rng(seed)
    if env == MOUNTAIN_CAR:
        return np.stack([rng.uniform(-0.6, -0.4, B), np.zeros(B)], 1)
    return rng.uniform(-0.1, 0.1, (B, 4))


def setup(env: str, B: int, N: int):
    S, A = (2, 3) if env == MOUNTAIN_CAR else (6, 3)
    ecfg = EngineConfig(variant=DISCRETE, max_rollouts=N, max_trees=B, num_actions=A, state_dim=S, hidden=128, n_hidden=2,
                        activation=ACT_RELU, c_uct=1.5, epsilon=0.1, env=env)
    assert ecfg.is_fused() and ecfg.is_q8()
    make = mc_oracle.config if env == MOUNTAIN_CAR else acrobot_oracle.config
    ocfg = make(n_rollouts=N, n_hidden=2, activation=ACT_RELU, epsilon=0.1)
    ocfg.math_mode, ocfg.eval_mode = azo.MATH_DET, azo.EVAL_Q8
    w = init_policy_weights(34, S, 128, 2, A)
    eng = SearchEngine(ecfg)
    eng.set_weights(w)
    rs = roots(env, B)
    return eng, (ocfg, env), w, rs, torch.from_numpy(rs).cuda()


def check(eng, oc, w, rs, n=256) -> bool:
    ocfg, env = oc
    got = {k: v.cpu().numpy() for k, v in eng.root_results().items()}
    search = mc_oracle.search if env == MOUNTAIN_CAR else acrobot_oracle.search
    ref = search(ocfg, w, rs[:n], dump=False, n_threads=8)
    return bool(np.array_equal(got["counts"][:n], ref["counts"]) and np.array_equal(got["Q"][:n], ref["Q"])
                and np.array_equal(got["V_target"][:n], ref["V_target"]))


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
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    info = card()
    print(f"card: {info['name']}, power limit {info['power_limit']}, max SM clock {info['max_sm_clock']}")
    results = []
    for B, N in ((4096, 50), (65536, 100)):
        runs = {env: setup(env, B, N) for env in (ACROBOT, MOUNTAIN_CAR)}
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
            print(f"{env:16s} {B:6d} x {N:3d}  {kernel:34s}  ms/search {' '.join(f'{x:.3f}' for x in ms[env])}  "
                  f"best {rec['m_sims_per_s_best']:.0f} M sims/s  median {rec['m_sims_per_s_median']:.0f} M sims/s  oracle ok {ok}")
            eng.close()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump({"card": info, "results": results}, f, indent=1)
    return 0 if all(r["oracle_first_256_trees_bit_identical"] for r in results) else 1


if __name__ == "__main__":
    sys.exit(main())
