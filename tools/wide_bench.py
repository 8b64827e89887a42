"""Searches with a 256-wide trunk (streamed FP32 evaluation, csrc/mlp_stream.cuh) against the same searches with a 128-wide trunk
(k_mlp, csrc/mlp.cuh), measured alternately in one process.

    python tools/wide_bench.py [--out FILE] [--reps 5] [--rounds 3]

Configurations, all FP32 evaluation with one launch per simulation (the schedule every width other than 128 runs):
  Pendulum-v0   65536 trees x 100 simulations, ELU, K = 2, trunks 3 x 128 and 3 x 256;
  CartPole-v0    4096 x 50 and 65536 x 100, ReLU, epsilon 0.1, trunks 2 x 128 and 2 x 256.
For each: sims/s from CUDA events around `reps` searches (best and median of `rounds` alternating rounds, after warm-up); the
evaluation kernel's time from azg_profile_search (a CUDA-event pair around every launch, in a separate search); its achieved TFLOP/s
from shapes (2 x (S H + (L - 1) H^2 + H (1 + P)) per row, every row of every evaluation launch); the weight bytes the kernel reads
from L2; and the first 256 trees' root results against the CPU oracle bit for bit.

Besides the searches, the evaluation alone (azg_mlp_forward, 65536 dense rows, CUDA events around 20 launches) at each trunk and at
the same width with one hidden layer: the difference is the time of the streamed hidden layers, so their FMA rate is separated from
the phases around them (layer 0, heads, post-processing).  The FP32 peak is measured in the same call by tools/fp32_peak.cu (built
into a temporary directory).  Prints the card and its power limit first and writes JSON to --out.
"""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from alphazero_gym_b200._cabi import ACT_ELU, ACT_RELU  # noqa: E402
from alphazero_gym_b200.engine import EngineConfig, SearchEngine, _ptr, check as azg_check  # noqa: E402
from alphazero_gym_b200.network import init_policy_weights  # noqa: E402
from oracle import azo  # noqa: E402

SMS = 148
SMEM_OPTIN = 232448
CONFIGS = [("Pendulum-v0", 65536, 100), ("CartPole-v0", 4096, 50), ("CartPole-v0", 65536, 100)]


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    name, power, clock = (q[0].split(", ") + ["?", "?", "?"])[:3] if q else ("?", "?", "?")
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def fp32_peak() -> dict:
    """tools/fp32_peak.cu: the best packed-FFMA2 rate over its block shapes (TFLOP/s) and every line it printed."""
    nvcc = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")
    with tempfile.TemporaryDirectory() as d:
        exe = os.path.join(d, "fp32_peak")
        subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-o", exe, os.path.join(ROOT, "tools", "fp32_peak.cu")],
                       check=True, capture_output=True)
        out = subprocess.run([exe], check=True, capture_output=True, text=True).stdout
    ffma2 = [float(m) for m in re.findall(r"mode FFMA2.*?: ([0-9.]+) TFLOP/s", out)]
    return {"ffma2_tflops": max(ffma2), "lines": out.strip().splitlines()}


def oracle_config(env: str, H: int, N: int) -> azo.Config:
    if env == "CartPole-v0":
        cfg = azo.discrete_config(n_rollouts=N, hidden=H, n_hidden=2, activation=ACT_RELU, epsilon=0.1)
    else:
        cfg = azo.continuous_config(n_rollouts=N, hidden=H, n_hidden=3, num_components=2, activation=ACT_ELU)
    cfg.math_mode, cfg.eval_mode = azo.MATH_DET, azo.EVAL_FP32
    return cfg


def engine(cfg: azo.Config, B: int, L: int = None) -> SearchEngine:
    ecfg = EngineConfig(variant=cfg.variant, max_rollouts=cfg.n_rollouts, max_trees=B, num_actions=cfg.num_actions,
                        num_components=cfg.num_components, state_dim=cfg.state_dim, hidden=cfg.hidden, n_hidden=L or cfg.n_hidden,
                        activation=cfg.activation, c_uct=cfg.c_uct, c_pw=cfg.c_pw, kappa=cfg.kappa, epsilon=cfg.epsilon,
                        action_bound=cfg.action_bound, eval_q8=False, fused=False)
    assert not ecfg.is_q8() and not ecfg.is_fused()
    return SearchEngine(ecfg)


def flops_per_row(cfg: azo.Config, L: int = None) -> int:
    L, H = L or cfg.n_hidden, cfg.hidden
    return 2 * (cfg.state_dim * H + (L - 1) * H * H + H * (1 + cfg.head_dim))


def streamed_bytes(cfg: azo.Config, n: int, L: int = None) -> int:
    """Weight bytes one evaluation launch over n rows reads from L2: k_mlp stages the whole network once per CTA; k_mlp_stream
    streams the hidden layers once per pass of every CTA (engine.cu azg_create / mlp_stream.cuh) plus layer 0 and the heads once."""
    L, H, S = L or cfg.n_hidden, cfg.hidden, cfg.state_dim
    po = (1 + cfg.head_dim + 3) // 4 * 4
    resident = S * H + H + H * po + po
    if H in (64, 128):
        ctas = min(SMS, ((n + 31) // 32 + 3) // 4)
        return ctas * (resident + (L - 1) * (H * H + H)) * 4
    rb = max(1, 16 // (H // 32))
    while rb > 1 and 4 * (32 * H + resident + H * 64 * rb + po * 64 * rb + S * 64 * rb + 64 * rb) + 8 * 64 * rb + 72 > SMEM_OPTIN:
        rb -= 1
    rp = 64 * rb
    grid = min(SMS, (n + 63) // 64)
    passes = sum(-(-(((b + 1) * n) // grid - (b * n) // grid) // rp) for b in range(grid))
    return (grid * resident + passes * (L - 1) * (H * H + H)) * 4


def roots(env: str, B: int, seed: int = 5) -> np.ndarray:
    rng = np.random.default_rng(seed)
    if env == "Pendulum-v0":
        return np.stack([rng.uniform(-np.pi, np.pi, B), rng.uniform(-1.0, 1.0, B)], 1)
    return rng.uniform(-0.05, 0.05, (B, 4))


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


def time_forward(cfg: azo.Config, L: int, n: int = 65536, reps: int = 20) -> float:
    """ms per azg_mlp_forward over n dense rows (device buffers, CUDA events around `reps` launches after warm-up)."""
    eng = engine(cfg, 1, L)
    try:
        eng.set_weights(init_policy_weights(34, cfg.state_dim, cfg.hidden, L, cfg.head_dim))
        x = torch.from_numpy(np.random.default_rng(1).uniform(-1, 1, (n, cfg.state_dim)).astype(np.float32)).cuda()
        V = torch.empty(n, dtype=torch.float32, device="cuda")
        head = torch.empty((n, eng.head_dim), dtype=torch.float32, device="cuda")

        def launch():
            azg_check(eng._lib.azg_mlp_forward(eng._h, n, _ptr(x), _ptr(V), _ptr(head), eng._stream()))

        for _ in range(3):
            launch()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            launch()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps
    finally:
        eng.close()


def check_oracle(eng, cfg, w, rs, n=256) -> bool:
    got = {k: v.cpu().numpy() for k, v in eng.root_results().items()}
    ref = azo.search(cfg, w, rs[:n], dump=False, n_threads=os.cpu_count() or 8)
    c = ref["counts"].shape[1]
    return bool(np.array_equal(got["counts"][:n, :c], ref["counts"]) and np.array_equal(got["Q"][:n, :c], ref["Q"])
                and np.array_equal(got["actions"][:n, :c], ref["actions"]) and np.array_equal(got["V_target"][:n], ref["V_target"]))


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        print("no CUDA device: this benchmark measures the GPU", file=sys.stderr)
        return 2
    info = card()
    print(f"card: {info['name']}, power limit {info['power_limit']}, max SM clock {info['max_sm_clock']}", flush=True)
    peak = fp32_peak()
    print(f"FP32 peak (tools/fp32_peak.cu, FFMA2): {peak['ffma2_tflops']:.2f} TFLOP/s", flush=True)
    results = []
    for env, B, N in CONFIGS:
        runs = {}
        for H in (128, 256):
            cfg = oracle_config(env, H, N)
            eng = engine(cfg, B)
            w = init_policy_weights(34, cfg.state_dim, H, cfg.n_hidden, cfg.head_dim)
            eng.set_weights(w)
            rs = roots(env, B)
            runs[H] = (eng, cfg, w, rs, torch.from_numpy(rs).cuda())
        ms = {H: [] for H in runs}
        for _ in range(a.rounds):
            for H, (eng, _, _, _, rs_t) in runs.items():
                ms[H].append(time_searches(eng, rs_t, N, a.reps))
        for H, (eng, cfg, w, rs, rs_t) in runs.items():
            prof = eng.profile_search(rs_t, N)
            eng.status()
            ev = prof["evaluation"]
            eng.search(rs_t, N)
            ok = check_oracle(eng, cfg, w, rs)
            fl = flops_per_row(cfg)
            best = min(ms[H])
            rec = {"env": env, "trees": B, "n_rollouts": N, "trunk": f"{cfg.n_hidden} x {H}", "kernel": "k_mlp" if H == 128 else "k_mlp_stream",
                   "ms_per_search": ms[H], "m_sims_per_s_best": B * N / best / 1e3,
                   "m_sims_per_s_median": B * N / float(np.median(ms[H])) / 1e3,
                   "eval_ms_total": ev["ms"], "eval_launches": ev["launches"], "eval_us_per_launch": 1e3 * ev["ms"] / ev["launches"],
                   "flops_per_row": fl, "eval_tflops": ev["launches"] * B * fl / (ev["ms"] * 1e-3) / 1e12,
                   "eval_share_of_fp32_peak": ev["launches"] * B * fl / (ev["ms"] * 1e-3) / 1e12 / peak["ffma2_tflops"],
                   "weight_bytes_per_eval": streamed_bytes(cfg, B), "oracle_first_256_trees_bit_identical": ok}
            results.append(rec)
            print(f"{env:12s} {B:6d} x {N:3d}  {rec['trunk']:8s} {rec['kernel']:12s}  best {rec['m_sims_per_s_best']:7.1f} M sims/s  "
                  f"median {rec['m_sims_per_s_median']:7.1f}  eval {rec['eval_us_per_launch']:7.1f} us/launch  "
                  f"{rec['eval_tflops']:6.2f} TFLOP/s ({100 * rec['eval_share_of_fp32_peak']:.1f} % of peak)  "
                  f"weights {rec['weight_bytes_per_eval'] / 1e6:7.1f} MB/eval  oracle ok {ok}", flush=True)
            eng.close()
    forward = []
    for env in ("Pendulum-v0", "CartPole-v0"):
        for H in (128, 256):
            cfg = oracle_config(env, H, 8)
            n = 65536
            t_full, t_one = time_forward(cfg, cfg.n_hidden, n), time_forward(cfg, 1, n)
            hid_fl = (cfg.n_hidden - 1) * 2 * H * H * n
            rec = {"env": env, "trunk": f"{cfg.n_hidden} x {H}", "rows": n, "ms": t_full, "ms_one_hidden_layer": t_one,
                   "tflops": flops_per_row(cfg) * n / (t_full * 1e-3) / 1e12,
                   "share_of_fp32_peak": flops_per_row(cfg) * n / (t_full * 1e-3) / 1e12 / peak["ffma2_tflops"],
                   "hidden_layers_tflops": hid_fl / ((t_full - t_one) * 1e-3) / 1e12,
                   "hidden_layers_share_of_fp32_peak": hid_fl / ((t_full - t_one) * 1e-3) / 1e12 / peak["ffma2_tflops"],
                   "floor_us_at_peak": flops_per_row(cfg) * n / (peak["ffma2_tflops"] * 1e12) * 1e6,
                   "weight_bytes": streamed_bytes(cfg, n)}
            forward.append(rec)
            print(f"forward {env:12s} {rec['trunk']:8s} {n} rows: {1e3 * t_full:7.1f} us ({100 * rec['share_of_fp32_peak']:.1f} % of peak; "
                  f"floor {rec['floor_us_at_peak']:.0f} us), 1 hidden layer {1e3 * t_one:7.1f} us, hidden layers alone "
                  f"{100 * rec['hidden_layers_share_of_fp32_peak']:.1f} % of peak", flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump({"card": info, "fp32_peak": peak, "searches": results, "evaluation_only": forward}, f, indent=1)
    return 0 if all(r["oracle_first_256_trees_bit_identical"] for r in results) else 1


if __name__ == "__main__":
    sys.exit(main())
