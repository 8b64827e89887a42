#!/usr/bin/env python
"""bench.py -- MCTS simulations/sec of the batched search hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
           bench.py --gpus N --steps K --warmup W

A "step" is one full batched search over one batch of synthetic roots: root evaluation, n_rollouts
simulations (backup + select + env step + leaf evaluation) and root-result extraction.
Headline workload (BASELINE.json configs[3], SURVEY 8d config 4): 65536 Pendulum-v0 trees per GPU x 100
simulations, progressive widening, GMM K=2 policy, MLP 3-128-128-128 ELU, default-initialised weights
(torch.manual_seed(34)), roots from numpy default_rng(34).  Trees are independent, so N GPUs run N shards
with no data-path collective (weak scaling: 65536 trees per GPU).

One JSON line on stdout.  Top level = the headline workload:
  value      whole-job sims/s, roots already resident in HBM, results left on the device (CUDA events)
  e2e        the same through the host-buffer C-ABI calls: pinned H2D of the roots and D2H of
             (actions, counts, Q, V_target, n_children) inside the timed region
  roofline   for the dominant kernel, times taken live with CUDA events; `traffic` measured in this run (ncu, 2 metrics)
  cpu_baseline  the CPU oracle (a C port of the reference search) on a bounded sample of the same workload
  parity     every rank checks a sample of its own trees against the CPU oracle, bit for bit
Without --workload the line also carries
  workloads  {cartpole_4096x50 (configs[2]), selfplay_pendulum_32768x200 (configs[4])}: the same record for each
  strong     (N > 1) the headline workload with the 65536 trees SPLIT over the N GPUs (BASELINE config 4 as worded)
`--dump-outputs DIR` writes what the last timed step of the headline workload returned (rank 0's trees) as DIR/<name>.npy, so
that two builds can be compared output for output: the root results (actions, counts, Q, V_target, n_children), or for a
self-play workload the tensors of SelfPlayDriver.step.
`--impl reference` times the CPU port alone (the reference itself is Python + gym and cannot travel to the
GPU box; its single-core numbers measured in the build container are in BASELINE.md / DESIGN.md).
"""
from __future__ import annotations

import argparse
import csv
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (variant, trees per GPU, n_rollouts)
    "pendulum_65536x100": ("continuous", 65536, 100),
    "cartpole_4096x50": ("discrete", 4096, 50),
    "pendulum_32768x200": ("continuous", 32768, 200),
    "pendulum_1024x25": ("continuous", 1024, 25),  # quick sanity size
    # BASELINE.json configs[4]: self-play loop, 32768 Pendulum environments per GPU (262144 on 8 GPUs) x 200 sims per env step,
    # weight broadcast every SELFPLAY_BROADCAST_EVERY steps, replay rows all-gathered every step
    "selfplay_pendulum_32768x200": ("continuous", 32768, 200),
    "selfplay_pendulum_2048x25": ("continuous", 2048, 25),  # quick sanity size
}


class _Workloads(dict):
    """Named BASELINE configs plus any `pendulum_<trees>x<sims>` / `cartpole_<trees>x<sims>` size (sweeps, strong-scaling shards)."""

    def __missing__(self, name):
        import re
        m = re.fullmatch(r"(selfplay_)?(pendulum|cartpole)_(\d+)x(\d+)", name)
        if not m:
            raise KeyError(name)
        return ("continuous" if m.group(2) == "pendulum" else "discrete", int(m.group(3)), int(m.group(4)))


WORKLOADS = _Workloads(WORKLOADS)
HEADLINE = "pendulum_65536x100"
EXTRA_WORKLOADS = ("cartpole_4096x50", "selfplay_pendulum_32768x200")
SELFPLAY_BROADCAST_EVERY = 4
FLOP_PER_EVAL = {"discrete": 2 * 17280, "continuous": 2 * 34048}  # SURVEY 8d
PARITY_SAMPLE = 256  # trees per rank compared with the oracle inside the bench
DUMP_LIMIT_BYTES = 64 << 20  # --dump-outputs: larger outputs are written as a fixed sample of their rows


def make_roots(variant: str, B: int, seed: int = 34) -> np.ndarray:
    rng = np.random.default_rng(seed)
    if variant == "discrete":
        return rng.uniform(-0.05, 0.05, size=(B, 4))
    return np.stack([rng.uniform(-np.pi, np.pi, B), rng.uniform(-1.0, 1.0, B)], 1)


def make_weights(variant: str) -> np.ndarray:
    from alphazero_gym_b200.network import init_policy_weights
    if variant == "discrete":
        return init_policy_weights(34, 4, 128, 2, 2)
    return init_policy_weights(34, 3, 128, 3, 6)


def engine_config(variant: str, B: int, N: int, device: int, q8: bool = False, fused=None):
    from alphazero_gym_b200.engine import EngineConfig
    from alphazero_gym_b200._cabi import ACT_ELU, ACT_RELU, CONTINUOUS, DISCRETE
    if variant == "discrete":  # run_discrete.yaml / MCTSDiscrete.yaml / DiscretePolicy.yaml
        return EngineConfig(variant=DISCRETE, max_rollouts=N, max_trees=B, num_actions=2, state_dim=4, hidden=128, n_hidden=2,
                            activation=ACT_RELU, c_uct=1.5, gamma=1.0, epsilon=0.1, device=device, seed=34, eval_q8=q8, fused=fused)
    return EngineConfig(variant=CONTINUOUS, max_rollouts=N, max_trees=B, num_components=2, state_dim=3, hidden=128, n_hidden=3,
                        activation=ACT_ELU, c_uct=0.05, c_pw=1.0, kappa=0.5, gamma=1.0, epsilon=0.0, action_bound=2.0,
                        device=device, seed=34, eval_q8=q8, fused=fused)


def oracle_config(variant: str, N: int, q8: bool = False):
    from oracle import azo
    cfg = (azo.discrete_config(n_rollouts=N, epsilon=0.1, math_mode=azo.MATH_DET) if variant == "discrete"
           else azo.continuous_config(n_rollouts=N, math_mode=azo.MATH_DET))
    if q8:
        cfg.eval_mode = azo.EVAL_Q8
    return cfg


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device, self.rows, self.proc, self.thread = device, [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.device)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for r in self.rows:
            if len(r) < 7:
                continue
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def measured_peaks():
    """(HBM GB/s, SM max MHz, dense bf16 TFLOP/s burst, source)"""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d.get("hbm_gbs", 6650.0), d.get("sm_max_mhz", 1965.0), d.get("bf16_tflops", 1650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1965.0, 1650.0, "fallback (B200_PROFILING.md)"


def algorithmic_bytes(variant: str, c: dict) -> float:
    """Algorithmic node-table bytes of the tree-step kernels for one search (SURVEY 8d):
    select  sum_levels [4 node.n + 4 V + 4 chosen link] + children scanned * (8 W + 4 n [+4 prior]);
    backup  sum_levels [8 r + 4 parent link + 2*(8+4) edge W,n rw + 2*4 parent n rw];
    expansion one node row (env state + r 8 + V 4 + n 4 + links 8 [+ priors]) + edge init."""
    per_child = 16 if variant == "discrete" else 12
    expansions = c["sims"] - c["terminal_leaf_sims"]
    exp_bytes = (32 + 8 + 4 + 4 + 8 + 8 + 24) if variant == "discrete" else (16 + 8 + 4 + 4 + 8 + 16)
    return c["levels"] * (12 + 44) + c["children_scanned"] * per_child + expansions * exp_bytes


def measure_traffic(workload: str):
    """DRAM bytes (read + write) of ONE launch of the whole-search kernel, measured now: a two-metric ncu pass over
    tools/ncu_one.py (same workload, same library).  Returns (bytes or None, how)."""
    ncu = "/usr/local/cuda/bin/ncu"
    if not os.path.exists(ncu):
        return None, "ncu not found"
    cmd = [ncu, "--metrics", "dram__bytes_read.sum,dram__bytes_write.sum", "--clock-control", "none", "-k", "regex:k_search_wg|k_qmlp2",
           "-s", "2", "-c", "1", "--csv", sys.executable, os.path.join(ROOT, "tools", "ncu_one.py"), workload]
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=240).stdout
        total = 0.0
        for row in csv.reader(l for l in out.splitlines() if l.startswith('"')):
            if len(row) > 14 and row[12].startswith("dram__bytes_") and row[12].endswith(".sum"):
                scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(row[13])
                if scale is None:
                    return None, f"unknown ncu unit {row[13]}"
                total += float(row[14].replace(",", "")) * scale
        if total > 0:
            return total, "ncu dram__bytes_read.sum + dram__bytes_write.sum of one launch, measured in this run"
        return None, "ncu gave no counters (permissions?)"
    except Exception as exc:  # noqa: BLE001
        return None, f"ncu failed: {exc}"


def dump_outputs(outs: dict, directory: str) -> None:
    """Write each tensor of `outs` (one row per tree or environment) as directory/<name>.npy: float32 as it is, every other
    dtype as float64 (exact for the int32 counts).  Above DUMP_LIMIT_BYTES only a seeded sample of rows is written, the
    same rows for every array, and their indices go to rows.npy."""
    arrs = {k: v.cpu().numpy() for k, v in outs.items()}
    arrs = {k: a if a.dtype == np.float32 else a.astype(np.float64) for k, a in arrs.items()}
    n_rows = len(next(iter(arrs.values())))
    row_bytes = sum(a.nbytes for a in arrs.values()) / n_rows
    budget = DUMP_LIMIT_BYTES - 4096  # room for the .npy headers
    if row_bytes * n_rows > budget:
        rows = np.sort(np.random.default_rng(0).choice(n_rows, int(budget // (row_bytes + 8)), replace=False))
        arrs = {k: a[rows] for k, a in arrs.items()}
        arrs["rows"] = rows.astype(np.float64)
    os.makedirs(directory, exist_ok=True)
    for k, a in arrs.items():
        np.save(os.path.join(directory, k + ".npy"), a)


def cpu_port_throughput(variant: str, N: int, roots: np.ndarray, weights: np.ndarray, seconds: float, threads: int):
    """Time the CPU oracle (C port of the reference search) on a bounded sample; returns (sims/s, sample text)."""
    from oracle import azo
    cfg = oracle_config(variant, N)
    n0 = min(len(roots), 32 * threads)
    t0 = time.perf_counter()
    azo.search(cfg, weights, roots[:n0], dump=False, n_threads=threads)
    rate = n0 * N / (time.perf_counter() - t0)
    n = int(max(n0, min(len(roots), rate * seconds / N)))
    passes = max(1, int(round(rate * seconds / (n * N))))  # the whole batch fits the budget several times: repeat it
    t0 = time.perf_counter()
    for i in range(passes):
        azo.search(cfg, weights, roots[:n], dump=False, n_threads=threads, tree_id0=i * n)
    dt = time.perf_counter() - t0
    return passes * n * N / dt, f"{passes} x first {n} trees x {N} sims of the workload, {threads} threads, {dt:.1f} s"


def run_reference(args, variant, B, N, rank, world):
    """--impl reference: the CPU port on all host cores, each step a bounded sample of the workload."""
    if rank != 0:
        return
    from oracle import azo
    threads = os.cpu_count() or 1
    roots, weights = make_roots(variant, B), make_weights(variant)
    cfg = oracle_config(variant, N)
    # size one step to ~ (120 s budget) / (steps + warmup)
    n0 = min(B, 32 * threads)
    t0 = time.perf_counter()
    azo.search(cfg, weights, roots[:n0], dump=False, n_threads=threads)
    rate = n0 * N / (time.perf_counter() - t0)
    budget = 120.0 / max(1, args.steps + args.warmup)
    n = int(max(n0, min(B, rate * budget / N)))
    for _ in range(args.warmup):
        azo.search(cfg, weights, roots[:n], dump=False, n_threads=threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        azo.search(cfg, weights, roots[:n], dump=False, n_threads=threads)
    dt = time.perf_counter() - t0
    v = n * N * args.steps / dt
    sample = f"{n} of {B} trees x {N} sims per step, {threads} threads"
    line = {"impl": "reference", "metric": "MCTS simulations/sec (batched trees)", "value": v, "unit": "sims/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64 tree statistics / f32 network", "data": "synthetic",
            "config": {"workload": args.workload or HEADLINE, "trees_per_step": n, "n_rollouts": N,
                       "note": "CPU C port (oracle/azg_oracle.c) of the reference's python search; the python reference cannot travel"},
            "cpu_baseline": {"value": v, "unit": "sims/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": "sims/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    _emit(line)


_JSON_OUT = None


def _claim_stdout():
    """stdout carries the ONE JSON line and nothing else: keep a private handle on the real stdout for it and point file descriptor 1 at
    stderr, so that whatever a library prints there (NCCL's version banner under NCCL_DEBUG=VERSION, which ignores NCCL_DEBUG_FILE)
    ends up on stderr."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def _emit(line: dict) -> None:
    print(json.dumps(line), file=_JSON_OUT or sys.stdout, flush=True)


class Ctx:
    """One process per GPU: rank / world / local device and the barrier + max-over-ranks reduction of the timing contract."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback")
        torch.cuda.set_device(self.local)
        if self.world > 1:
            # stdout carries the one JSON line and nothing else: NCCL's own log (its version banner under NCCL_DEBUG=VERSION/INFO) goes to stderr
            os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, values):
        t = self.torch.tensor(list(values), dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(x) for x in t]

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def measure(ctx: Ctx, args, name: str, trees_per_gpu=None, scaling: str = "weak", cpu_baseline: bool = True, traffic: bool = True,
            dump_dir=None) -> dict:
    """One workload on every rank; returns the record (meaningful on rank 0).  With dump_dir, rank 0 writes the outputs of the
    last timed step there (dump_outputs)."""
    torch, dist = ctx.torch, ctx.dist
    from alphazero_gym_b200.engine import SearchEngine
    variant, B_full, N = WORKLOADS[name]
    B = int(trees_per_gpu or B_full)
    rank, world, local = ctx.rank, ctx.world, ctx.local
    q8 = args.eval == "q8"
    tree_id0 = rank * B  # global tree ids: shard r owns trees [r*B, (r+1)*B)
    roots_h = make_roots(variant, B * world)[rank * B:(rank + 1) * B].copy()
    weights = make_weights(variant)
    eng = SearchEngine(engine_config(variant, B, N, local, q8=q8, fused={"auto": None, "on": True, "off": False}[args.fused]))
    eng.set_weights(weights)
    roots_d = torch.from_numpy(roots_h).cuda()
    selfplay = name.startswith("selfplay")
    sp_times = {}
    e2e_blocking_s = None
    if selfplay:
        # ---- self-play loop (BASELINE config 5): search -> final action -> real env step, replay rows all-gathered every
        # step (C2: ONE all_gather_into_tensor of the packed row buffer), weights re-broadcast from rank 0 and re-loaded every
        # SELFPLAY_BROADCAST_EVERY steps (C1)
        from alphazero_gym_b200.selfplay import DeviceReplayBuffer, ROW_KEYS, SelfPlayDriver
        drv = SelfPlayDriver(eng, B, N, max_episode_length=200, tree_id0=tree_id0, total_envs=B * world, seed=34)
        replay = DeviceReplayBuffer(max_size=2 * B * world, batch_size=256, obs_dim=3 if variant == "continuous" else 4,
                                    cmax=eng.cmax, device=eng.device)
        wflat = torch.from_numpy(weights).cuda()
        w_pinned = torch.from_numpy(weights).pin_memory()
        rows_pinned = {k: torch.empty_like(drv.t[k], device="cpu").pin_memory() for k in ROW_KEYS}
        ev_pairs = {"allgather": [], "broadcast": []}

        def timed(kind, fn, record):
            if not record:
                return fn()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            out = fn()
            b.record()
            ev_pairs[kind].append((a, b))
            return out

        def device_step(i, record=False):
            if i % SELFPLAY_BROADCAST_EVERY == 0:
                timed("broadcast", lambda: drv.sync_weights(wflat), record)
            drv.step(store=False)
            replay.store(timed("allgather", drv.gathered_rows, record))

        def host_step(i):
            if i % SELFPLAY_BROADCAST_EVERY == 0:
                wflat.copy_(w_pinned, non_blocking=True)  # the trainer's new weights arrive from the host
                drv.sync_weights(wflat)
            drv.step(store=False)
            replay.store(drv.gathered_rows())
            for k in ROW_KEYS:  # this step's replay rows leave for a host-side consumer
                rows_pinned[k].copy_(drv.t[k], non_blocking=True)
            torch.cuda.synchronize()

        api = "SelfPlayDriver.step (azg_selfplay_step) + per-step D2H of the replay rows, H2D of the weights at broadcast steps"
        h2d = weights.nbytes / SELFPLAY_BROADCAST_EVERY
        d2h = sum(rows_pinned[k].numel() * rows_pinned[k].element_size() for k in ROW_KEYS)
        extra_launches = 2  # root results + the self-play kernel (+ set_seed)
    else:
        res_d = eng.root_results(B)  # result tensors allocated once (a cudaMalloc inside the timed loop synchronises the device)

        def device_step(i, record=False):
            eng.search(roots_d, N, tree_id0=tree_id0)
            return eng.root_results(B, out=res_d)

        host_out = eng.host_buffers(B)  # page-locked, as the contract asks: results arrive by DMA, no staging copy
        roots_pinned = torch.from_numpy(roots_h).pin_memory().numpy()

        def host_step(i):
            return eng.search_host(roots_pinned, N, tree_id0=tree_id0, out=host_out)

        host_out2 = eng.host_buffers(B)

        def host_pipeline(steps):
            """The same K searches through the pipelined entry points (azg_search_host_begin / _end, two slots in flight): every
            step still copies its roots in from pinned host memory and its results out; the D2H of step i runs under step i + 1."""
            outs = (host_out, host_out2)
            for i in range(steps):
                if i >= 2:
                    eng.search_host_end(i & 1)
                eng.search_host_begin(i & 1, roots_pinned, N, outs[i & 1], tree_id0=tree_id0)
            for i in range(max(0, steps - 2), steps):
                eng.search_host_end(i & 1)
            return outs[(steps - 1) & 1]

        h2d = roots_h.nbytes
        extra_launches = 1  # the root-results kernel

    # ---- device-resident throughput ("value") ---------------------------------------------------------
    for i in range(max(args.warmup, 3)):
        device_step(i)
    eng.status()
    clocks = ClockSampler(local)
    ctx.barrier()
    clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        res = device_step(i, record=True)
    e1.record()
    ctx.barrier()
    ms = e0.elapsed_time(e1)
    eng.status()
    if dump_dir and rank == 0:  # before the e2e and roofline passes below reuse the engine
        dump_outputs(drv.t if selfplay else res, dump_dir)
    counters = eng.counters()
    launches_per_step = counters["launches"] + extra_launches
    if selfplay:
        sp_times = {k: (sum(a.elapsed_time(b) for a, b in v) / max(1, len(v)), len(v)) for k, v in ev_pairs.items()}

    # ---- parity inside the bench: a sample of THIS rank's trees against the CPU oracle, bit for bit -------------------
    parity = None
    if not selfplay and q8:
        from oracle import azo
        n = min(PARITY_SAMPLE, B)
        ref = azo.search(oracle_config(variant, N, q8=True), weights, roots_h[:n], tree_id0=tree_id0, dump=False, n_threads=os.cpu_count() or 1)
        c = ref["counts"].shape[1]
        same = all(np.array_equal(res[k][:n].cpu().numpy()[:, :c] if res[k].dim() == 2 else res[k][:n].cpu().numpy(), ref[k])
                   for k in ("counts", "actions", "Q", "V_target", "n_children"))
        assert same, f"rank {rank}: root results of the first {n} trees differ from the CPU oracle"
        flag = torch.tensor([1.0 if same else 0.0], device="cuda")
        if world > 1:
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        parity = {"trees_per_rank": n, "ranks": world, "bit_identical_to_oracle": bool(flag.item() == 1.0),
                  "compared": "counts, actions, Q, V_target, n_children of each rank's first trees (global tree ids rank*B ...)"}

    # ---- end to end through the host-facing entry point ("e2e") -------------------------------------
    for i in range(2):
        out = host_step(i)
    ctx.barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        out = host_step(i)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if selfplay:
        api_s = api
    else:  # the pipelined entry points: the number reported as e2e; the blocking call's stays next to it
        host_pipeline(2)
        ctx.barrier()
        t0 = time.perf_counter()
        out = host_pipeline(args.steps)
        e2e_blocking_s, e2e_s = e2e_s, time.perf_counter() - t0
        api_s = ("azg_search_host_begin / azg_search_host_end via SearchEngine.search_host_begin / _end, two searches in flight, page-locked "
                 "host buffers (wall clock from the first begin to the last end); blocking_value = azg_search_host, one call per step")
    clk = clocks.stop()
    checksum = int(drv.t["counts"].sum()) if selfplay else int(out["counts"].sum())
    assert checksum == B * N, f"visit counts do not add up: {checksum} != {B * N}"
    if selfplay:
        roots_d = drv.env_state.clone()
    else:
        d2h = sum(out[k].nbytes for k in ("actions", "counts", "Q", "V_target", "n_children"))

    # ---- roofline of the dominant kernel, timed live ----------------------------------------------------
    hbm_peak, sm_max_mhz, bf16_peak, peak_src = measured_peaks()
    sm_count = torch.cuda.get_device_properties(local).multi_processor_count
    fp32_peak = sm_count * 128 * 2 * sm_max_mhz * 1e6 / 1e12
    roof_all = {}
    if eng.cfg.is_fused():
        # the search is ONE persistent launch per chunk of trees (search_wg.cuh): CUDA events around back-to-back launches
        eng.fused_stats()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = max(3, args.steps)
        f0.record()
        for _ in range(reps):
            eng.search(roots_d, N, tree_id0=tree_id0)
        f1.record()
        torch.cuda.synchronize()
        k_ms = f0.elapsed_time(f1) / reps / max(1, counters["launches"])
        st = eng.fused_stats()
        fc = eng.counters()
        flop = FLOP_PER_EVAL[variant] * fc["evals"] / max(1, counters["launches"])
        tflops = flop / (k_ms * 1e-3) / 1e12
        tbytes = algorithmic_bytes(variant, fc) / max(1, counters["launches"])
        hh = 2 * 128 * 128 * ((3 if variant == "continuous" else 2) - 1)
        tr_bytes, tr_how = (measure_traffic(name) if (traffic and rank == 0 and world == 1 and not selfplay) else (None, "not measured for this record"))
        if tr_bytes is None:
            tp = os.path.join(ROOT, "profiles", "traffic.json")
            if os.path.exists(tp):
                with open(tp) as f:
                    tr_bytes = json.load(f).get(name, {}).get("k_search")
                tr_how += "; value from profiles/traffic.json (an earlier ncu capture)" if tr_bytes else ""
        tree_s, slot_s, mma_s = st["tree_phase"], st["wait_for_post_processing"], st.get("x_wait_mma", 0.0)
        two_phase = st["kernel"] != "warpgroups"  # engine.cu launch_fused_t picks by batch size
        tsm = st["kernel"] == "two_phase_trees_in_shared_memory"
        wg_time = ({"evaluation_phases": 1.0 - tree_s, "tree_phases": tree_s, "evaluation_warps_waiting_for_row_finish": slot_s,
                    "source": "in-kernel cycle counters (azg_fused_stats), CTA average; the two phases alternate for the whole CTA"} if two_phase else
                   {"evaluation_with_tmem_slot": 1.0 - tree_s - slot_s, "of_which_waiting_for_mma": mma_s, "tree_step_and_row_finish": tree_s,
                    "waiting_for_a_tmem_slot": slot_s, "source": "in-kernel cycle counters (azg_fused_stats), average over warpgroups"})
        dominant = {
            "kernel": ("k_qmlp2<FUSED, TSM> (whole search in one persistent kernel, the CTA's trees resident in SHARED MEMORY for the whole search: "
                       "per simulation an evaluation phase on tcgen05 kind::i8 and a tree phase with a group of 8 lanes per tree)" if tsm else
                       "k_qmlp2<FUSED> (whole search in one persistent kernel, thin batches: per simulation an evaluation phase on tcgen05 kind::i8 with "
                       "16 warps per tile pair and a tree phase, one thread per tree)" if two_phase else
                       "k_search_wg (whole search in one persistent kernel; four independent warpgroups per SM, a thread owns its tree's step "
                       "and its row of the tcgen05 kind::i8 evaluation)"),
            "bound": "tensor", "achieved": tflops, "peak": bf16_peak, "unit": "TFLOP/s", "frac": tflops / bf16_peak,
            "traffic": tr_bytes, "traffic_source": tr_how, "peak_source": peak_src + " dense bf16; int8 digits: 6 digit products per algorithmic product",
            "avg_launch_ms": k_ms, "launches": counters["launches"], "flop_per_launch": flop,
            "tensor_tops_issued": 6 * hh * fc["evals"] / max(1, counters["launches"]) / (k_ms * 1e-3) / 1e12,
            "frac_of_fp32_cuda_core_peak": tflops / fp32_peak, "share_of_step": k_ms * counters["launches"] / (ms / args.steps) if not selfplay else None,
            "hbm": {"algorithmic_bytes_per_launch": tbytes, "algorithmic_gbs": tbytes / (k_ms * 1e-3) / 1e9,
                    "frac_of_hbm_peak": tbytes / (k_ms * 1e-3) / 1e9 / hbm_peak,
                    "traffic_over_algorithmic": (tr_bytes / tbytes) if tr_bytes else None,
                    "note": ("select + backup + expansion bytes (SURVEY 8d formula from the engine's own counters) over the WHOLE kernel's time; "
                             "in this kernel they are served from shared memory (the rows reach HBM once, when the search ends), so the HBM "
                             "roofline does not bound it" if tsm else
                             "select + backup + expansion bytes (SURVEY 8d formula from the engine's own counters) over the WHOLE kernel's time: "
                             "the tree step overlaps the evaluation of other warpgroups, so it has no time of its own")},
            "time_split": wg_time,
        }
        roof_all = {"whole_search_kernel": dominant}
    else:
        eng.profile_search(roots_d, N, tree_id0=tree_id0)
        prof = eng.profile_search(roots_d, N, tree_id0=tree_id0)
        pc = eng.counters()
        ev, tr = prof["evaluation"], prof["tree_step"]
        ev_avg_ms, tr_avg_ms = ev["ms"] / max(1, ev["launches"]), tr["ms"] / max(1, tr["launches"])
        ev_tflops = FLOP_PER_EVAL[variant] * B / (ev_avg_ms * 1e-3) / 1e12
        tr_bytes = algorithmic_bytes(variant, pc) / max(1, tr["launches"])
        tr_gbs = tr_bytes / (tr_avg_ms * 1e-3) / 1e9
        tot = ev["ms"] + tr["ms"] + prof["setup"]["ms"]
        roof_eval = {"kernel": "k_qmlp2 (tcgen05 kind::i8)" if q8 else "k_mlp (FP32 FMA)", "bound": "tensor" if q8 else "fp32", "achieved": ev_tflops,
                     "peak": bf16_peak if q8 else fp32_peak, "unit": "TFLOP/s", "frac": ev_tflops / (bf16_peak if q8 else fp32_peak), "traffic": None,
                     "avg_launch_ms": ev_avg_ms, "launches": ev["launches"], "share_of_step": ev["ms"] / tot}
        roof_tree = {"kernel": "k_step (backup + select + expansion/env step)", "bound": "hbm", "achieved": tr_gbs, "peak": hbm_peak, "unit": "GB/s",
                     "frac": tr_gbs / hbm_peak, "traffic": None, "peak_source": peak_src, "avg_launch_ms": tr_avg_ms, "launches": tr["launches"],
                     "algorithmic_bytes_per_launch": tr_bytes, "share_of_step": tr["ms"] / tot}
        dominant = roof_eval if ev["ms"] >= tr["ms"] else roof_tree
        roof_all = {"evaluation": roof_eval, "tree_step": roof_tree}
        fc = pc

    # ---- CPU baseline (rank 0, N=1 only) ------------------------------------------------------------------
    cpu = None
    if cpu_baseline and rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        v, sample = cpu_port_throughput(variant, N, roots_h, weights, args.cpu_seconds, threads)
        if selfplay:
            sample += " (searches only; the env step and bookkeeping are negligible next to them)"
        cpu = {"value": v, "unit": "sims/s", "cores": threads, "kind": "port", "sample": sample}

    # ---- max over ranks ---------------------------------------------------------------------------------------
    ms_max, e2e_ms_max, e2e_blocking_ms_max = ctx.max_over_ranks([ms, e2e_s * 1e3, (e2e_blocking_s or 0.0) * 1e3])
    total_sims = world * B * N * args.steps
    rec = {
        "workload": name, "value": total_sims / (ms_max * 1e-3), "unit": "sims/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_max / args.steps, "scaling": scaling,
        "config": {"workload": name, "eval": args.eval, "whole_search_kernel": bool(eng.cfg.is_fused()),
                   "env": "Pendulum-v0" if variant == "continuous" else "CartPole-v0",
                   "trees_per_gpu": B, "global_trees": B * world, "n_rollouts": N,
                   "parallelism": f"tree-sharded x{world}, no data-path collective" + (" in the search; C1 + C2 around it" if selfplay else ""),
                   "weights": "default init, torch.manual_seed(34)", "roots": "numpy default_rng(34)",
                   "l2": ("node tables per GPU (%.0f MB) exceed the 126 MB L2; no explicit flush" % (eng.rows * B * (64 + 32) / 1e6))
                   if eng.rows * B * 96 > 126e6 else "tables are L2-resident at this size; no explicit flush (SURVEY 8d says so for config 3)"},
        "e2e": {"value": total_sims / (e2e_ms_max * 1e-3), "unit": "sims/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_ms_max / args.steps, "api": api_s,
                **({"blocking_value": total_sims / (e2e_blocking_ms_max * 1e-3)} if e2e_blocking_ms_max > 0 else {})},
        "gpu_launches": launches_per_step * args.steps,
        **({"selfplay": {"max_episode_length": 200, "weight_broadcast_every_steps": SELFPLAY_BROADCAST_EVERY,
                         "collectives": "C2 = ONE all_gather_into_tensor of the packed replay-row buffer per step (%d B per rank); "
                                        "C1 = broadcast of the flat f32 weights (%d B) every %d steps" % (drv.packed.nbytes, weights.nbytes, SELFPLAY_BROADCAST_EVERY),
                         "allgather_ms_per_step": sp_times.get("allgather", (None, 0))[0], "broadcast_plus_set_weights_ms": sp_times.get("broadcast", (None, 0))[0],
                         "backend": "nccl" if world > 1 else "none (1 GPU: the gather is the identity)"}} if selfplay else {}),
        "clocks": clk, "roofline": dominant, "roofline_all": roof_all,
        "counters_per_sim": {k: fc[k] / max(1, fc["sims"]) for k in ("levels", "children_scanned", "pw_inserts", "evals")},
        "cpu_baseline": cpu, "parity": parity,
    }
    eng.close()
    return rec


class _CartPoleEnv:  # what the drop-in classes read of a gym env: the class name and the hidden state (search/mcts.py env_hidden_state)
    def __init__(self, state):
        self.state, self.unwrapped = np.asarray(state, np.float64), self


class _PendulumEnv(_CartPoleEnv):
    pass


def single_tree_latency(searches: int = 200) -> dict:
    """BASELINE configs[0] and configs[1]: ONE tree through the reference-facing drop-in call `MCTS*.search(Env)` +
    `return_results` (run_discrete.yaml / run_continuous.yaml defaults: 8 / 25 rollouts), host buffers in and out, and the CPU
    port on one core next to it.  (The Python reference itself measured 1431 / 935 sims/s on one core of the build container.)"""
    import torch
    from oracle import azo
    from alphazero_gym_b200.network import PolicyNet
    from alphazero_gym_b200.search.mcts import MCTSContinuous, MCTSDiscrete
    out = {}
    for name, variant, N in (("cartpole_1x8", "discrete", 8), ("pendulum_1x25", "continuous", 25)):
        w, roots = make_weights(variant), make_roots(variant, searches)
        if variant == "discrete":
            net = PolicyNet(4, 128, 2, 2, "relu", num_actions=2).load_flat(w)
            m = MCTSDiscrete(model=net, num_actions=2, n_rollouts=N, c_uct=1.5, gamma=1, epsilon=0.1, V_target_policy="off_policy", device="cuda:0", root_state=None)
            envs = [_CartPoleEnv(r) for r in roots]
        else:
            net = PolicyNet(3, 128, 3, 6, "elu", num_components=2, action_bound=2.0).load_flat(w)
            m = MCTSContinuous(model=net, n_rollouts=N, c_uct=0.05, c_pw=1, kappa=0.5, gamma=1, epsilon=0, V_target_policy="off_policy", device="cuda:0", root_state=None)
            envs = [_PendulumEnv(r) for r in roots]
        for e in envs[:10]:
            m.root_node, m.root_state = None, None
            m.search(Env=e)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for e in envs:
            m.root_node, m.root_state = None, None  # reset_mcts (agents.py:146-155)
            m.search(Env=e)
            m.return_results("max_visit")
        dt = time.perf_counter() - t0
        m.close()
        cfg = oracle_config(variant, N)
        t0 = time.perf_counter()
        for i in range(searches):
            azo.search(cfg, w, roots[i:i + 1], dump=False, n_threads=1, tree_id0=i)
        dc = time.perf_counter() - t0
        out[name] = {"ms_per_search": 1e3 * dt / searches, "sims_per_s": searches * N / dt, "searches": searches,
                     "api": "MCTSDiscrete/MCTSContinuous.search(Env) + return_results (drop-in classes, tensor-core evaluation, one launch per search)",
                     "cpu_port_one_core": {"ms_per_search": 1e3 * dc / searches, "sims_per_s": searches * N / dc}}
    return out


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None,
                    help="one workload only: %s or any pendulum_<trees>x<sims> / cartpole_<trees>x<sims> "
                         "(default: the headline workload + the other BASELINE configs under `workloads`)" % ", ".join(sorted(WORKLOADS)))
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU baseline sample budget")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="headline workload only: no `workloads`, no `strong` record")
    ap.add_argument("--fused", default="auto", choices=["auto", "on", "off"],
                    help="whole-search persistent kernel (AZG_FLAG_FUSED); auto = the engine's default")
    ap.add_argument("--eval", default="q8", choices=["fp32", "q8"],
                    help="leaf evaluation arithmetic: int8-sliced tcgen05 products (default) or FP32 FMA (mlp.cuh)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the headline workload's last timed step as DIR/<name>.npy (float32/float64, at most 64 MB)")
    args = ap.parse_args()
    head = args.workload or HEADLINE
    variant, B, N = WORKLOADS[head]
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs needs --impl ours")
        run_reference(args, variant, B, N, int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")))
        return
    ctx = Ctx()
    rec = measure(ctx, args, head, dump_dir=args.dump_outputs)
    extras, strong = {}, None
    if args.workload is None and not args.no_extra:
        for name in EXTRA_WORKLOADS:
            extras[name] = measure(ctx, args, name, traffic=not name.startswith("selfplay"))  # (measure() skips the ncu pass at N > 1)
        if ctx.world > 1 and B % ctx.world == 0:
            # BASELINE config 4 as worded: the SAME 65536 trees sharded B / N per GPU (parallel.shard_range): strong scaling
            strong = measure(ctx, args, head, trees_per_gpu=B // ctx.world, scaling="strong", cpu_baseline=False, traffic=False)
    if ctx.rank == 0:
        line = {"metric": "MCTS simulations/sec (batched trees)", "higher_is_better": True, "vs_baseline": None,
                "dtype": "f64 tree statistics + env dynamics / " + ("f32 network with exact int8-sliced tensor-core products" if args.eval == "q8" else "f32 network"),
                "data": "synthetic"}
        line.update({k: v for k, v in rec.items() if k != "workload"})
        if extras:
            line["workloads"] = extras
        if args.workload is None and not args.no_extra and ctx.world == 1:
            line["single_tree"] = single_tree_latency()
        if strong is not None:
            line["strong"] = {k: strong[k] for k in ("value", "unit", "n_gpus", "ms_per_step", "scaling", "config", "e2e", "gpu_launches", "parity", "clocks")}
            line["strong"]["roofline_frac"] = strong["roofline"]["frac"]
        _emit(line)
    ctx.close()


if __name__ == "__main__":
    main()
