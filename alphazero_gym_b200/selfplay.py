"""Batched self-play on the device: the reference's episode loop (run_continuous.py:112-142, run_discrete.py:95-122)
for B independent environments per GPU, plus the replay buffer (alphazero/agent/buffers.py) as device tensors.

One `SelfPlayDriver.step()` = `azg_selfplay_step` (include/azg.h): search -> replay row -> final action -> real env step ->
episode bookkeeping, all enqueued on the current CUDA stream; nothing returns to the host.  Across GPUs (one process per
GPU) the environments are sharded by global tree id; the only exchanges are the periodic weight broadcast (C1) and the
all-gather of replay rows (C2), both outside the search (alphazero_gym_b200/parallel.py).  PyTorch is plumbing here:
tensors, streams, torch.distributed.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional

import numpy as np
import torch

from . import _cabi
from ._cabi import CONTINUOUS, DISCRETE, check
from .engine import ACROBOT, MOUNTAIN_CAR, MOUNTAIN_CAR_CONTINUOUS, SearchEngine
from .parallel import PackedRows, allgather_results, broadcast_weights

ROW_KEYS = ("obs", "actions", "counts", "Q", "V_target")  # buffer.store((s, actions, counts, Qs, V)), buffers.py:61


def initial_states(variant: int, B: int, seed: int = 34, tree_id0: int = 0, total: Optional[int] = None,
                   env: Optional[str] = None) -> np.ndarray:
    """Env.reset() for every environment: the same rule as SURVEY 8d configs 3/4 (numpy default_rng(seed) over the GLOBAL
    batch, this shard's slice).  env (engine.EngineConfig.env): MOUNTAIN_CAR (discrete) and MOUNTAIN_CAR_CONTINUOUS draw
    position ~ U(-0.6, -0.4), velocity 0; ACROBOT draws the four state entries ~ U(-0.1, 0.1)."""
    if total is None:
        # the draw below runs over the GLOBAL batch, so every rank must use the same `total`: tree_id0 + B is only right for a
        # single shard (or the last one)
        if _dist_world() > 1:
            raise ValueError("initial_states: pass total (the global number of environments) when torch.distributed is initialised")
        total = tree_id0 + B
    rng = np.random.default_rng(seed)
    if variant == DISCRETE and env == ACROBOT:
        s = rng.uniform(-0.1, 0.1, size=(total, 4))
    elif variant == DISCRETE and env != MOUNTAIN_CAR:
        s = rng.uniform(-0.05, 0.05, size=(total, 4))
    elif env in (MOUNTAIN_CAR, MOUNTAIN_CAR_CONTINUOUS):
        s = np.stack([rng.uniform(-0.6, -0.4, total), np.zeros(total)], 1)
    else:
        s = np.stack([rng.uniform(-np.pi, np.pi, total), rng.uniform(-1.0, 1.0, total)], 1)
    return np.ascontiguousarray(s[tree_id0:tree_id0 + B])


def _dist_world() -> int:
    import torch.distributed as dist
    return dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1


class DeviceReplayBuffer:
    """FIFO replay buffer of root-result rows, resident in HBM (reference: ReplayBuffer, buffers.py:6-129).

    Same semantics as the reference's list + insertion index: rows are appended until `max_size`, then overwrite the
    oldest (buffers.py:61-79); `reshuffle` + iteration yield shuffled mini-batches, the last one taking the remainder
    (buffers.py:98-127), collated as stacked tensors (the reference's np.stack).  Rows arrive B at a time."""

    def __init__(self, max_size: int, batch_size: int, obs_dim: int, cmax: int, device):
        self.max_size, self.batch_size = int(max_size), int(batch_size)
        self.device = torch.device(device)
        f32, i32, f64 = torch.float32, torch.int32, torch.float64
        self.data = dict(obs=torch.zeros((max_size, obs_dim), dtype=f32, device=self.device),
                         actions=torch.zeros((max_size, cmax), dtype=f32, device=self.device),
                         counts=torch.zeros((max_size, cmax), dtype=i32, device=self.device),
                         Q=torch.zeros((max_size, cmax), dtype=f64, device=self.device),
                         V_target=torch.zeros(max_size, dtype=f64, device=self.device))
        self.clear()
        self.sample_array: Optional[torch.Tensor] = None
        self.sample_index = 0

    def clear(self) -> None:
        self.insert_index = 0
        self.size = 0

    def __len__(self) -> int:
        return self.size

    def store(self, rows: Dict[str, torch.Tensor]) -> None:
        """Append n rows (dict of tensors with a leading dimension n) in order, overwriting the oldest when full."""
        n = rows["obs"].shape[0]
        done = 0
        while done < n:
            if self.size < self.max_size:
                pos, room = self.size, self.max_size - self.size
            else:
                pos, room = self.insert_index, self.max_size - self.insert_index
            k = min(room, n - done)
            for key in ROW_KEYS:
                self.data[key][pos:pos + k].copy_(rows[key][done:done + k])
            if self.size < self.max_size:
                self.size += k
            else:
                self.insert_index = (self.insert_index + k) % self.max_size
            done += k

    def reshuffle(self, generator: Optional[torch.Generator] = None) -> None:
        self.sample_array = torch.randperm(self.size, device=self.device, generator=generator)
        self.sample_index = 0

    def __iter__(self):
        return self

    def __next__(self) -> Dict[str, torch.Tensor]:
        if self.sample_array is None:
            self.reshuffle()
        if self.sample_index + self.batch_size > self.size and self.sample_index != 0:
            self.reshuffle()
            raise StopIteration
        if self.sample_index + 2 * self.batch_size > self.size:
            idx = self.sample_array[self.sample_index:]
        else:
            idx = self.sample_array[self.sample_index:self.sample_index + self.batch_size]
        self.sample_index += self.batch_size
        return {k: self.data[k][idx] for k in ROW_KEYS}


class SelfPlayDriver:
    """B environments of one GPU advancing in lock step.  `tree_id0` is the global id of environment 0 (rank * B under
    torchrun), which keys every random stream, so results do not depend on how the environments are sharded."""

    def __init__(self, engine: SearchEngine, B: int, n_rollouts: int, max_episode_length: int = 200, tree_id0: int = 0,
                 total_envs: Optional[int] = None, seed: int = 34, deterministic: bool = False, final_selection: str = "max_visit",
                 temperature: float = 1.0, replay: Optional[DeviceReplayBuffer] = None):
        self.eng, self.B, self.N = engine, int(B), int(n_rollouts)
        self.max_episode_length, self.tree_id0, self.seed = int(max_episode_length), int(tree_id0), int(seed)
        if total_envs is None:
            # equal shards of B environments per rank (bench.py, the gloo tests); a ragged split must say its total
            total_envs = _dist_world() * B if _dist_world() > 1 else tree_id0 + B
        self.total = int(total_envs)
        self.deterministic = bool(deterministic)
        self.by_value = final_selection == "max_value"  # any other value means visit counts (agents.py:294-301)
        self.temperature = float(temperature)
        self.replay = replay
        self.step_index = 0
        dev = engine.device
        cfg = engine.cfg
        sd, S, cm = engine.state_cols, cfg.state_dim, engine.cmax
        self.variant = cfg.variant
        z = lambda shape, dt: torch.zeros(shape, dtype=dt, device=dev)
        self.env_state = torch.from_numpy(initial_states(cfg.variant, B, seed, tree_id0, self.total, cfg.env_name())).to(dev)
        # the replay row of a step (ROW_KEYS) lives in ONE byte buffer, so that its all-gather is a single collective (parallel.PackedRows)
        self.packed = PackedRows([("Q", (cm,), torch.float64), ("V_target", (), torch.float64), ("obs", (S,), torch.float32),
                                  ("actions", (cm,), torch.float32), ("counts", (cm,), torch.int32)], B, dev)
        self.t = dict(ep_step=z(B, torch.int32), episode=z(B, torch.int32), root_n=z(B, torch.int32), n_children=z(B, torch.int32),
                      action_taken=z(B, torch.float32), reward=z(B, torch.float64), done=z(B, torch.int32), **self.packed.views)
        t = self.t
        self._io = _cabi.SelfPlayIO(self.env_state.data_ptr(), t["ep_step"].data_ptr(), t["episode"].data_ptr(),
                                    t["root_n"].data_ptr() if cfg.variant == DISCRETE else None, t["obs"].data_ptr(),
                                    t["actions"].data_ptr(), t["counts"].data_ptr(), t["Q"].data_ptr(), t["V_target"].data_ptr(),
                                    t["n_children"].data_ptr(), t["action_taken"].data_ptr(), t["reward"].data_ptr(),
                                    t["done"].data_ptr())
        self.episode_return = z(B, torch.float64)  # return of the running episode (of the finished one where done is set)
        self._prev_done = torch.zeros(B, dtype=torch.bool, device=dev)

    def set_states(self, states: np.ndarray) -> None:
        self.env_state.copy_(torch.from_numpy(np.ascontiguousarray(states, np.float64)).to(self.env_state.device))

    def step(self, store: bool = True) -> Dict[str, torch.Tensor]:
        """One env step of every environment; returns this step's tensors (views that the next step overwrites)."""
        eng = self.eng
        with torch.cuda.device(eng.device):
            check(eng._lib.azg_selfplay_step(eng._h, self.B, C.byref(self._io), self.N, self.tree_id0, self.step_index, self.seed,
                                             self.max_episode_length, int(self.deterministic), int(self.by_value),
                                             self.temperature, torch.cuda.current_stream().cuda_stream))
        eng.last_B = self.B
        self.step_index += 1
        self.episode_return = torch.where(self._prev_done, torch.zeros_like(self.episode_return), self.episode_return) + self.t["reward"]
        self._prev_done = self.t["done"] != 0  # the NEXT step starts a new episode for these environments
        if store and self.replay is not None:
            self.replay.store(self.rows())
        return self.t

    def rows(self) -> Dict[str, torch.Tensor]:
        return {k: self.t[k] for k in ROW_KEYS}

    def gathered_rows(self) -> Dict[str, torch.Tensor]:
        """(C2) this step's replay rows of every rank, in global environment order: ONE all_gather_into_tensor of the packed row
        buffer when every rank owns B environments (the sharding of bench.py), the per-tensor pad-and-trim gather otherwise."""
        if self.total == _dist_world() * self.B:
            return self.packed.gathered()
        return allgather_results(self.rows(), self.total)

    def sync_weights(self, flat: torch.Tensor, src: int = 0) -> None:
        """(C1) broadcast the trainer rank's flat weight vector and load it into the engine."""
        broadcast_weights(flat, src=src)
        self.eng.set_weights(flat)
