"""DeviceReplayBuffer (alphazero_gym_b200/selfplay.py) keeps the semantics of the reference's list-based ReplayBuffer
(alphazero/agent/buffers.py): FIFO with overwrite of the oldest entry, shuffled mini-batches with the remainder folded into
the last batch.  Runs on CPU tensors here; the same code holds CUDA tensors in the self-play driver."""
import pytest
import torch

from alphazero_gym_b200.selfplay import DeviceReplayBuffer, ROW_KEYS


def _rows(lo, hi, cmax=3, S=3):
    n = hi - lo
    ids = torch.arange(lo, hi)
    return dict(obs=ids[:, None].float().repeat(1, S), actions=ids[:, None].float().repeat(1, cmax),
                counts=ids[:, None].int().repeat(1, cmax), Q=ids[:, None].double().repeat(1, cmax), V_target=ids.double())


class _RefBuffer:
    """restatement of buffers.py:61-79 (store) for single experiences"""
    def __init__(self, max_size):
        self.max_size, self.exp, self.ins = max_size, [], 0

    def store(self, e):
        if len(self.exp) < self.max_size:
            self.exp.append(e)
        else:
            self.exp[self.ins] = e
            self.ins += 1
            if self.ins >= len(self.exp):
                self.ins = 0


@pytest.mark.parametrize("chunks", [[4, 4, 4, 4, 4], [7, 7, 7], [3, 10, 2, 9], [25]])
def test_fifo_matches_reference_order(chunks):
    rb = DeviceReplayBuffer(max_size=10, batch_size=4, obs_dim=3, cmax=3, device="cpu")
    ref = _RefBuffer(10)
    lo = 0
    for n in chunks:
        rb.store(_rows(lo, lo + n))
        for i in range(lo, lo + n):
            ref.store(i)
        lo += n
    assert len(rb) == len(ref.exp)
    assert rb.data["V_target"][: len(rb)].tolist() == [float(x) for x in ref.exp]
    for k in ROW_KEYS:
        assert rb.data[k][: len(rb)].reshape(len(rb), -1)[:, 0].tolist() == [float(x) for x in ref.exp]


def test_batches_cover_the_buffer_once_per_epoch():
    rb = DeviceReplayBuffer(max_size=64, batch_size=8, obs_dim=3, cmax=3, device="cpu")
    rb.store(_rows(0, 37))
    rb.reshuffle(torch.Generator().manual_seed(0))
    sizes, seen = [], []
    for b in rb:
        sizes.append(b["V_target"].shape[0])
        seen += b["V_target"].tolist()
        assert b["actions"].shape == (sizes[-1], 3) and b["counts"].dtype == torch.int32
    # buffers.py:98-127: full batches, the last one takes the remainder (37 = 8 + 8 + 8 + 13)
    assert sizes == [8, 8, 8, 13]
    assert sorted(seen) == [float(i) for i in range(37)]


# What the reference's ReplayBuffer(max_size=10, batch_size=4) holds after the rows 0..26 were stored one by one: V of its
# experience list in list order, and the sizes of the mini-batches it yields after reshuffle().  Recorded here because the
# reference is not part of this repository.
REF_EXPERIENCE_V = [20, 21, 22, 23, 24, 25, 26, 17, 18, 19]
REF_BATCH_SIZES = [4, 6]


def test_against_the_reference_class():
    rb = DeviceReplayBuffer(max_size=10, batch_size=4, obs_dim=3, cmax=3, device="cpu")
    for lo in range(0, 27, 3):
        rb.store(_rows(lo, lo + 3))
    assert [float(v) for v in REF_EXPERIENCE_V] == rb.data["V_target"][: len(rb)].tolist()
    rb.reshuffle()
    assert REF_BATCH_SIZES == [b["obs"].shape[0] for b in rb]
