"""CPU checks of the slot schedule of eval_drag.evaluate_stream (continuous batching of clips over a fixed number of engine rows)."""
import numpy as np
import pytest

from dragposer_b200.eval_drag import boundary_period, slot_schedule


@pytest.mark.parametrize("slots,period", [(1, 4), (3, 4), (8, 16), (8, 4), (32, 16)])
def test_slot_schedule_runs_every_clip_on_its_own_frames_from_a_boundary(slots, period):
    rng = np.random.default_rng(slots * 100 + period)
    lens = [int(n) for n in rng.integers(1, 400, 50)]
    starts, total = slot_schedule(lens, slots, period)
    assert len(starts) == len(lens)
    runs = {}
    for i, ((s, t), n) in enumerate(zip(starts, lens)):
        assert 0 <= s < slots and t % period == 0  # restarts land on boundaries
        assert t + n <= total  # every clip runs all of its own frames inside the run
        runs.setdefault(s, []).append((t, t + n, i))
    assert total == max(t + n for (_, t), n in zip(starts, lens))
    assert [i for i in range(min(slots, len(lens)))] == [i for i, (_, t) in enumerate(starts) if t == 0][: min(slots, len(lens))]
    for s, rs in runs.items():
        rs.sort()
        for (a0, a1, i), (b0, b1, j) in zip(rs[:-1], rs[1:]):
            assert a1 <= b0  # no slot holds two clips at once
            assert b0 - a1 < period  # and it waits less than one period for the next clip
            assert i < j  # files are taken in order
    assert [t for _, t in starts] == sorted(t for _, t in starts)  # a later file never starts before an earlier one


def test_slot_schedule_edge_cases():
    assert slot_schedule([], 4, 16) == ([], 0)
    assert slot_schedule([5], 3, 16) == ([(0, 0)], 5)  # fewer clips than slots
    starts, total = slot_schedule([10, 3, 7], 2, 4)
    assert starts == [(0, 0), (1, 0), (1, 4)] and total == 11  # slot 1 frees at frame 3 and takes the third clip at frame 4
    assert boundary_period(0) == 4 and boundary_period(16) == 16
