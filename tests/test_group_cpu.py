"""Row routing of a multi-GPU index (wise_b200/routing.py): quotas, splits of adds at shard boundaries, the fill-first
rule without a reservation, the ids of rows added without ids, and the WISE_B200_DEVICES switch.  No GPU needed."""
import numpy as np
import pytest

from wise_b200 import routing
from wise_b200.faiss_compat import resolve_devices


@pytest.mark.parametrize("n,world", [(0, 2), (1, 2), (7, 3), (10, 4), (1000003, 8)])
def test_quotas_are_balanced_and_contiguous(n, world):
    q = routing.quotas(n, world)
    assert sum(q) == n and max(q) - min(q) <= 1
    lo = 0
    for s in range(world):
        assert routing.shard_range(n, s, world) == (lo, lo + q[s])
        lo += q[s]


def _apply(plan, counts):
    for s, _, c in plan:
        counts[s] += c


def test_reserved_adds_fill_each_quota_and_split_at_boundaries():
    n, world = 103, 3
    quota = routing.quotas(n, world)  # [34, 34, 35]
    counts = [0] * world
    pieces = []
    for m in (20, 20, 20, 43):  # the second add straddles the 0|1 boundary, the fourth the 1|2 boundary
        plan = routing.plan_add(m, counts, quota)
        assert sum(c for _, _, c in plan) == m
        assert [a for _, a, _ in plan] == list(np.cumsum([0] + [c for _, _, c in plan])[:-1])
        pieces.append(plan)
        _apply(plan, counts)
    assert counts == quota
    assert pieces[1] == [(0, 0, 14), (1, 14, 6)]
    assert pieces[3] == [(1, 0, 8), (2, 8, 35)]


def test_past_the_reservation_the_last_shard_takes_the_rest():
    counts = [5, 5]
    assert routing.plan_add(7, counts, [5, 5]) == [(1, 0, 7)]


def test_without_a_reservation_a_shard_fills_until_its_memory_is_used():
    row = 64 * 4 + 8
    free = routing._MEM_RESERVE + 3000 * row
    # a store of 1024 rows whose 1.5x growth fits: the shard can reach the rows that fit in the free memory
    assert routing.rows_that_fit(1000, 1024, free, row) == 3000
    # the growth to 1.5x the capacity no longer fits: the shard is full at its capacity
    assert routing.rows_that_fit(1000, 2500, free, row) == 2500
    counts = [1000, 0, 0]
    limits = [3000, 3000, None]
    plan = routing.plan_add(6000, counts, limits)
    assert plan == [(0, 0, 2000), (1, 2000, 3000), (2, 5000, 1000)]
    # a later add goes on from the last shard that holds rows: shard ranges stay contiguous
    assert routing.plan_add(10, [3000, 3000, 1000], [3000, 3000, None]) == [(2, 0, 10)]
    # an empty first shard stays empty only if nothing was routed to it: rows start at shard 0
    assert routing.plan_add(4, [0, 0], [None, None]) == [(0, 0, 4)]


def test_ids_of_rows_added_without_ids_are_global_positions():
    # IndexFlatIP.add on a multi-GPU index passes the global positions as explicit ids, split like the rows
    counts = [0, 0]
    quota = routing.quotas(10, 2)
    got = {0: [], 1: []}
    total = 0
    for m in (3, 4, 3):
        ids = np.arange(total, total + m)
        for s, a, c in routing.plan_add(m, counts, quota):
            got[s] += ids[a:a + c].tolist()
            counts[s] += c
        total += m
    assert got == {0: [0, 1, 2, 3, 4], 1: [5, 6, 7, 8, 9]}


def test_devices_come_from_the_argument_then_the_environment(monkeypatch):
    monkeypatch.delenv("WISE_B200_DEVICES", raising=False)
    monkeypatch.delenv("WISE_B200_DEVICE", raising=False)
    monkeypatch.delenv("LOCAL_RANK", raising=False)
    assert resolve_devices() == [0]
    assert resolve_devices(device=3) == [3]
    monkeypatch.setenv("WISE_B200_DEVICES", "0, 1,2,3")
    assert resolve_devices() == [0, 1, 2, 3]
    assert resolve_devices([2, 5]) == [2, 5]
    assert resolve_devices(device=1) == [1]
    monkeypatch.setenv("WISE_B200_DEVICES", "")
    monkeypatch.setenv("WISE_B200_DEVICE", "2")
    assert resolve_devices() == [2]


class _FakeShard:
    """Stands in for one GPU's index: holds a row count; the memory rule must not be consulted under a reservation."""

    def __init__(self):
        self.ntotal = 0

    def reserve(self, n):
        pass

    @property
    def _h(self):
        raise AssertionError("the free-memory rule was consulted inside the reservation")


def _fake_group(world):
    from wise_b200 import faiss_compat as fc
    idx = fc.Index()
    idx.d = 8
    idx._shards = [_FakeShard() for _ in range(world)]
    return idx


def _add(idx, m):
    for s, _, c in idx._plan_add(m):
        idx._shards[s].ntotal += c


def test_reservation_holds_when_adds_end_exactly_on_shard_boundaries():
    # one add per equal-sized store file, as the pinned ingest makes them
    idx = _fake_group(2)
    idx.reserve(1_000_000)
    for _ in range(10):
        _add(idx, 100_000)
    assert [sh.ntotal for sh in idx._shards] == [500_000, 500_000]
    idx = _fake_group(4)
    idx.reserve(1 << 18)
    for _ in range(4):
        _add(idx, 1 << 16)
    assert [sh.ntotal for sh in idx._shards] == [1 << 16] * 4


def test_reservation_smaller_than_the_world_skips_empty_quotas():
    idx = _fake_group(8)
    idx.reserve(3)
    assert routing.quotas(3, 8) == [0, 0, 1, 0, 0, 1, 0, 1]
    _add(idx, 3)
    assert [sh.ntotal for sh in idx._shards] == [0, 0, 1, 0, 0, 1, 0, 1]
    idx = _fake_group(8)
    idx.reserve(3)
    for _ in range(3):
        _add(idx, 1)
    assert [sh.ntotal for sh in idx._shards] == [0, 0, 1, 0, 0, 1, 0, 1]


def test_shard_limits_switch_to_memory_only_past_the_reserved_total():
    room = lambda s: 10 ** 9
    assert routing.shard_limits([50, 50], [50, 50], room) == [10 ** 9] * 2
    assert routing.shard_limits([50, 0], [50, 50], room) == [50, 50]
    assert routing.shard_limits([0, 0], None, room) == [10 ** 9] * 2
