"""Row routing of a multi-GPU index: which shard receives which rows of an add.

Shard s holds the s-th contiguous range of insertion positions, so rows always go to the last shard that holds any,
and to the next one only when that shard is full.  A shard is full at its quota (reserve(n): shard_range(n, s, world))
or, without a reservation, when its GPU's memory is used up; the last shard takes whatever is left.  Pure arithmetic:
no GPU, no torch.
"""
from __future__ import annotations

_MEM_RESERVE = 1 << 30  # free memory a shard leaves for search scratch (the int8 image keeps the same margin)


def shard_range(n_total: int, rank: int, world: int) -> tuple[int, int]:
    """Contiguous row range [lo, hi) of `rank` (balanced to within one row)."""
    return n_total * rank // world, n_total * (rank + 1) // world


def quotas(n_total: int, world: int) -> list[int]:
    """Rows of each shard after reserve(n_total)."""
    return [hi - lo for lo, hi in (shard_range(n_total, s, world) for s in range(world))]


def rows_that_fit(count: int, cap: int, free_bytes: int, row_bytes: int) -> int:
    """Largest row count a shard holding `count` rows in a store of `cap` rows can reach before its GPU is full.  A
    growth allocates max(need, 1.5 * cap) rows while the old store still exists, so it fits only when that many rows
    fit in the free memory (less the scratch margin)."""
    fit = max(0, free_bytes - _MEM_RESERVE) // row_bytes
    grown = max(cap + cap // 2, 1024)
    return max(count, cap, fit if fit >= grown else cap)


def shard_limits(counts: list[int], quota: list[int] | None, room) -> list[int | None]:
    """Rows each shard may hold for the next add.  While a reservation is not used up (sum(counts) < sum(quota)), a
    shard is full at its quota - also when an add ended exactly on its boundary, and when its quota is 0 (n < world).
    Past the reserved total, or without a reservation, a shard is full at `room(s)`, the rows that fit on its GPU."""
    if quota is not None and sum(counts) < sum(quota):
        return list(quota)
    return [room(s) for s in range(len(counts))]


def plan_add(m: int, counts: list[int], limits: list[int | None]) -> list[tuple[int, int, int]]:
    """Split an add of `m` rows into (shard, first row of the batch, row count) pieces.  counts[s]: rows shard s holds;
    limits[s]: rows it may hold (None: no limit).  The last shard has no limit."""
    world = len(counts)
    s = max([i for i in range(world) if counts[i] > 0], default=0)
    out, off = [], 0
    while off < m:
        room = m - off if s == world - 1 or limits[s] is None else max(0, limits[s] - counts[s])
        take = min(room, m - off)
        if take:
            out.append((s, off, take))
            off += take
        if off < m:
            s += 1
    return out
