"""Pinned, overlapped FeatureStore -> HBM ingest (SURVEY.md 8f-1, K9).

Replaces the add loop of /root/reference/src/index/feature_search_index.py:78-82
(`for ids, X in feature_store.iter_batch(): index.add_with_ids(X, ids)`, one synchronous call per 512 rows after a
per-vector tar + pickle decode in python): whole shards are decoded by the C++ reader (csrc/tarstore.h) straight
into a ring of pinned host buffers on a helper thread, and every decoded shard is handed to
`wb_add_with_ids_pinned`, which only ENQUEUES the host->HBM copy and - for IndexIVFFlat - the coarse assignment on
the index's stream.  While the copy engine and the SMs work on shard i the helper thread decodes shard i+1; a
buffer is reused only after `wb_add_slot_wait` says the GPU has finished reading it.
"""
from __future__ import annotations

import ctypes as C
from concurrent.futures import ThreadPoolExecutor

import numpy as np

from . import _capi

RING = 3  # buffers: one being decoded into, one in flight to the GPU, one spare


class PinnedRing:
    """RING pinned (page-locked) host buffers of `rows` x (int64 id + d floats), as numpy views."""

    def __init__(self, rows: int, d: int, nbuf: int = RING, with_assign: bool = False):
        L = _capi.lib()
        self._ptrs = []
        self.ids, self.x, self.assign = [], [], []
        self.rows, self.d, self.nbuf = max(rows, 1), d, nbuf
        for _ in range(nbuf):
            if with_assign:
                p_a = C.c_void_p()
                _capi.check(L.wb_pinned_alloc(max(rows, 1) * 4, C.byref(p_a)))
                self._ptrs.append(p_a)
                self.assign.append(np.ctypeslib.as_array((C.c_int32 * max(rows, 1)).from_address(p_a.value)))
            p_ids, p_x = C.c_void_p(), C.c_void_p()
            _capi.check(L.wb_pinned_alloc(max(rows, 1) * 8, C.byref(p_ids)))
            self._ptrs.append(p_ids)
            _capi.check(L.wb_pinned_alloc(max(rows, 1) * d * 4, C.byref(p_x)))
            self._ptrs.append(p_x)
            self.ids.append(np.ctypeslib.as_array((C.c_int64 * max(rows, 1)).from_address(p_ids.value)))
            self.x.append(np.ctypeslib.as_array((C.c_float * (max(rows, 1) * d)).from_address(p_x.value)).reshape(max(rows, 1), d))

    def close(self):
        L = _capi.lib()
        self.ids, self.x, self.assign = [], [], []
        for p in self._ptrs:
            L.wb_pinned_free(p)
        self._ptrs = []

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def add_store_pipelined(index, store) -> int:
    """index.add_with_ids over every shard of an un-shuffled WebdatasetStore (already enable_read()),
    in shard order = the reference's insertion order.  Returns the number of rows added.
    Shards the C++ reader does not understand go through the python reader (synchronously, same order).

    Threads: the helper thread only decodes and calls wb_add_slot_wait (an event wait on a slot the main thread is not
    using); every call that changes the index (wb_add_with_ids_pinned, add_with_ids) is made by the calling thread, in
    shard order, and the future hand-off orders the two."""
    files = list(store.shard_files())
    rows_by = getattr(store, "_shard_rows", {})
    if not files:
        return 0
    cap = max([rows_by.get(fn, 0) for fn in files] + [1])
    d = store.feature_dim
    ring = PinnedRing(cap, d)
    added = 0

    def decode(i):
        slot = i % RING
        index._slot_wait(slot)  # the GPU has finished reading this buffer (two shards ago)
        return store.decode_shard_into(files[i], ring.ids[slot], ring.x[slot])

    try:
        with ThreadPoolExecutor(max_workers=1) as pool:
            fut = pool.submit(decode, 0)
            for i, fn in enumerate(files):
                n = fut.result()
                if i + 1 < len(files):
                    fut = pool.submit(decode, i + 1)
                slot = i % RING
                if n is None:  # foreign pickle dialect / irregular shard: python reader, ordinary synchronous add
                    ids, x = store._python_shard(fn)
                    if len(ids):
                        index.add_with_ids(np.ascontiguousarray(x, np.float32), np.ascontiguousarray(ids, np.int64))
                    added += len(ids)
                    continue
                if n:  # (a multi-GPU index splits the shard at its shard boundaries)
                    index._add_pinned(n, ring.x[slot], ring.ids[slot], slot)
                added += n
        index._sync()
    finally:
        index._sync(check=False)
        ring.close()
    return added
