"""Reader / writer for the `.faiss` index files WISE keeps on disk
(`<index_dir>/<media_type>-<IndexType>.faiss`, /root/reference/src/index/feature_search_index.py:30-31,84,96).

Byte layout restated from upstream faiss `impl/index_write.cpp` / `index_read.cpp`
[faiss-upstream; no faiss build is available in this image to cross-check - SURVEY.md 8f-2]:

  header(idx)  = int32 d | int64 ntotal | int64 1<<20 | int64 1<<20 | uint8 is_trained | int32 metric_type
  IndexFlatIP  = "IxFI" header  uint64 nfloats  float32[nfloats]
  IndexIDMap   = "IxMp" header  <nested index>  uint64 n  int64[n]
  IndexIVFFlat = "IwFl" header  uint64 nlist  uint64 nprobe  <nested quantizer>
                 direct_map{uint8 type | uint64 n | int64[n]}
                 "ilar" uint64 nlist  uint64 code_size
                 ("full" uint64 nlist  uint64 sizes[nlist]  |  "sprs" uint64 2m  (list, size)[m])
                 then for every non-empty list: codes uint8[n*code_size]  ids int64[n]

Rows stream between the file and HBM in bounded chunks, so an index larger than host RAM
can be written or read.
"""
from __future__ import annotations

import os
import struct

import numpy as np

from . import _capi
from . import faiss_compat as fc

_CHUNK_ROWS = 1 << 16
_DUMMY = 1 << 20


def _hdr(f, d: int, ntotal: int, is_trained: bool, metric: int) -> None:
    f.write(struct.pack("<iqqqBi", d, ntotal, _DUMMY, _DUMMY, 1 if is_trained else 0, metric))


def _read_hdr(f):
    d, ntotal, _, _, trained, metric = struct.unpack("<iqqqBi", _need(f, 4 + 8 * 3 + 1 + 4))
    if metric > 1:
        _need(f, 4)  # metric_arg
    return d, ntotal, bool(trained), metric


def _need(f, n: int) -> bytes:
    b = f.read(n)
    if len(b) != n:
        raise RuntimeError(f"read error in index file: wanted {n} bytes, got {len(b)}")  # faiss READANDCHECK
    return b


def _read_array(f, count: int, dtype) -> np.ndarray:
    """`count` items of `dtype` read straight into a fresh array (no intermediate bytes object)."""
    a = np.empty(count, dtype)
    if count:
        got = f.readinto(memoryview(a).cast("B"))
        if got != a.nbytes:
            raise RuntimeError(f"read error in index file: wanted {a.nbytes} bytes, got {got}")
    return a


def _write_array(f, a: np.ndarray) -> None:
    a = np.ascontiguousarray(a)
    if a.size:
        f.write(memoryview(a).cast("B"))  # no .tobytes() copy of multi-GB blocks


def _write_flat(f, index, centroids: np.ndarray | None = None) -> None:
    """IxFI block for an IndexFlatIP (or for an IVF quantizer given its centroid table)."""
    f.write(b"IxFI")
    if centroids is not None:
        n, d = centroids.shape
        _hdr(f, d, n, True, fc.METRIC_INNER_PRODUCT)
        f.write(struct.pack("<Q", n * d))
        _write_array(f, np.ascontiguousarray(centroids, np.float32))
        return
    n, d = index.ntotal, index.d
    _hdr(f, d, n, True, fc.METRIC_INNER_PRODUCT)
    f.write(struct.pack("<Q", n * d))
    for sh in _parts(index):  # a multi-GPU index: the shards in order are the rows in insertion order
        _stream_rows_out(f, sh, 0, sh.ntotal)


def _parts(index) -> list:
    """The single-GPU indices that hold `index`'s rows, in insertion order."""
    return index._shards if index._shards is not None else [index]


def _stream_rows_out(f, index, start: int, n: int) -> None:
    """Storage rows [start, start+n) -> file: HBM -> pinned host buffer (one cudaMemcpy2D per chunk) while a helper
    thread writes the previous chunk, so the copy engine and the file system work at the same time (a 30 GB index
    took 23 s through fresh pageable arrays; the file write is what remains)."""
    from concurrent.futures import ThreadPoolExecutor
    from .ingest import PinnedRing
    if n <= 0:
        return
    L = _capi.lib()
    chunk = min(_CHUNK_ROWS, n)
    ring = PinnedRing(chunk, index.d, nbuf=2)
    try:
        with ThreadPoolExecutor(max_workers=1) as pool:
            pending = [None, None]
            for i, s0 in enumerate(range(start, start + n, chunk)):
                m = min(chunk, start + n - s0)
                b = i % 2
                if pending[b] is not None:
                    pending[b].result()  # the file write that last used this buffer
                _capi.check(L.wb_export_rows(index._h, s0, m, _capi.ptr(ring.x[b]), None, None))
                pending[b] = pool.submit(f.write, memoryview(ring.x[b][:m]).cast("B"))
            for p_ in pending:
                if p_ is not None:
                    p_.result()
    finally:
        ring.close()


def write_index(index, fname: str) -> None:
    tmp = f"{fname}.tmp.{os.getpid()}"
    with open(tmp, "wb") as f:
        if isinstance(index, fc.IndexIDMap):
            n = index.ntotal
            f.write(b"IxMp")
            _hdr(f, index.d, n, True, fc.METRIC_INNER_PRODUCT)
            _write_flat(f, index)
            f.write(struct.pack("<Q", n))
            for sh in _parts(index):
                m = sh.ntotal
                for s in range(0, m, _CHUNK_ROWS):
                    _, ids, _ = sh._export(s, min(_CHUNK_ROWS, m - s), want_x=False)
                    _write_array(f, ids)
        elif isinstance(index, fc.IndexFlatIP):
            _write_flat(f, index)
        elif isinstance(index, fc.IndexIVFFlat):
            _write_ivf(f, index)
        else:
            raise RuntimeError(f"don't know how to serialize this type of index: {type(index).__name__}")
    os.replace(tmp, fname)  # atomic: an index file either exists completely or not at all


def _write_ivf(f, index) -> None:
    n, d, nlist = index.ntotal, index.d, index.nlist
    parts = [sh for sh in _parts(index) if sh.ntotal]
    if n and index.is_trained:
        # group the row store list by list first (K8 on the device): every inverted list is then ONE contiguous run of
        # storage rows and is exported with one copy per chunk.  Without it (train, add, write - no search in between,
        # which is exactly /root/reference/src/index/feature_search_index.py:75-84) the rows are still in insertion order
        # and a list would be gathered row by row.
        for sh in parts:
            _capi.check(_capi.lib().wb_ivf_finalize(sh._hd.h))
    f.write(b"IwFl")
    _hdr(f, d, n, index.is_trained, fc.METRIC_INNER_PRODUCT)
    f.write(struct.pack("<QQ", nlist, int(index.nprobe)))
    _write_flat(f, None, index.centroids() if index.is_trained else np.zeros((0, d), np.float32))
    # direct map: only the type byte and an (empty or sequential) array
    dm_type = index.direct_map.type
    f.write(struct.pack("<B", dm_type))
    # list membership, per part: a list of a multi-GPU index is its rows of every shard in shard order, which is its
    # rows in insertion order
    members = []  # (part, ids, assign, order, sizes)
    for sh in parts:
        m_all = sh.ntotal
        assign = np.empty((m_all,), np.int32)
        ids = np.empty((m_all,), np.int64)
        for s in range(0, m_all, 1 << 20):
            m = min(1 << 20, m_all - s)
            _capi.check(_capi.lib().wb_export_rows(sh._hd.h, s, m, None, _capi.ptr(ids[s:s + m]),
                                                   _capi.ptr(assign[s:s + m])))
        order = np.argsort(assign, kind="stable")  # CSR: rows of each list in insertion order
        members.append((sh, ids, assign, order, np.bincount(assign, minlength=nlist).astype(np.uint64)))
    sizes = np.zeros(nlist, np.uint64)
    for *_, sz in members:
        sizes += sz
    if dm_type == fc.DirectMap.Array:
        # lo_build(list, offset) = list << 32 | offset, indexed by id (ids are 0..n-1 here)
        arr = np.full(n, -1, np.int64)
        before = np.zeros(nlist, np.int64)  # rows of each list in the earlier parts
        for _, ids, assign, order, sz in members:
            m_all = ids.shape[0]
            off_in_list = np.empty(m_all, np.int64)
            starts = np.concatenate([[0], np.cumsum(sz)[:-1]]).astype(np.int64)
            off_in_list[order] = np.arange(m_all, dtype=np.int64) - starts[assign[order]]
            arr[ids] = (assign.astype(np.int64) << 32) | (off_in_list + before[assign])
            before += sz.astype(np.int64)
        f.write(struct.pack("<Q", n))
        f.write(arr.tobytes())
    else:
        f.write(struct.pack("<Q", 0))
    f.write(b"ilar")
    f.write(struct.pack("<QQ", nlist, d * 4))
    non0 = int((sizes > 0).sum())
    if non0 > nlist // 2:
        f.write(b"full")
        f.write(struct.pack("<Q", nlist))
        f.write(sizes.tobytes())
    else:
        f.write(b"sprs")
        nz = np.nonzero(sizes)[0].astype(np.uint64)
        pairs = np.stack([nz, sizes[nz]], axis=1).reshape(-1)
        f.write(struct.pack("<Q", pairs.size))
        f.write(pairs.tobytes())
    pos = [0] * len(members)
    for l in range(nlist):
        if int(sizes[l]) == 0:
            continue
        runs = []
        for j, (sh, ids, _, order, sz) in enumerate(members):
            m = int(sz[l])
            runs.append((sh, ids, order[pos[j]:pos[j] + m]))
            pos[j] += m
        for sh, _, rows in runs:
            m = rows.shape[0]
            if m > 4096 and rows[-1] - rows[0] == m - 1:  # one long contiguous run (a finalized store): pinned streaming
                _stream_rows_out(f, sh, int(rows[0]), m)
            else:
                for s in range(0, m, _CHUNK_ROWS):
                    _write_array(f, _gather_rows(sh, rows[s:s + _CHUNK_ROWS]))
        for _, ids, rows in runs:
            _write_array(f, ids[rows])


def _gather_rows(index, rows: np.ndarray) -> np.ndarray:
    """Rows by insertion position (contiguous runs are exported in one call)."""
    out = np.empty((rows.size, index.d), np.float32)
    if rows.size == 0:
        return out
    breaks = np.nonzero(np.diff(rows) != 1)[0] + 1
    starts = np.concatenate([[0], breaks])
    ends = np.concatenate([breaks, [rows.size]])
    for s, e in zip(starts, ends):
        x, _, _ = index._export(int(rows[s]), int(e - s), want_ids=False)
        out[s:e] = x
    return out


# ------------------------------------------------------------------------------------------------
def read_index(fname: str, io_flags: int = 0):
    try:
        f = open(fname, "rb")
    except OSError as e:  # faiss raises RuntimeError from its FileIOReader
        raise RuntimeError(f"could not open {fname} for reading: {e.strerror}") from e
    with f:
        return _read_any(f)


def _read_flat_body(f, add_rows) -> tuple[int, int]:
    d, ntotal, _, metric = _read_hdr(f)
    if metric != fc.METRIC_INNER_PRODUCT:
        raise RuntimeError("wise_b200 reads METRIC_INNER_PRODUCT indices only")
    (nfl,) = struct.unpack("<Q", _need(f, 8))
    if nfl != ntotal * d:
        raise RuntimeError(f"corrupt IndexFlat block: {nfl} floats for {ntotal} x {d}")
    add_rows(d, ntotal)
    return d, ntotal


def _readinto(f, a: np.ndarray) -> None:
    if a.size:
        got = f.readinto(memoryview(a).cast("B"))
        if got != a.nbytes:
            raise RuntimeError(f"read error in index file: wanted {a.nbytes} bytes, got {got}")


def _stream_rows_in(f, index, d: int, n: int, rows_at: int, ids_at: int | None) -> None:
    """File -> pinned ring -> HBM: the file read of chunk i+1 overlaps the host->device copy of chunk i
    (wb_add_with_ids_pinned only enqueues).  ids_at None: rows get their position as id (IndexFlatIP.add)."""
    from .ingest import PinnedRing, RING
    if n <= 0:
        return
    L = _capi.lib()
    chunk = min(_CHUNK_ROWS, n)
    ring = PinnedRing(chunk, d)
    try:
        for i, s0 in enumerate(range(0, n, chunk)):
            m = min(chunk, n - s0)
            slot = i % RING
            index._slot_wait(slot)
            f.seek(rows_at + s0 * d * 4)
            _readinto(f, ring.x[slot][:m])
            if ids_at is not None:
                f.seek(ids_at + s0 * 8)
                _readinto(f, ring.ids[slot][:m])
            index._add_pinned(m, ring.x[slot], ring.ids[slot] if ids_at is not None else None, slot,
                              pos_buf=ring.ids[slot])
        index._sync()
    finally:
        index._sync(check=False)
        ring.close()


def _read_any(f):
    tag = _need(f, 4)
    if tag == b"IxFI":
        box = {}

        def add_rows(d, n):
            idx = fc.IndexFlatIP(d)
            idx.reserve(n)
            at = f.tell()
            _stream_rows_in(f, idx, d, n, at, None)
            f.seek(at + n * d * 4)
            box["i"] = idx

        _read_flat_body(f, add_rows)
        return box["i"]
    if tag == b"IxMp":
        d, ntotal, _, _ = _read_hdr(f)
        sub = _need(f, 4)
        if sub != b"IxFI":
            raise RuntimeError(f"IndexIDMap over {sub!r} is not supported (WISE wraps IndexFlatIP)")
        # rows come before ids in the file: stage rows with provisional ids, then rewrite the ids
        flat = fc.IndexFlatIP(d)
        idmap = fc.IndexIDMap(flat)
        hdr_d, n, _, _ = _read_hdr(f)
        (nfl,) = struct.unpack("<Q", _need(f, 8))
        if hdr_d != d or nfl != n * d:
            raise RuntimeError("corrupt IndexIDMap block")
        rows_at = f.tell()
        f.seek(rows_at + n * d * 4)
        (nid,) = struct.unpack("<Q", _need(f, 8))
        if nid != n:
            raise RuntimeError("corrupt IndexIDMap block: id_map size mismatch")
        ids_at = f.tell()
        idmap.reserve(n)
        _stream_rows_in(f, idmap, d, n, rows_at, ids_at)
        f.seek(ids_at + n * 8)
        return idmap
    if tag == b"IwFl":
        return _read_ivf(f)
    raise RuntimeError(f"Index type {tag!r} not recognized")  # faiss message shape


def _read_ivf_lists(f, index, d: int, sizes: np.ndarray) -> None:
    """Inverted lists -> pinned ring -> HBM.  A file stores list after list (codes, then ids); several lists are packed
    into one pinned buffer together with their list number and handed to wb_ivf_add_preassigned_pinned, which only
    enqueues - a build with tens of thousands of short lists no longer pays one synchronous call per list."""
    from .ingest import PinnedRing, RING
    total = int(sizes.sum())
    if total == 0:
        return
    cap = min(max(_CHUNK_ROWS, int(sizes.max())), max(total, 1))
    ring = PinnedRing(cap, d, with_assign=True)
    state = {"i": 0, "fill": 0}

    def flush():
        slot = state["i"] % RING
        if state["fill"]:
            index._add_pinned(state["fill"], ring.x[slot], ring.ids[slot], slot, assign=ring.assign[slot])
        state["i"] += 1
        state["fill"] = 0
        index._slot_wait(state["i"] % RING)

    try:
        for l in range(sizes.shape[0]):
            m = int(sizes[l])
            if m == 0:
                continue
            if state["fill"] + m > cap:
                flush()
            slot, o = state["i"] % RING, state["fill"]
            _readinto(f, ring.x[slot][o:o + m])
            _readinto(f, ring.ids[slot][o:o + m])
            ring.assign[slot][o:o + m] = l
            state["fill"] = o + m
        flush()
        index._sync()
    finally:
        index._sync(check=False)
        ring.close()


def _read_ivf(f):
    d, ntotal, trained, metric = _read_hdr(f)
    if metric != fc.METRIC_INNER_PRODUCT:
        raise RuntimeError("wise_b200 reads METRIC_INNER_PRODUCT indices only")
    nlist, nprobe = struct.unpack("<QQ", _need(f, 16))
    qtag = _need(f, 4)
    if qtag != b"IxFI":
        raise RuntimeError(f"IVF quantizer {qtag!r} is not supported (WISE uses IndexFlatIP)")
    qd, qn, _, _ = _read_hdr(f)
    (nfl,) = struct.unpack("<Q", _need(f, 8))
    cent = np.frombuffer(_need(f, nfl * 4), np.float32).reshape(qn, qd) if nfl else np.zeros((0, d), np.float32)
    quant = fc.IndexFlatIP(d)
    index = fc.IndexIVFFlat(quant, d, int(nlist), fc.METRIC_INNER_PRODUCT)
    index.nprobe = int(nprobe)
    if trained:
        if qn != nlist:
            raise RuntimeError("corrupt IVF block: quantizer size != nlist")
        index.set_centroids(cent.copy())
    (dm_type,) = struct.unpack("<B", _need(f, 1))
    (dm_n,) = struct.unpack("<Q", _need(f, 8))
    f.seek(dm_n * 8, os.SEEK_CUR)
    if dm_type == fc.DirectMap.Hashtable:
        (hn,) = struct.unpack("<Q", _need(f, 8))
        f.seek(hn * 16, os.SEEK_CUR)
    if _need(f, 4) != b"ilar":
        raise RuntimeError("only ArrayInvertedLists ('ilar') are supported")
    il_nlist, code_size = struct.unpack("<QQ", _need(f, 16))
    if il_nlist != nlist or code_size != d * 4:
        raise RuntimeError("corrupt inverted lists header")
    ltype = _need(f, 4)
    (nsz,) = struct.unpack("<Q", _need(f, 8))
    raw = np.frombuffer(_need(f, nsz * 8), np.uint64)
    sizes = np.zeros(nlist, np.int64)
    if ltype == b"full":
        sizes[:] = raw.astype(np.int64)
    elif ltype == b"sprs":
        sizes[raw[0::2].astype(np.int64)] = raw[1::2].astype(np.int64)
    else:
        raise RuntimeError(f"unknown inverted list encoding {ltype!r}")
    index.reserve(int(sizes.sum()))
    _read_ivf_lists(f, index, d, sizes)
    if dm_type == fc.DirectMap.Array:
        index.direct_map.type = fc.DirectMap.Array
    return index
