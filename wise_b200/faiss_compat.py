"""The subset of the `faiss` Python API that WISE touches, served by libwiseb200.so on a B200.

Drop-in for `import faiss` in /root/reference/src/index/feature_search_index.py:1 (see
INTEGRATION.md).  Mirrored surface (SURVEY.md section 8b):

  module : IndexFlatIP(d) | IndexIDMap(index) | IndexIVFFlat(quantizer, d, nlist, metric)
           METRIC_INNER_PRODUCT | IO_FLAG_READ_ONLY | write_index | read_index
  index  : .d .ntotal .is_trained .train .add .add_with_ids .search(x, k, params=None)
           .range_search(x, thresh, params=None) -> lims (uint64, n+1), D, I
  search : SearchParameters(sel) | SearchParametersIVF(sel, nprobe)
           IDSelectorBatch | IDSelectorRange | IDSelectorNot (filtered search, faiss >= 1.7.3)
           IVF only: .nprobe .parallel_mode .make_direct_map .direct_map .reconstruct_batch
           (Flat/IDMap deliberately have no `nprobe`/`direct_map`: /root/reference/api/routes.py:899
            and :1317 branch on hasattr())

Arrays in, arrays out: inputs are borrowed numpy arrays (float32 C-contiguous, like faiss's
SWIG wrappers require), outputs are fresh numpy arrays; errors are RuntimeError like faiss.
All arithmetic runs in hand-written sm_100a kernels; there is no CPU path in this module.
"""
from __future__ import annotations

import ctypes as C
import os
import sys

import numpy as np

from . import _capi, routing

METRIC_INNER_PRODUCT = 0
METRIC_L2 = 1
IO_FLAG_MMAP = 1
IO_FLAG_READ_ONLY = 2

_MAX_POINTS_PER_CENTROID = 256  # faiss ClusteringParameters defaults [faiss-upstream]
_MIN_POINTS_PER_CENTROID = 39
_KMEANS_NITER_IVF = 10
_KMEANS_SEED = 1234


def default_device() -> int:
    """GPU of this process: WISE_B200_DEVICE, else LOCAL_RANK (one process per GPU), else 0."""
    for var in ("WISE_B200_DEVICE", "LOCAL_RANK"):
        v = os.environ.get(var)
        if v not in (None, ""):
            return int(v)
    return 0


def resolve_devices(devices=None, device: int | None = None) -> list[int]:
    """GPUs of a new index: `devices`, else [device], else WISE_B200_DEVICES (a comma-separated list such as
    "0,1,2,3": one index over those GPUs of this process), else [default_device()]."""
    if devices is None and device is not None:
        devices = [device]
    if devices is None:
        v = os.environ.get("WISE_B200_DEVICES", "").strip()
        devices = [int(t) for t in v.split(",") if t.strip()] if v else [default_device()]
    devices = [int(g) for g in devices]
    if not devices:
        raise RuntimeError("an index needs at least one device")
    return devices


def _as_f32_matrix(x, d: int, what: str) -> np.ndarray:
    x = np.asarray(x)
    if x.dtype != np.float32:
        raise TypeError(f"{what} must be float32 (got {x.dtype})")  # faiss: "input not a numpy array of float32"
    if x.ndim != 2 or x.shape[1] != d:
        raise AssertionError(f"{what} must have shape (n, {d}), got {x.shape}")  # faiss asserts d == self.d
    return np.ascontiguousarray(x)


def _as_ids(ids, n: int) -> np.ndarray:
    ids = np.ascontiguousarray(np.asarray(ids), dtype=np.int64)
    if ids.shape != (n,):
        raise AssertionError(f"ids must have shape ({n},), got {ids.shape}")  # faiss: 'not same nb of vectors as ids'
    return ids


class _Handle:
    """Owns one wb_index*."""

    def __init__(self, h):
        self.h = h

    def __del__(self):
        h, self.h = getattr(self, "h", None), None
        if h:
            try:
                _capi.lib().wb_free(h)
            except Exception:  # interpreter shutdown
                pass


class _Group:
    """Owns one wb_group* over the handles of `shards` (kept alive here, so the group is freed before them)."""

    MAX_QUERIES = 4096  # exchange mailbox: larger searches merge on the root instead (the sizes of PeerExchange)
    MAX_ENTRIES = 1 << 20

    def __init__(self, shards, max_queries: int = MAX_QUERIES, max_entries: int = MAX_ENTRIES):
        self.hds = [sh._hd for sh in shards]
        arr = (C.c_void_p * len(shards))(*[hd.h.value for hd in self.hds])
        g = C.c_void_p()
        _capi.check(_capi.lib().wb_group_create(len(shards), arr, int(max_queries), int(max_entries), C.byref(g)))
        self.g = g

    def __del__(self):
        g, self.g = getattr(self, "g", None), None
        if g:
            try:
                _capi.lib().wb_group_free(g)
            except Exception:  # interpreter shutdown
                pass


class Index:
    """Common behaviour of the faiss index classes WISE constructs.

    An index over several GPUs (devices=[g0, g1, ...] or WISE_B200_DEVICES) keeps one single-GPU index per device in
    `_shards` (shard s holds the s-th contiguous range of insertion positions, see routing.py) and searches them as one
    through a wb_group; it behaves exactly like one index holding all the rows in insertion order."""

    metric_type = METRIC_INNER_PRODUCT

    def __init__(self):
        self._hd: _Handle | None = None
        self.d = 0
        self._shards: list | None = None  # multi-GPU: one single-GPU index per device
        self._grp: _Group | None = None
        self._quota: list[int] | None = None  # rows of each shard after reserve()

    # -- properties ---------------------------------------------------------------------------
    @property
    def _h(self):
        if self._shards is not None:
            raise RuntimeError("a multi-GPU index has one handle per shard (index._shards)")
        return self._hd.h

    @property
    def ntotal(self) -> int:
        if self._shards is not None:
            return sum(sh.ntotal for sh in self._shards)
        return int(_capi.lib().wb_ntotal(self._h))

    @property
    def is_trained(self) -> bool:
        if self._shards is not None:
            return self._shards[0].is_trained
        return bool(_capi.lib().wb_is_trained(self._h))

    def _make_shards(self, devices: list[int], create) -> None:
        """One device: this object is the index (`create(device)` returns its handle).  Several: one shard per device
        and the group over them."""
        if len(devices) == 1:
            self._device = devices[0]
            self._hd = _Handle(create(devices[0]))
            return
        if len(set(devices)) != len(devices):
            raise RuntimeError(f"each GPU can hold one shard of an index (devices {devices})")
        self._device = devices[0]
        self._shards = []
        for g in devices:
            sh = _Shard(self.d)
            sh._device = g
            sh._hd = _Handle(create(g))
            self._shards.append(sh)

    def _group(self) -> _Group:
        """The wb_group over the shards, built by the first search (an index that is never searched, such as the
        quantizer of a multi-GPU IndexIVFFlat, allocates no exchange mailboxes)."""
        if self._grp is None:
            self._grp = _Group(self._shards)
        return self._grp

    def _regroup(self) -> None:
        """Drop the group after the IVF centroids changed: the next search builds one over the new centroids (the group
        checks that they are equal on every shard)."""
        self._grp = None

    @property
    def devices(self) -> list[int]:
        return [sh._device for sh in self._shards] if self._shards is not None else [self._device]

    # -- build ----------------------------------------------------------------------------------
    def reserve(self, n: int) -> None:
        """Pre-size HBM for n rows (not in faiss; optional, avoids re-allocation while adding).  A multi-GPU index
        also sets the shards' quotas to the balanced split of n (routing.quotas); without a reservation, rows fill one
        GPU after the other."""
        if self._shards is None:
            _capi.check(_capi.lib().wb_reserve(self._h, int(n)))
            return
        self._quota = routing.quotas(int(n), len(self._shards))
        for sh, q in zip(self._shards, self._quota):
            sh.reserve(q)

    def _plan_add(self, m: int) -> list[tuple[int, int, int]]:
        """(shard, first row, rows) pieces of an add of m rows to a multi-GPU index (routing.plan_add with the limits of
        routing.shard_limits)."""
        row_bytes = ((self.d + 3) & ~3) * 4 + 8 + (4 if isinstance(self, IndexIVFFlat) else 0)
        counts = [sh.ntotal for sh in self._shards]

        def room(s):
            cap, free = C.c_int64(0), C.c_int64(0)
            _capi.check(_capi.lib().wb_capacity(self._shards[s]._h, C.byref(cap), C.byref(free)))
            return routing.rows_that_fit(counts[s], cap.value, free.value, row_bytes)

        return routing.plan_add(m, counts, routing.shard_limits(counts, self._quota, room))

    def _add_pinned(self, m: int, x, ids, slot: int, assign=None, pos_buf=None) -> None:
        """Enqueue the add of m rows held in pinned buffers (x [m, d], ids [m] or None: ids = insertion positions,
        assign [m] for rows whose IVF list is known).  A multi-GPU index splits the batch at shard boundaries and,
        without ids, writes the global positions into the pinned `pos_buf`."""
        L = _capi.lib()
        if self._shards is None:
            if assign is not None:
                _capi.check(L.wb_ivf_add_preassigned_pinned(self._h, m, _capi.ptr(x), _capi.ptr(ids), _capi.ptr(assign),
                                                            slot))
            else:
                _capi.check(L.wb_add_with_ids_pinned(self._h, m, _capi.ptr(x), _capi.ptr(ids), slot))
            return
        if ids is None:
            pos_buf[:m] = np.arange(self.ntotal, self.ntotal + m, dtype=np.int64)
            ids = pos_buf
        for s, a, c in self._plan_add(m):
            sh = self._shards[s]
            if assign is not None:
                _capi.check(L.wb_ivf_add_preassigned_pinned(sh._h, c, _capi.ptr(x[a:a + c]), _capi.ptr(ids[a:a + c]),
                                                            _capi.ptr(assign[a:a + c]), slot))
            else:
                _capi.check(L.wb_add_with_ids_pinned(sh._h, c, _capi.ptr(x[a:a + c]), _capi.ptr(ids[a:a + c]), slot))

    def _slot_wait(self, slot: int) -> None:
        """wb_add_slot_wait on every shard: the GPUs have finished reading pinned buffer `slot`."""
        for sh in (self._shards or [self]):
            _capi.check(_capi.lib().wb_add_slot_wait(sh._hd.h, slot))

    def _sync(self, check: bool = True) -> None:
        for sh in (self._shards or [self]):
            rc = _capi.lib().wb_sync(sh._hd.h)
            if check:
                _capi.check(rc)

    def train(self, x) -> None:  # IndexFlat / IndexIDMap: nothing to train (faiss: no-op)
        _as_f32_matrix(x, self.d, "x")

    def _add(self, x, ids) -> None:
        x = _as_f32_matrix(x, self.d, "x")
        n = x.shape[0]
        if self._shards is not None:
            # rows without ids get their global insertion position as id
            ids = np.arange(self.ntotal, self.ntotal + n, dtype=np.int64) if ids is None else _as_ids(ids, n)
            for s, a, c in self._plan_add(n):
                self._shards[s]._add(x[a:a + c], ids[a:a + c])
            return
        idp = None
        if ids is not None:
            ids = _as_ids(ids, n)
            idp = _capi.ptr(ids)
        _capi.check(_capi.lib().wb_add_with_ids(self._h, n, _capi.ptr(x), idp))

    def add(self, x) -> None:
        self._add(x, None)

    def add_with_ids(self, x, ids) -> None:
        self._add(x, ids)

    # -- search ---------------------------------------------------------------------------------
    def _nprobe(self) -> int:
        return 1

    def _search_params(self, params):
        """(nprobe, wb_filter* or None) of a search with faiss SearchParameters `params` (None: the index's own).
        A multi-GPU index gets a list with one wb_filter* per shard, all built from the same selector."""
        if params is None:
            return self._nprobe(), None
        if not isinstance(params, SearchParameters):
            raise TypeError("params must be a SearchParameters")
        if params.sel is None:
            return self._nprobe(), None
        if self._shards is not None:
            return self._nprobe(), [params.sel._filter(sh._hd) for sh in self._shards]
        return self._nprobe(), params.sel._filter(self._hd)

    def search(self, x, k: int, *, params=None):
        """D, I = index.search(x, k)  (/root/reference/src/index/feature_search_index.py:113,
        /root/reference/api/routes.py:1407): D float32 (n,k) descending, I int64 (n,k), -1 padded.
        params=SearchParameters(sel=...) restricts the result to the rows whose id the selector keeps (exact top-k
        of those rows; IVF takes SearchParametersIVF, whose nprobe replaces index.nprobe for this call)."""
        x = _as_f32_matrix(x, self.d, "x")
        k = int(k)
        if k <= 0:
            raise AssertionError("k must be positive")  # faiss: assert k > 0
        nprobe, flt = self._search_params(params)
        n = x.shape[0]
        D = np.empty((n, k), np.float32)
        I = np.empty((n, k), np.int64)
        if n and self._shards is not None:
            fl = (C.c_void_p * len(flt))(*flt) if flt is not None else None
            _capi.check(_capi.lib().wb_group_search(self._group().g, fl, n, _capi.ptr(x), k, nprobe, _capi.ptr(D),
                                                    _capi.ptr(I)))
        elif n:
            L = _capi.lib()
            _capi.check(L.wb_search_filtered(self._h, flt, n, _capi.ptr(x), k, nprobe, _capi.ptr(D), _capi.ptr(I)))
        return D, I

    def range_search(self, x, thresh, *, params=None):
        """lims, D, I = index.range_search(x, thresh): every row whose inner product with a query is strictly greater
        than `thresh` (used as float32).  Query i's results are D[lims[i]:lims[i+1]] (float32, descending; equal scores
        by insertion order) and I[...] (int64).  lims is uint64 of length n+1, as faiss returns it; there is no cap on
        the number of results.  params as in search (IVF: the rows of the probed lists are the candidates)."""
        x = _as_f32_matrix(x, self.d, "x")
        thresh = np.float32(thresh)
        nprobe, flt = self._search_params(params)
        n = x.shape[0]
        if self._shards is not None:
            return self._group_range_search(x, float(thresh), nprobe, flt)
        lims = np.zeros((n + 1,), np.int64)
        L = _capi.lib()
        res = C.c_void_p()
        _capi.check(L.wb_range_search(self._h, flt, n, _capi.ptr(x) if n else None, float(thresh), nprobe,
                                      _capi.ptr(lims), C.byref(res)))
        try:
            total = int(lims[-1])
            D = np.empty((total,), np.float32)
            I = np.empty((total,), np.int64)
            _capi.check(L.wb_range_result_copy(res, _capi.ptr(D), _capi.ptr(I)))
        finally:
            L.wb_range_result_free(res)
        return lims.astype(np.uint64), D, I

    def _group_range_search(self, x: np.ndarray, thresh: float, nprobe: int, flt):
        """Range search of a multi-GPU index: every shard's wb_range_search_dev on a thread of its own (each call
        synchronises once per query chunk), the parts copied into the padded layout on the root GPU, and the exact merge
        there (wb_range_merge_dev) - the steps of ShardedIndex.range_search_dev without the collectives."""
        from concurrent.futures import ThreadPoolExecutor

        import torch

        from .sharded import _cuda_local_range_search, _cuda_range_merge
        world = len(self._shards)
        q = torch.from_numpy(x)
        flts = flt if flt is not None else [None] * world
        with ThreadPoolExecutor(max_workers=world) as pool:
            parts = list(pool.map(lambda s: _cuda_local_range_search(self._shards[s], q, thresh, nprobe, flts[s]),
                                  range(world)))
        root = torch.device("cuda", self._shards[0]._device)
        lims_parts = torch.stack([lims for lims, _, _ in parts])
        merged = lims_parts.sum(dim=0)
        stride = int(lims_parts[:, -1].max())
        if stride == 0:
            return merged.numpy().astype(np.uint64), np.empty((0,), np.float32), np.empty((0,), np.int64)
        Dp = torch.empty((world, stride), dtype=torch.float32, device=root)
        Ip = torch.empty((world, stride), dtype=torch.int64, device=root)
        for s, (lims, D, I) in enumerate(parts):
            torch.cuda.synchronize(D.device)  # the part was written on its GPU's stream by another thread
            m = int(lims[-1])
            Dp[s, :m] = D.to(root)
            Ip[s, :m] = I.to(root)
        del parts
        D, I = _cuda_range_merge(lims_parts, Dp, Ip, merged)
        return merged.numpy().astype(np.uint64), D.cpu().numpy(), I.cpu().numpy()

    # -- bulk access used by write_index --------------------------------------------------------
    def _export(self, start: int, n: int, want_assign: bool = False, want_ids: bool = True, want_x: bool = True):
        """Storage rows [start, start+n): insertion order for flat indices, list by list for a finalized IVF index."""
        x = np.empty((n, self.d), np.float32) if want_x else None
        ids = np.empty((n,), np.int64) if want_ids else None
        a = np.empty((n,), np.int32) if want_assign else None
        _capi.check(_capi.lib().wb_export_rows(self._h, start, n, _capi.ptr(x), _capi.ptr(ids), _capi.ptr(a)))
        return x, ids, a


class _Shard(Index):
    """One GPU's part of a multi-GPU index: a plain single-GPU handle (created by Index._make_shards)."""

    def __init__(self, d: int):
        super().__init__()
        self.d = d


class IndexFlatIP(Index):
    """faiss.IndexFlatIP(d)  (/root/reference/src/index/feature_search_index.py:47).  `devices` (a list of GPUs; default
    resolve_devices(): WISE_B200_DEVICES, else one GPU) puts the rows on several GPUs of this process."""

    def __init__(self, d: int, device: int | None = None, devices=None):
        super().__init__()
        self.d = int(d)

        def create(g):
            h = C.c_void_p()
            _capi.check(_capi.lib().wb_flat_create(self.d, g, C.byref(h)))
            return h

        self._make_shards(resolve_devices(devices, device), create)

    def add_with_ids(self, x, ids) -> None:
        # faiss: IndexFlat has no id storage - that is why the reference wraps it in IndexIDMap
        raise RuntimeError("add_with_ids not implemented for this type of index")

    def reconstruct_batch(self, keys):
        return _reconstruct(self, keys)


class IndexIDMap(Index):
    """faiss.IndexIDMap(index)  (/root/reference/src/index/feature_search_index.py:52).
    Shares the wrapped index's HBM row store; the id map lives beside the rows on the GPU."""

    def __init__(self, index: IndexFlatIP):
        super().__init__()
        if not isinstance(index, IndexFlatIP):
            raise TypeError("IndexIDMap wraps an IndexFlatIP")
        if index.ntotal != 0:
            raise RuntimeError("index must be empty on input")  # faiss IndexIDMap ctor
        self.index = index
        self.d = index.d
        self._hd = index._hd
        self._device = index._device
        self._shards = index._shards

    def _group(self):
        return self.index._group()  # one group per set of shards

    def add(self, x) -> None:
        raise RuntimeError("add does not make sense with IndexIDMap, use add_with_ids")


class DirectMap:
    """faiss.DirectMap: only .type and the NoMap/Array/Hashtable constants are read
    (/root/reference/api/routes.py:1317)."""

    NoMap, Array, Hashtable = 0, 1, 2

    def __init__(self):
        self.type = DirectMap.NoMap


class ClusteringParameters:
    """faiss.ClusteringParameters as IndexIVF.cp holds it [faiss-upstream defaults for IndexIVFFlat built with the
    plain constructor, /root/reference/src/index/feature_search_index.py:60]: niter 10 (Level1Quantizer), seed 1234,
    spherical False (only index_factory switches it on for inner-product indices), 39..256 points per centroid."""

    def __init__(self):
        self.niter = _KMEANS_NITER_IVF
        self.seed = _KMEANS_SEED
        self.spherical = False
        self.min_points_per_centroid = _MIN_POINTS_PER_CENTROID
        self.max_points_per_centroid = _MAX_POINTS_PER_CENTROID


class IndexIVFFlat(Index):
    """faiss.IndexIVFFlat(quantizer, d, nlist, METRIC_INNER_PRODUCT)
    (/root/reference/src/index/feature_search_index.py:60)."""

    def __init__(self, quantizer: IndexFlatIP, d: int, nlist: int, metric: int = METRIC_INNER_PRODUCT):
        super().__init__()
        if metric != METRIC_INNER_PRODUCT:
            raise RuntimeError("wise_b200 implements METRIC_INNER_PRODUCT only (the metric WISE uses)")
        if quantizer is not None and quantizer.d != d:
            raise AssertionError("quantizer dimension mismatch")
        self.d = int(d)
        self.nlist = int(nlist)
        self.nprobe = 1  # faiss default; the REST API raises it (api/routes.py:899-902), the CLI does not
        self.parallel_mode = 0  # accepted and ignored: the GPU always fans one query over all probed lists
        self.quantizer = quantizer
        self.direct_map = DirectMap()
        self.cp = ClusteringParameters()

        def create(g):
            h = C.c_void_p()
            _capi.check(_capi.lib().wb_ivf_create(self.d, self.nlist, g, C.byref(h)))
            return h

        # the index lives where its quantizer does
        self._make_shards(quantizer.devices if quantizer is not None else resolve_devices(), create)

    def _nprobe(self) -> int:
        return max(1, int(self.nprobe))

    def _search_params(self, params):
        if params is None:
            return self._nprobe(), None
        if not isinstance(params, SearchParametersIVF):
            raise RuntimeError("IndexIVF params have incorrect type")  # faiss IndexIVF::search
        _, flt = super()._search_params(params)
        return max(1, int(params.nprobe)), flt

    def train(self, x) -> None:
        """index.train(train_features) (/root/reference/src/index/feature_search_index.py:75): k-means with
        max-inner-product assignment, faiss Clustering defaults in self.cp (niter=10, seed=1234, spherical=False,
        at most 256 training points per centroid: a larger set is subsampled, a set below 39 per centroid warns)."""
        x = _as_f32_matrix(x, self.d, "x")
        if self.is_trained:
            return  # faiss: "IVF quantizer does not need training"
        n = x.shape[0]
        cp = self.cp
        if n > self.nlist * cp.max_points_per_centroid:  # faiss Clustering::train subsamples [faiss-upstream]
            keep = self.nlist * cp.max_points_per_centroid
            print(f"Sampling a subset of {keep} / {n} for training", file=sys.stderr)
            sel = np.random.RandomState(cp.seed).permutation(n)[:keep]
            x = np.ascontiguousarray(x[sel])
            n = keep
        elif n < self.nlist * cp.min_points_per_centroid:
            print(f"WARNING clustering {n} points to {self.nlist} centroids: please provide at least "
                  f"{self.nlist * cp.min_points_per_centroid} training points", file=sys.stderr)
        L = _capi.lib()
        # a multi-GPU index trains on its root shard and copies the centroids, bit for bit, to the others
        root = self._shards[0] if self._shards is not None else self
        _capi.check(L.wb_ivf_set_spherical(root._hd.h, int(bool(cp.spherical))))
        _capi.check(L.wb_ivf_train(root._hd.h, n, _capi.ptr(x), int(cp.niter), int(cp.seed)))
        if self._shards is not None:
            self._set_shard_centroids(self.centroids())
        self._sync_quantizer()

    def _set_shard_centroids(self, c: np.ndarray) -> None:
        L = _capi.lib()
        for sh in self._shards:
            _capi.check(L.wb_ivf_set_spherical(sh._h, int(bool(self.cp.spherical))))
            _capi.check(L.wb_ivf_set_centroids(sh._h, _capi.ptr(c)))
        self._regroup()

    def _sync_quantizer(self) -> None:
        """Keep the user-visible quantizer object in the state faiss leaves it in (holding the centroids)."""
        if self.quantizer is not None and self.quantizer.ntotal == 0:
            self.quantizer.add(self.centroids())

    def centroids(self) -> np.ndarray:
        c = np.empty((self.nlist, self.d), np.float32)
        root = self._shards[0] if self._shards is not None else self
        _capi.check(_capi.lib().wb_ivf_get_centroids(root._hd.h, _capi.ptr(c)))
        return c

    def set_centroids(self, c) -> None:
        """Install trained centroids (read_index, or 'the reference's own trained centroids')."""
        c = _as_f32_matrix(c, self.d, "centroids")
        if c.shape[0] != self.nlist:
            raise AssertionError(f"expected {self.nlist} centroids, got {c.shape[0]}")
        if self._shards is not None:
            self._set_shard_centroids(c)
        else:
            _capi.check(_capi.lib().wb_ivf_set_centroids(self._h, _capi.ptr(c)))
        self._sync_quantizer()

    def _add(self, x, ids) -> None:
        if self.direct_map.type == DirectMap.Array and ids is not None:
            raise RuntimeError("cannot have array direct map and add with ids")  # faiss DirectMapAdd
        super()._add(x, ids)

    def make_direct_map(self, new_maintain_direct_map: bool = True) -> None:
        """/root/reference/api/routes.py:907.  faiss's Array direct map exists only for ids 0..ntotal-1
        and throws otherwise (WISE ids start at 1, so the caller's except-branch is the usual path)."""
        if not new_maintain_direct_map:
            self.direct_map.type = DirectMap.NoMap
            return
        n = self.ntotal
        for sh in (self._shards or [self]):
            m = sh.ntotal
            for s in range(0, m, 1 << 20):
                _, ids, _ = sh._export(s, min(1 << 20, m - s), want_x=False)
                if ids.size and (ids.min() < 0 or ids.max() >= n):
                    raise RuntimeError("direct map supported only for seqential ids")  # (sic) faiss message
        self.direct_map.type = DirectMap.Array

    def reconstruct_batch(self, keys):
        """/root/reference/api/routes.py:1078."""
        if self.direct_map.type == DirectMap.NoMap:
            raise RuntimeError("direct map not initialized")
        return _reconstruct(self, keys)


class _Filter:
    """Owns one wb_filter*.  Holds the _Handle of its index, so the filter is freed before the index is."""

    def __init__(self, hd: _Handle, f):
        self.hd = hd
        self.f = f

    def __del__(self):
        f, self.f = getattr(self, "f", None), None
        if f:
            try:
                _capi.lib().wb_filter_free(f)
            except Exception:  # interpreter shutdown
                pass

    @property
    def count(self) -> int:
        """Rows selected when the filter was last evaluated."""
        return int(_capi.lib().wb_filter_count(self.f))


class IDSelector:
    """faiss.IDSelector: decides per external id whether a row takes part in a search.  The selectors here are
    evaluated on the GPU into one bitmap per index (kept while the selector lives, re-evaluated after adds)."""

    _invert = False

    def __init__(self):
        self._filters: dict[int, _Filter] = {}

    def _create(self, h, invert: bool, out) -> int:
        raise NotImplementedError

    def _filter(self, hd: _Handle):
        """This selector's wb_filter* for the index owning `hd`, created on first use."""
        f = self._filters.get(id(hd))
        if f is None:
            p = C.c_void_p()
            _capi.check(self._create(hd.h, self._invert, C.byref(p)))
            f = self._filters[id(hd)] = _Filter(hd, p)
        return f.f


class IDSelectorBatch(IDSelector):
    """faiss.IDSelectorBatch(ids) or (n, ids): the ids in a set (any order, duplicates allowed)."""

    def __init__(self, *args):
        super().__init__()
        if len(args) == 2:
            n, ids = int(args[0]), args[1]
            ids = np.asarray(ids).reshape(-1)[:n]
        elif len(args) == 1:
            ids = np.asarray(args[0]).reshape(-1)
        else:
            raise TypeError("IDSelectorBatch(ids) or IDSelectorBatch(n, ids)")
        if ids.size and ids.dtype.kind not in "iu":
            raise TypeError(f"ids must be integers (got {ids.dtype})")
        self.ids = np.unique(ids.astype(np.int64))  # sorted and unique: the device set is searched by bisection

    def _create(self, h, invert, out):
        return _capi.lib().wb_filter_create_ids(h, self.ids.size, _capi.ptr(self.ids), int(invert), out)


class IDSelectorRange(IDSelector):
    """faiss.IDSelectorRange(imin, imax): imin <= id < imax (empty when imin >= imax)."""

    def __init__(self, imin: int, imax: int):
        super().__init__()
        for v in (imin, imax):
            if not isinstance(v, (int, np.integer)) or isinstance(v, bool):
                raise TypeError(f"IDSelectorRange bounds must be integers (got {type(v).__name__})")
        self.imin, self.imax = int(imin), int(imax)

    def _create(self, h, invert, out):
        return _capi.lib().wb_filter_create_range(h, self.imin, self.imax, int(invert), out)


class IDSelectorNot(IDSelector):
    """faiss.IDSelectorNot(sel): the ids `sel` rejects.  `sel` is an IDSelectorBatch, IDSelectorRange or another
    IDSelectorNot (Not of Not keeps what the inner selector keeps)."""

    def __init__(self, sel: IDSelector):
        super().__init__()
        if not isinstance(sel, (IDSelectorBatch, IDSelectorRange, IDSelectorNot)):
            raise TypeError("IDSelectorNot takes an IDSelectorBatch, IDSelectorRange or IDSelectorNot")
        self.sel = sel
        self._base = sel._base if isinstance(sel, IDSelectorNot) else sel
        self._invert = not sel._invert

    def _create(self, h, invert, out):
        return self._base._create(h, invert, out)


class SearchParameters:
    """faiss.SearchParameters(sel=...): per-call search options of a flat index."""

    def __init__(self, sel: IDSelector | None = None):
        if sel is not None and not isinstance(sel, IDSelector):
            raise TypeError("sel must be an IDSelector")
        self.sel = sel


class SearchParametersIVF(SearchParameters):
    """faiss.SearchParametersIVF(sel=..., nprobe=...): an IVF index's per-call options; nprobe (default 1, as in
    faiss) replaces index.nprobe for the call."""

    def __init__(self, sel: IDSelector | None = None, nprobe: int = 1):
        super().__init__(sel)
        self.nprobe = int(nprobe)


def _reconstruct(index: Index, keys) -> np.ndarray:
    keys = np.ascontiguousarray(np.asarray(keys), dtype=np.int64).reshape(-1)
    out = np.empty((keys.shape[0], index.d), np.float32)
    if not keys.shape[0]:
        return out
    L = _capi.lib()
    if index._shards is None:
        _capi.check(L.wb_reconstruct_batch(index._h, keys.shape[0], _capi.ptr(keys), _capi.ptr(out)))
        return out
    # multi-GPU: each id is looked up in every shard and read from the one that holds it
    found = np.zeros(keys.shape[0], bool)
    pos = np.empty(keys.shape[0], np.int64)
    for sh in index._shards:
        _capi.check(L.wb_lookup_ids(sh._h, keys.shape[0], _capi.ptr(keys), _capi.ptr(pos)))
        mine = np.nonzero((pos >= 0) & ~found)[0]
        if mine.size:
            sub = np.ascontiguousarray(keys[mine])
            rows = np.empty((mine.size, index.d), np.float32)
            _capi.check(L.wb_reconstruct_batch(sh._h, mine.size, _capi.ptr(sub), _capi.ptr(rows)))
            out[mine] = rows
            found[mine] = True
    if not found.all():
        raise RuntimeError(f"reconstruct: id {int(keys[np.argmin(found)])} not found in the index")
    return out


def write_index(index: Index, fname: str) -> None:
    """faiss.write_index  (/root/reference/src/index/feature_search_index.py:84)."""
    from . import faiss_io
    faiss_io.write_index(index, fname)


def read_index(fname: str, io_flags: int = 0) -> Index:
    """faiss.read_index(fname, faiss.IO_FLAG_READ_ONLY)  (feature_search_index.py:96)."""
    from . import faiss_io
    return faiss_io.read_index(fname, io_flags)
