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

from . import _capi

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


class Index:
    """Common behaviour of the faiss index classes WISE constructs."""

    metric_type = METRIC_INNER_PRODUCT

    def __init__(self):
        self._hd: _Handle | None = None
        self.d = 0

    # -- properties ---------------------------------------------------------------------------
    @property
    def _h(self):
        return self._hd.h

    @property
    def ntotal(self) -> int:
        return int(_capi.lib().wb_ntotal(self._h))

    @property
    def is_trained(self) -> bool:
        return bool(_capi.lib().wb_is_trained(self._h))

    # -- build ----------------------------------------------------------------------------------
    def reserve(self, n: int) -> None:
        """Pre-size HBM for n rows (not in faiss; optional, avoids re-allocation while adding)."""
        _capi.check(_capi.lib().wb_reserve(self._h, int(n)))

    def train(self, x) -> None:  # IndexFlat / IndexIDMap: nothing to train (faiss: no-op)
        _as_f32_matrix(x, self.d, "x")

    def _add(self, x, ids) -> None:
        x = _as_f32_matrix(x, self.d, "x")
        n = x.shape[0]
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
        """(nprobe, wb_filter* or None) of a search with faiss SearchParameters `params` (None: the index's own)."""
        if params is None:
            return self._nprobe(), None
        if not isinstance(params, SearchParameters):
            raise TypeError("params must be a SearchParameters")
        return self._nprobe(), (params.sel._filter(self._hd) if params.sel is not None else None)

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
        if n:
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

    # -- bulk access used by write_index --------------------------------------------------------
    def _export(self, start: int, n: int, want_assign: bool = False, want_ids: bool = True, want_x: bool = True):
        """Storage rows [start, start+n): insertion order for flat indices, list by list for a finalized IVF index."""
        x = np.empty((n, self.d), np.float32) if want_x else None
        ids = np.empty((n,), np.int64) if want_ids else None
        a = np.empty((n,), np.int32) if want_assign else None
        _capi.check(_capi.lib().wb_export_rows(self._h, start, n, _capi.ptr(x), _capi.ptr(ids), _capi.ptr(a)))
        return x, ids, a


class IndexFlatIP(Index):
    """faiss.IndexFlatIP(d)  (/root/reference/src/index/feature_search_index.py:47)."""

    def __init__(self, d: int, device: int | None = None):
        super().__init__()
        self.d = int(d)
        self._device = default_device() if device is None else int(device)
        h = C.c_void_p()
        _capi.check(_capi.lib().wb_flat_create(self.d, self._device, C.byref(h)))
        self._hd = _Handle(h)

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
        self._device = quantizer._device if quantizer is not None else default_device()
        h = C.c_void_p()
        _capi.check(_capi.lib().wb_ivf_create(self.d, self.nlist, self._device, C.byref(h)))
        self._hd = _Handle(h)

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
        _capi.check(L.wb_ivf_set_spherical(self._h, int(bool(cp.spherical))))
        _capi.check(L.wb_ivf_train(self._h, n, _capi.ptr(x), int(cp.niter), int(cp.seed)))
        self._sync_quantizer()

    def _sync_quantizer(self) -> None:
        """Keep the user-visible quantizer object in the state faiss leaves it in (holding the centroids)."""
        if self.quantizer is not None and self.quantizer.ntotal == 0:
            self.quantizer.add(self.centroids())

    def centroids(self) -> np.ndarray:
        c = np.empty((self.nlist, self.d), np.float32)
        _capi.check(_capi.lib().wb_ivf_get_centroids(self._h, _capi.ptr(c)))
        return c

    def set_centroids(self, c) -> None:
        """Install trained centroids (read_index, or 'the reference's own trained centroids')."""
        c = _as_f32_matrix(c, self.d, "centroids")
        if c.shape[0] != self.nlist:
            raise AssertionError(f"expected {self.nlist} centroids, got {c.shape[0]}")
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
        for s in range(0, n, 1 << 20):
            _, ids, _ = self._export(s, min(1 << 20, n - s), want_x=False)
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
    if keys.shape[0]:
        _capi.check(_capi.lib().wb_reconstruct_batch(index._h, keys.shape[0], _capi.ptr(keys), _capi.ptr(out)))
    return out


def write_index(index: Index, fname: str) -> None:
    """faiss.write_index  (/root/reference/src/index/feature_search_index.py:84)."""
    from . import faiss_io
    faiss_io.write_index(index, fname)


def read_index(fname: str, io_flags: int = 0) -> Index:
    """faiss.read_index(fname, faiss.IO_FLAG_READ_ONLY)  (feature_search_index.py:96)."""
    from . import faiss_io
    return faiss_io.read_index(fname, io_flags)
