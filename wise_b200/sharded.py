"""Row-sharded search across the GPUs of one box: one process per GPU, torch.distributed for the
plumbing (SURVEY.md section 8e).

Every rank holds a CONTIGUOUS range of the database rows in its own index (IndexIDMap-style: the
rows keep their global ids), queries are replicated, each GPU produces its local top-k with the
same kernels as the single-GPU path, and the only exchange step moves the `nq * k` (score, id)
candidates of every rank to every other rank (<= 1.2 MB per rank at nq=1024, k=100).  On GPUs that is
the library's NVLink peer-memory mailbox (csrc/exchange.cuh) - fused into the scan kernel's tail for
small batches, one extra kernel otherwise; `WISE_B200_EXCHANGE=nccl` (and every CPU/gloo test) takes
one all-gather followed by the K3 merge kernel instead.  Because a row's score does not depend on
which GPU holds it and the merge orders ties by (rank, local order) == global insertion position,
the sharded result is bit-identical to the single-GPU result (tests/test_flat_gpu.py,
tests/test_sharded_cpu.py).

IVF: centroids are replicated, each rank keeps its slice of every inverted list; the candidate
set of a query is the union over ranks, so the same merge applies.

Filtered search (params=SearchParameters(sel=...)): every rank applies the same selector to its own rows, so the
candidate set is again the union over ranks and the exchange is unchanged.  A rank whose rows the selector rejects
entirely contributes padding and still takes part in the exchange.

Range search (range_search / range_search_dev): every rank runs wb_range_search_dev on its rows, leaving its hits on
its GPU.  One all-gather of [status, count per query] tells every rank every rank's lims; a non-zero status (the local
call failed) makes every rank raise.  Two all-gathers then move D and I, each padded to the largest rank total (skipped
when no rank has a hit), and wb_range_merge_dev places every hit at its rank in the merged result: score descending,
equal scores by (rank, local order) == global insertion position, as on one index.  The payload varies per call from
nothing to gigabytes, so it goes through torch.distributed, not through the fixed-size peer mailbox, whose sequence
range search leaves untouched.
"""
from __future__ import annotations

import os
from typing import Callable

import numpy as np
import torch
import torch.distributed as dist

from .routing import shard_range  # noqa: F401  (part of this module's interface)


def _cuda_local_search(index, q: torch.Tensor, k: int, nprobe: int, flt=None):
    """Local top-k on this rank's GPU; `flt` (a wb_filter* of `index`, or None) restricts the rows."""
    from . import _capi
    nq = q.shape[0]
    D = torch.empty((nq, k), dtype=torch.float32, device=q.device)
    I = torch.empty((nq, k), dtype=torch.int64, device=q.device)
    st = torch.cuda.current_stream(q.device).cuda_stream
    _capi.check(_capi.lib().wb_search_filtered_dev(index._h, flt, nq, q.data_ptr(), k, nprobe, D.data_ptr(),
                                                   I.data_ptr(), st))
    return D, I


def _cuda_merge(Dp: torch.Tensor, Ip: torch.Tensor):
    """Dp, Ip: [parts, nq, k] on the GPU -> merged [nq, k] (wb_merge_topk_dev, K3)."""
    from . import _capi
    parts, nq, k = Dp.shape
    D = torch.empty((nq, k), dtype=torch.float32, device=Dp.device)
    I = torch.empty((nq, k), dtype=torch.int64, device=Dp.device)
    st = torch.cuda.current_stream(Dp.device).cuda_stream
    _capi.check(_capi.lib().wb_merge_topk_dev(Dp.device.index or 0, nq, k, parts, Dp.data_ptr(), Ip.data_ptr(),
                                              D.data_ptr(), I.data_ptr(), st))
    return D, I


def _cuda_local_range_search(index, q: torch.Tensor, thresh: float, nprobe: int, flt=None):
    """Local range search on the index's GPU (wb_range_search_dev): lims [nq + 1] int64 CPU tensor, D / I on that GPU.
    Queries elsewhere (host queries of a single process without an NCCL group) are moved there first."""
    import ctypes as C
    from . import _capi
    L = _capi.lib()
    dev = torch.device("cuda", index._device)
    q = q.to(dev).contiguous()
    nq = q.shape[0]
    lims = torch.zeros(nq + 1, dtype=torch.int64)
    st = torch.cuda.current_stream(dev).cuda_stream
    res = C.c_void_p()
    _capi.check(L.wb_range_search_dev(index._h, flt, nq, q.data_ptr() if nq else None, float(thresh), nprobe,
                                      lims.data_ptr(), C.byref(res), st))
    try:
        total = int(lims[-1])
        D = torch.empty(total, dtype=torch.float32, device=q.device)
        I = torch.empty(total, dtype=torch.int64, device=q.device)
        _capi.check(L.wb_range_result_copy_dev(res, D.data_ptr(), I.data_ptr(), st))
    finally:
        # cudaFree waits for the device, so the copies just enqueued on `st` finish before the result's memory goes;
        # an asynchronous free would need an explicit synchronisation of `st` here
        L.wb_range_result_free(res)
    return lims, D, I


def _cuda_range_merge(lims_parts: torch.Tensor, Dp: torch.Tensor, Ip: torch.Tensor, lims: torch.Tensor):
    """lims_parts [parts, nq + 1] and lims [nq + 1] (int64, CPU); Dp, Ip [parts, stride] on the GPU, part p's hits of
    query q at [lims_parts[p, q], lims_parts[p, q + 1]) of row p -> merged (D, I) (wb_range_merge_dev)."""
    from . import _capi
    parts, stride = Dp.shape
    nq = lims.shape[0] - 1
    dev = Dp.device
    lp = lims_parts.to(dev)
    ld = lims.to(dev)
    total = int(lims[-1])
    D = torch.empty(total, dtype=torch.float32, device=dev)
    I = torch.empty(total, dtype=torch.int64, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream
    _capi.check(_capi.lib().wb_range_merge_dev(dev.index or 0, nq, parts, lp.data_ptr(), stride, Dp.data_ptr(),
                                               Ip.data_ptr(), ld.data_ptr(), D.data_ptr(), I.data_ptr(), st))
    return D, I


class PeerExchange:
    """wb_exchange: the all-gather + merge as one kernel over NVLink peer memory (exchange.cuh).
    Mailbox handles travel once through torch.distributed; after that no NCCL call is on the search path."""

    def __init__(self, group=None, max_queries: int = 4096, max_entries: int = 1 << 20):
        import ctypes as C
        from . import _capi
        self._capi, self._C = _capi, C
        L = _capi.lib()
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.device = torch.cuda.current_device()
        self.h = C.c_void_p()
        _capi.check(L.wb_exch_create(self.device, self.rank, self.world, max_queries, max_entries, C.byref(self.h)))
        mine = C.create_string_buffer(64)
        _capi.check(L.wb_exch_local_handle(self.h, mine))
        handles = [None] * self.world
        dist.all_gather_object(handles, bytes(mine.raw), group=group)
        blob = C.create_string_buffer(b"".join(handles), 64 * self.world)
        _capi.check(L.wb_exch_open_peers(self.h, blob))
        dist.barrier(group=group)
        self.max_queries, self.max_entries = max_queries, max_entries

    def fits(self, nq: int, k: int) -> bool:
        return nq <= self.max_queries and nq * k <= self.max_entries

    def merge(self, D: torch.Tensor, I: torch.Tensor):
        nq, k = D.shape
        Do = torch.empty_like(D)
        Io = torch.empty_like(I)
        st = torch.cuda.current_stream(D.device).cuda_stream
        self._capi.check(self._capi.lib().wb_exch_merge_dev(self.h, nq, k, D.data_ptr(), I.data_ptr(), Do.data_ptr(),
                                                            Io.data_ptr(), st))
        return Do, Io

    def search_dev(self, index, q: torch.Tensor, k: int, nprobe: int, flt=None):
        """Local search + exchange + merge in one C call (one kernel launch for scan-served searches); `flt` is an
        optional wb_filter* of `index`."""
        nq = q.shape[0]
        D = torch.empty((nq, k), dtype=torch.float32, device=q.device)
        I = torch.empty((nq, k), dtype=torch.int64, device=q.device)
        st = torch.cuda.current_stream(q.device).cuda_stream
        self._capi.check(self._capi.lib().wb_exch_search_filtered_dev(index._h, self.h, flt, nq, q.data_ptr(), k, nprobe,
                                                                      D.data_ptr(), I.data_ptr(), st))
        return D, I

    def timed_out(self) -> bool:
        """True when a search gave up waiting for a peer GPU (call after synchronising the stream)."""
        t = self._C.c_int(0)
        self._capi.check(self._capi.lib().wb_exch_status(self.h, self._C.byref(t)))
        return bool(t.value)

    def __del__(self):
        h, self.h = getattr(self, "h", None), None
        if h:
            try:
                self._capi.lib().wb_exch_free(h)
            except Exception:
                pass


class ShardedIndex:
    """A faiss-like index whose rows live on `world_size` GPUs (this process owns one shard).

    local_search / merge and local_range_search / range_merge are injectable so the rank arithmetic and the exchange
    steps can be tested on CPU with the gloo backend; the defaults are the CUDA kernels and nothing else.
    """

    def __init__(self, local_index, group=None,
                 local_search: Callable | None = None, merge: Callable | None = None,
                 local_range_search: Callable | None = None, range_merge: Callable | None = None):
        self.local = local_index
        self.group = group
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self._local_search = local_search or _cuda_local_search
        self._merge = merge or _cuda_merge
        self._local_range_search = local_range_search or _cuda_local_range_search
        self._range_merge = range_merge or _cuda_range_merge
        self.d = local_index.d
        # exchange step: "peer" = one fused kernel over NVLink peer memory (default on GPUs),
        # "nccl" = all-gather + merge kernel.  CPU/gloo tests always take the all-gather path.
        self.exchange = None
        mode = os.environ.get("WISE_B200_EXCHANGE", "peer")
        if (self.world > 1 and mode == "peer" and local_search is None and merge is None
                and dist.get_backend(group) == "nccl"):
            self.exchange = PeerExchange(group)

    @property
    def ntotal(self) -> int:
        n = torch.tensor([self.local.ntotal], dtype=torch.int64, device=self._comm_device())
        if self.world > 1:
            dist.all_reduce(n, group=self.group)
        return int(n.item())

    def _comm_device(self):
        if dist.is_initialized() and dist.get_backend(self.group) == "nccl":
            return torch.device("cuda", torch.cuda.current_device())
        return torch.device("cpu")

    def add_with_ids(self, x, ids) -> None:
        """Each rank adds ITS OWN rows (the caller partitions the store with shard_range)."""
        self.local.add_with_ids(x, ids)

    def _params(self, nprobe: int, params):
        """(nprobe, wb_filter* or None): faiss SearchParameters resolved against this rank's index."""
        if params is None:
            return nprobe, None
        return self.local._search_params(params)

    def search_dev(self, q: torch.Tensor, k: int, nprobe: int = 1, params=None):
        """q: [nq, d] float32 tensor, replicated on every rank. Returns merged (D, I) tensors on every rank.
        params: faiss SearchParameters / SearchParametersIVF (the same selector on every rank; its nprobe replaces
        `nprobe`)."""
        nprobe, flt = self._params(nprobe, params)
        if self.exchange is not None and self.exchange.fits(q.shape[0], k):
            return self.exchange.search_dev(self.local, q.contiguous(), k, nprobe, flt)
        if flt is None:
            D, I = self._local_search(self.local, q, k, nprobe)
        else:
            D, I = self._local_search(self.local, q, k, nprobe, flt)
        if self.world == 1:
            return D, I
        nq, kk = D.shape
        Dp = torch.empty((self.world * nq, kk), dtype=D.dtype, device=D.device)
        Ip = torch.empty((self.world * nq, kk), dtype=I.dtype, device=I.device)
        dist.all_gather_into_tensor(Dp, D.contiguous(), group=self.group)  # concatenated along dim 0
        dist.all_gather_into_tensor(Ip, I.contiguous(), group=self.group)
        return self._merge(Dp.view(self.world, nq, kk), Ip.view(self.world, nq, kk))

    def search(self, x: np.ndarray, k: int, params=None):
        """faiss-style host API: numpy in, numpy out (same on every rank).  params as in search_dev."""
        x = np.ascontiguousarray(x, np.float32)
        if self.exchange is not None and self.exchange.fits(x.shape[0], int(k)):
            # one C call: H2D, local search, NVLink exchange + merge, D2H (no torch ops on the path)
            from . import _capi
            nprobe, flt = self._params(int(getattr(self.local, "nprobe", 1)), params)
            nq = x.shape[0]
            D = np.empty((nq, int(k)), np.float32)
            I = np.empty((nq, int(k)), np.int64)
            _capi.check(_capi.lib().wb_exch_search_filtered(self.local._h, self.exchange.h, flt, nq, _capi.ptr(x), int(k),
                                                           nprobe, _capi.ptr(D), _capi.ptr(I)))
            return D, I
        dev = self._comm_device()
        q = torch.from_numpy(np.ascontiguousarray(x, np.float32)).to(dev)
        nprobe = getattr(self.local, "nprobe", 1)
        D, I = self.search_dev(q, int(k), int(nprobe), params)
        return D.cpu().numpy(), I.cpu().numpy()

    def range_search_dev(self, q: torch.Tensor, thresh, nprobe: int = 1, params=None):
        """q: [nq, d] float32 tensor, replicated on every rank, with the same thresh on every rank.  Returns, on every
        rank, (lims [nq + 1] int64 CPU tensor, D, I on q's device): exactly the range search of one index holding all
        rows (score descending, equal scores by global insertion position).  params as in search_dev.  A failure on
        any rank raises RuntimeError on every rank; no rank is left waiting in a collective."""
        thresh = float(np.float32(thresh))
        try:
            nprobe, flt = self._params(nprobe, params)
            if flt is None:
                lims, D, I = self._local_range_search(self.local, q, thresh, nprobe)
            else:
                lims, D, I = self._local_range_search(self.local, q, thresh, nprobe, flt)
            err = None
        except Exception as e:  # reported through the counts exchange, so that every rank raises
            if self.world == 1:
                raise
            nq = q.shape[0]
            lims, D, I, err = torch.zeros(nq + 1, dtype=torch.int64), None, None, e
        if self.world == 1:
            return lims, D, I
        nq = lims.shape[0] - 1
        dev = self._comm_device()
        # counts: [status, count_0 .. count_{nq-1}] of every rank
        mine = torch.empty(nq + 1, dtype=torch.int64)
        mine[0] = 0 if err is None else 1
        mine[1:] = lims[1:] - lims[:-1]
        counts = torch.empty(self.world * (nq + 1), dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(counts, mine.to(dev), group=self.group)
        counts = counts.cpu().view(self.world, nq + 1)
        failed = torch.nonzero(counts[:, 0]).flatten().tolist()
        if failed:
            msg = f"range_search failed on rank(s) {failed}"
            raise RuntimeError(msg if err is None else f"{msg}: {err}") from err
        lims_parts = torch.zeros((self.world, nq + 1), dtype=torch.int64)
        lims_parts[:, 1:] = torch.cumsum(counts[:, 1:], dim=1)
        merged = lims_parts.sum(dim=0)
        stride = int(lims_parts[:, -1].max())
        if stride == 0:
            return merged, D, I
        # payload: D and I of every rank, padded to the largest rank total; every rank learns whether all could
        # allocate the buffers before any of them enters the gathers
        try:
            Ds = torch.empty(stride, dtype=D.dtype, device=D.device)
            Is = torch.empty(stride, dtype=I.dtype, device=I.device)
            Ds[:D.shape[0]] = D
            Is[:I.shape[0]] = I
            Dp = torch.empty(self.world * stride, dtype=D.dtype, device=D.device)
            Ip = torch.empty(self.world * stride, dtype=I.dtype, device=I.device)
            ok = 1
        except RuntimeError:  # torch.OutOfMemoryError
            Ds = Is = Dp = Ip = None
            ok = 0
        flag = torch.tensor([ok], dtype=torch.int64, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.group)
        if not int(flag.item()):
            raise RuntimeError(f"range_search: a rank could not allocate the {stride} x {self.world} result exchange")
        dist.all_gather_into_tensor(Dp, Ds, group=self.group)
        dist.all_gather_into_tensor(Ip, Is, group=self.group)
        del Ds, Is
        D, I = self._range_merge(lims_parts, Dp.view(self.world, stride), Ip.view(self.world, stride), merged)
        return merged, D, I

    def range_search(self, x: np.ndarray, thresh, params=None):
        """faiss-style host API: lims (uint64, nq + 1), D, I = sh.range_search(x, thresh), numpy in and out, the same on
        every rank (see range_search_dev)."""
        x = np.ascontiguousarray(x, np.float32)
        q = torch.from_numpy(x).to(self._comm_device())
        nprobe = int(getattr(self.local, "nprobe", 1))
        lims, D, I = self.range_search_dev(q, thresh, nprobe, params)
        return lims.numpy().astype(np.uint64), D.cpu().numpy(), I.cpu().numpy()


def train_ivf_sharded(index, x_local: torch.Tensor, niter: int = 10, seed: int = 1234, group=None, verbose: bool = False):
    """index.train() with the training rows sharded over the ranks (SURVEY.md 8e): every rank assigns and
    accumulates ITS rows (K6/K7 on its GPU), one all-reduce of [nlist*d sums | nlist counts] per iteration,
    then every rank applies the identical centroid update, so the centroids stay replicated bit for bit.
    Mirrors faiss Clustering::train for IndexIVFFlat(METRIC_INNER_PRODUCT): index.cp.spherical (default False, like
    the reference's plain-constructor index), niter=10, seed=1234, initial centroids = k random training rows.  `index` is this rank's (empty, untrained) IndexIVFFlat;
    x_local is a float32 [n_local, d] CUDA tensor.  Returns the objective (sum of max inner products) per iteration."""
    import ctypes as C
    from . import _capi
    L = _capi.lib()
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    dev = x_local.device
    x_local = x_local.contiguous()
    n_local, d = x_local.shape
    k = index.nlist
    counts = torch.zeros(world, dtype=torch.int64, device=dev)
    counts[rank] = n_local
    if world > 1:
        dist.all_reduce(counts, group=group)
    n_total = int(counts.sum().item())
    if n_total < k:
        raise RuntimeError(f"Number of training points ({n_total}) should be at least as large as number of clusters ({k})")
    finite = torch.isfinite(x_local.sum(dtype=torch.float64)).to(torch.int32).view(1)  # NaN and +-Inf both poison a sum
    if world > 1:
        dist.all_reduce(finite, op=dist.ReduceOp.MIN, group=group)
    if not int(finite.item()):
        raise RuntimeError("input contains NaN's or Inf's")  # faiss Clustering::train [faiss-upstream]
    # initial centroids: k distinct global rows from a seeded permutation (same on every rank)
    # (drawn on the GPU: a CPU permutation of 10M indices costs more than a training iteration; same seed and same
    # generator on every rank, so all ranks pick the same rows)
    g = torch.Generator(device=dev)
    g.manual_seed(seed + 1)
    pick = torch.randperm(n_total, generator=g, device=dev)[:k].cpu()
    lo = int(counts[:rank].sum().item())
    mine = (pick >= lo) & (pick < lo + n_local)
    init = torch.zeros((k, d), dtype=torch.float32, device=dev)
    init[mine.nonzero().squeeze(1).to(dev)] = x_local[(pick[mine] - lo).to(dev)]
    if world > 1:
        dist.all_reduce(init, group=group)
    spherical = bool(getattr(getattr(index, "cp", None), "spherical", False))
    if spherical:
        init = torch.nn.functional.normalize(init, dim=1)
    _capi.check(L.wb_ivf_set_spherical(index._h, int(spherical)))
    init_h = np.ascontiguousarray(init.cpu().numpy())  # keep a reference: the C call borrows this buffer
    _capi.check(L.wb_ivf_set_centroids(index._h, _capi.ptr(init_h)))
    st = torch.cuda.current_stream(dev).cuda_stream
    assign = torch.empty(n_local, dtype=torch.int32, device=dev)
    sums = torch.empty((k, d), dtype=torch.float32, device=dev)
    cnts = torch.empty(k, dtype=torch.int64, device=dev)
    objs = []
    import time
    timing = os.environ.get("WB_KMEANS_TIMING", "0") != "0"
    for it in range(niter):
        obj = C.c_double(0)
        t0 = time.perf_counter()
        _capi.check(L.wb_kmeans_assign_fast_dev(index._h, n_local, x_local.data_ptr(), assign.data_ptr(), C.byref(obj), st))
        t1 = time.perf_counter()
        _capi.check(L.wb_kmeans_accumulate_dev(index._h, n_local, x_local.data_ptr(), assign.data_ptr(), sums.data_ptr(),
                                               cnts.data_ptr(), st))
        o = torch.tensor([obj.value], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(sums, group=group)
            dist.all_reduce(cnts, group=group)
            dist.all_reduce(o, group=group)
        torch.cuda.synchronize(dev)
        t2 = time.perf_counter()
        nsplit = C.c_int64(0)
        _capi.check(L.wb_kmeans_update_dev(index._h, sums.data_ptr(), cnts.data_ptr(), n_total, 1234, C.byref(nsplit), st))
        torch.cuda.synchronize(dev)
        t3 = time.perf_counter()
        objs.append(float(o.item()))
        if (verbose or timing) and rank == 0:
            print(f"  k-means iteration {it}: objective {objs[-1]:.4f}, split {nsplit.value}; assign {1e3 * (t1 - t0):.1f} ms, "
                  f"group+sums+all-reduce {1e3 * (t2 - t1):.1f} ms, update {1e3 * (t3 - t2):.1f} ms", flush=True)
    _capi.check(L.wb_ivf_mark_trained(index._h))
    index._sync_quantizer()
    return objs
