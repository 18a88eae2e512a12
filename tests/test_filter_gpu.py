"""Filtered search (faiss SearchParameters with an IDSelector) on a B200: every search path against the unmodified
oracle over the selected subset.  The subset keeps insertion order, so ties agree with the oracle too."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from oracle import oracle as O
from wise_b200 import _capi
from wise_b200 import faiss_compat as faiss

pytestmark = pytest.mark.gpu

N, D = 200_000, 126  # ld = 128: the compact copy carries the padding columns
FRACTIONS = {"dense": 0.5, "above_cutoff": 0.14, "sparse": 0.01, "tiny": 1e-4}


def _keep(sel, ids):
    """Boolean mask of the rows `sel` keeps (the selector semantics, in numpy)."""
    if isinstance(sel, faiss.IDSelectorNot):
        return ~_keep(sel.sel, ids)
    if isinstance(sel, faiss.IDSelectorRange):
        return (ids >= sel.imin) & (ids < sel.imax)
    return np.isin(ids, sel.ids)


def _selector(kind, frac, ids, seed):
    rng = np.random.default_rng(seed)
    n = ids.size
    if kind == "batch":
        return faiss.IDSelectorBatch(rng.choice(ids, max(1, int(round(frac * n))), replace=False))
    if kind == "not_batch":
        return faiss.IDSelectorNot(faiss.IDSelectorBatch(rng.choice(ids, n - max(1, int(round(frac * n))), replace=False)))
    lo = int(np.sort(ids)[n // 3])  # ids are a shuffled arithmetic sequence: a range keeps scattered positions
    span = int(round(frac * n)) * 2
    return faiss.IDSelectorRange(lo, lo + max(span, 2))


def _gemm_stats(index):
    e, f = C.c_int64(0), C.c_int64(0)
    _capi.check(_capi.lib().wb_gemm_stats(index._h, C.byref(e), C.byref(f)))
    return e.value, f.value


@pytest.fixture(scope="module")
def flat():
    xb = O.unit_gaussian(N, D, 901)
    ids = np.random.default_rng(3).permutation(N).astype(np.int64) * 2 + 11
    index = faiss.IndexIDMap(faiss.IndexFlatIP(D))
    index.add_with_ids(xb, ids)
    return index, xb, ids


def _check_flat(index, xb, ids, sel, xq, k):
    keep = _keep(sel, ids)
    Dg, Ig = index.search(xq, k, params=faiss.SearchParameters(sel=sel))
    Dr, Ir = O.flat_search(xb[keep], xq, k, ids[keep])
    O.compare_topk(Dg, Ig, Dr, Ir, band=4e-6)
    assert np.all(np.isin(Ig[Ig >= 0], ids[keep]))
    return Dg, Ig


# (nq, force K2): K1 at 1 and 4 queries, K2 TS (16 queries, tensor-core path forced), K2 SS (200 queries)
PATHS = [(1, False), (4, False), (16, True), (200, True)]


@pytest.mark.parametrize("nq,force", PATHS)
@pytest.mark.parametrize("frac", list(FRACTIONS))
@pytest.mark.parametrize("kind", ["batch", "range", "not_batch"])
def test_flat_filtered_matches_oracle(flat, monkeypatch, nq, force, frac, kind):
    index, xb, ids = flat
    if force:
        monkeypatch.setenv("WB_GEMM_FORCE", "1")
    sel = _selector(kind, FRACTIONS[frac], ids, 17)
    xq = O.unit_gaussian(nq, D, 40 + nq)
    xq[0] = xb[int(np.nonzero(_keep(sel, ids))[0][0])]  # a query whose best row is selected
    _check_flat(index, xb, ids, sel, xq, 100)


@pytest.mark.parametrize("nq", [16, 200])
@pytest.mark.parametrize("k", [100, 1000])
@pytest.mark.parametrize("frac", [0.5, 0.14])
def test_flat_k2_mask_needs_no_fallback(flat, monkeypatch, nq, k, frac):
    """The K2 epoch schedule counts selected rows: a dense filter on random-order data never overflows into K1, and
    the store is large enough for several epochs."""
    index, xb, ids = flat
    monkeypatch.setenv("WB_GEMM_FORCE", "1")
    sel = faiss.IDSelectorBatch(np.random.default_rng(5).choice(ids, int(frac * N), replace=False))
    e0, f0 = _gemm_stats(index)
    _check_flat(index, xb, ids, sel, O.unit_gaussian(nq, D, 7 + k), k)
    e1, f1 = _gemm_stats(index)
    assert f1 == f0, "K2 fell back to the CUDA-core scan"
    assert e1 - e0 >= 2, f"only {e1 - e0} K2 epochs"


@pytest.mark.parametrize("nq,force", PATHS)
def test_flat_keep_everything_is_bytes_identical(flat, monkeypatch, nq, force):
    index, xb, ids = flat
    if force:
        monkeypatch.setenv("WB_GEMM_FORCE", "1")
    xq = O.unit_gaussian(nq, D, 99 + nq)
    D0, I0 = index.search(xq, 100)
    D1, I1 = index.search(xq, 100, params=faiss.SearchParameters(sel=faiss.IDSelectorNot(faiss.IDSelectorBatch([]))))
    assert np.array_equal(D0, D1) and np.array_equal(I0, I1)


@pytest.mark.parametrize("nq,force", [(1, False), (16, True)])
def test_flat_ties_and_padding(monkeypatch, nq, force):
    if force:
        monkeypatch.setenv("WB_GEMM_FORCE", "1")
    n = 50_000
    xb = O.unit_gaussian(n, 64, 12)
    xb[n - 1] = xb[5]  # planted duplicate: the copy at position 5 wins the tie while it is allowed
    ids = np.arange(n, dtype=np.int64) + 1000
    index = faiss.IndexIDMap(faiss.IndexFlatIP(64))
    index.add_with_ids(xb, ids)
    xq = np.repeat(xb[5:6], nq, axis=0)
    _, I = index.search(xq, 2, params=faiss.SearchParameters(sel=faiss.IDSelectorRange(0, 1 << 40)))
    assert I[0, 0] == ids[5] and I[0, 1] == ids[n - 1]
    _, I = index.search(xq, 2, params=faiss.SearchParameters(sel=faiss.IDSelectorNot(faiss.IDSelectorBatch([ids[5]]))))
    assert I[0, 0] == ids[n - 1]
    # fewer rows than k, and none at all: exact (-FLT_MAX, -1) padding
    few = faiss.IDSelectorBatch(ids[[3, 700, 40_000, 49_999]])
    Dg, Ig = index.search(xq, 10, params=faiss.SearchParameters(sel=few))
    Dr, Ir = O.flat_search(xb[[3, 700, 40_000, 49_999]], xq, 10, ids[[3, 700, 40_000, 49_999]])
    O.compare_topk(Dg, Ig, Dr, Ir)
    assert np.all(Ig[:, 4:] == -1) and np.all(Dg[:, 4:] == np.float32(-3.4028235e38))
    for none in (faiss.IDSelectorBatch([]), faiss.IDSelectorRange(5, 5), faiss.IDSelectorRange(9, 2)):
        Dg, Ig = index.search(xq, 10, params=faiss.SearchParameters(sel=none))
        assert np.all(Ig == -1) and np.all(Dg == np.float32(-3.4028235e38))


@pytest.mark.parametrize("frac", [0.5, 0.01])
def test_filter_follows_later_adds(frac):
    """A selector made before an add sees the new rows (the bitmap and the compact copy are rebuilt)."""
    n, d = 80_000, 64
    xb = O.unit_gaussian(n, d, 21)
    ids = np.arange(n, dtype=np.int64)
    index = faiss.IndexIDMap(faiss.IndexFlatIP(d))
    index.add_with_ids(xb[: n // 2], ids[: n // 2])
    sel = faiss.IDSelectorBatch(ids[:: int(round(1 / frac))])
    params = faiss.SearchParameters(sel=sel)
    xq = xb[[n - 100, n - 200, n - 300, n - 400]].copy()  # their best rows come with the later add, and are selected
    index.search(xq, 10, params=params)
    index.add_with_ids(xb[n // 2:], ids[n // 2:])
    keep = _keep(sel, ids)
    Dg, Ig = index.search(xq, 10, params=params)
    Dr, Ir = O.flat_search(xb[keep], xq, 10, ids[keep])
    O.compare_topk(Dg, Ig, Dr, Ir)
    assert Ig[0, 0] == n - 100


def test_filter_of_another_index_is_refused(flat):
    index, _, ids = flat
    other = faiss.IndexIDMap(faiss.IndexFlatIP(D))
    other.add_with_ids(O.unit_gaussian(100, D, 1), np.arange(100, dtype=np.int64))
    sel = faiss.IDSelectorRange(0, 50)
    f = sel._filter(other._hd)
    xq = O.unit_gaussian(1, D, 2)
    Dg, Ig = np.empty((1, 5), np.float32), np.empty((1, 5), np.int64)
    with pytest.raises(RuntimeError, match="another index"):
        _capi.check(_capi.lib().wb_search_filtered(index._h, f, 1, _capi.ptr(xq), 5, 1, _capi.ptr(Dg), _capi.ptr(Ig)))


# ---- IVF --------------------------------------------------------------------------------------------------------
NI, DI, NLIST = 60_000, 64, 64


def _ivf(xb, ids, cent, grouped_later=False):
    index = faiss.IndexIVFFlat(faiss.IndexFlatIP(DI), DI, NLIST, faiss.METRIC_INNER_PRODUCT)
    index.set_centroids(cent)
    if grouped_later:  # search once (the store is grouped), then add more: row_pos is no longer the identity
        index.add_with_ids(xb[: NI // 2], ids[: NI // 2])
        index.search(xb[:1], 1)
        index.add_with_ids(xb[NI // 2:], ids[NI // 2:])
    else:
        index.add_with_ids(xb, ids)
    return index


@pytest.fixture(scope="module")
def ivf_data():
    xb = O.unit_gaussian(NI, DI, 31)
    ids = np.random.default_rng(4).permutation(NI).astype(np.int64) * 3 + 2
    cent = O.unit_gaussian(NLIST, DI, 32)
    return xb, ids, cent, O.ivf_assign(xb, cent)


# (store, nq, env): fused coarse launch, two launches, list-major batch, un-grouped store, grouped then grown
IVF_PATHS = [("plain", 1, {}), ("plain", 4, {}), ("plain", 4, {"WB_IVF_FUSE_COARSE": "0"}),
             ("plain", 64, {"WB_IVF_LISTMAJOR": "1"}), ("ungrouped", 4, {}), ("ungrouped", 64, {}),
             ("grown", 1, {}), ("grown", 64, {"WB_IVF_LISTMAJOR": "1"})]


@pytest.mark.parametrize("store,nq,env", IVF_PATHS)
@pytest.mark.parametrize("kind", ["batch", "range", "not_batch"])
def test_ivf_filtered_matches_oracle(ivf_data, monkeypatch, store, nq, env, kind):
    xb, ids, cent, assign = ivf_data
    if store == "ungrouped":
        monkeypatch.setenv("WB_IVF_CONTIGUOUS", "0")
    index = _ivf(xb, ids, cent, grouped_later=store == "grown")
    for key, v in env.items():
        monkeypatch.setenv(key, v)
    xq = O.unit_gaussian(nq, DI, 50 + nq)
    for frac in (0.5, 0.02):
        sel = _selector(kind, frac, ids, 23)
        keep = _keep(sel, ids)
        Dg, Ig = index.search(xq, 50, params=faiss.SearchParametersIVF(sel=sel, nprobe=8))
        Dr, Ir = O.ivf_search(xb[keep], ids[keep], assign[keep], cent, xq, 50, 8)
        O.compare_topk(Dg, Ig, Dr, Ir)
    # a selector that keeps every row returns the unfiltered bytes
    index.nprobe = 8
    D0, I0 = index.search(xq, 50)
    D1, I1 = index.search(xq, 50, params=faiss.SearchParametersIVF(
        sel=faiss.IDSelectorNot(faiss.IDSelectorBatch([])), nprobe=8))
    assert np.array_equal(D0, D1) and np.array_equal(I0, I1)


def test_ivf_params_nprobe_and_type(ivf_data):
    xb, ids, cent, assign = ivf_data
    index = _ivf(xb, ids, cent)
    index.nprobe = 1
    sel = faiss.IDSelectorRange(0, int(ids.max()) // 2)
    keep = _keep(sel, ids)
    xq = O.unit_gaussian(4, DI, 8)
    Dg, Ig = index.search(xq, 20, params=faiss.SearchParametersIVF(sel=sel, nprobe=6))
    Dr, Ir = O.ivf_search(xb[keep], ids[keep], assign[keep], cent, xq, 20, 6)
    O.compare_topk(Dg, Ig, Dr, Ir)
    Dg, Ig = index.search(xq, 20, params=faiss.SearchParametersIVF(sel=sel))  # faiss default nprobe = 1
    Dr, Ir = O.ivf_search(xb[keep], ids[keep], assign[keep], cent, xq, 20, 1)
    O.compare_topk(Dg, Ig, Dr, Ir)
    with pytest.raises(RuntimeError, match="incorrect type"):
        index.search(xq, 20, params=faiss.SearchParameters(sel=sel))
    Dg, Ig = index.search(xq, 20, params=faiss.SearchParametersIVF(sel=faiss.IDSelectorBatch([]), nprobe=6))
    assert np.all(Ig == -1)


# ---- sharded ------------------------------------------------------------------------------------------------------
NS, DS = 60_000, 128


def _shard_data():
    xb = O.unit_gaussian(NS, DS, 61)
    ids = np.arange(NS, dtype=np.int64) * 2 + 5
    rng = np.random.default_rng(8)
    # sparse on rank 0 (1 % of its rows: the compact copy), dense on rank 1 (60 %: the mask)
    mixed = np.concatenate([rng.choice(ids[: NS // 2], NS // 200, replace=False),
                            rng.choice(ids[NS // 2:], NS * 3 // 10, replace=False)])
    return xb, ids, {"mixed": faiss.IDSelectorBatch(mixed),
                     "rank1_only": faiss.IDSelectorRange(int(ids[NS // 2]), 1 << 40),  # nothing on rank 0
                     "none": faiss.IDSelectorBatch([])}


CASES = [(1, 100), (4, 10), (40, 50)]


def _shard_worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), WISE_B200_EXCHANGE="peer",
                      WISE_B200_DEVICE=str(rank))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from wise_b200.sharded import ShardedIndex, shard_range
        xb, ids, sels = _shard_data()
        lo, hi = shard_range(NS, rank, world)
        idx = faiss.IndexIDMap(faiss.IndexFlatIP(DS, device=rank))
        idx.add_with_ids(xb[lo:hi], ids[lo:hi])
        sh = ShardedIndex(idx)
        assert sh.exchange is not None
        res = {}
        for name, sel in sels.items():
            params = faiss.SearchParameters(sel=sel)
            for nq, k in CASES:
                xq = O.unit_gaussian(nq, DS, 70 + nq)
                D, I = sh.search(xq, k, params=params)
                Dd, Id = sh.search_dev(torch.from_numpy(xq).cuda(rank), k, params=params)
                torch.cuda.synchronize()
                assert np.array_equal(Dd.cpu().numpy(), D) and np.array_equal(Id.cpu().numpy(), I)
                assert not sh.exchange.timed_out()
                res[f"{name}_D{nq}"], res[f"{name}_I{nq}"] = D, I
        np.savez(os.path.join(out, f"r{rank}.npz"), **res)
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpu_filtered_equals_single(tmp_path):
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_shard_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    xb, ids, sels = _shard_data()
    single = faiss.IndexIDMap(faiss.IndexFlatIP(DS, device=0))
    single.add_with_ids(xb, ids)
    r0, r1 = (np.load(tmp_path / f"r{r}.npz") for r in (0, 1))
    for name, sel in sels.items():
        for nq, k in CASES:
            xq = O.unit_gaussian(nq, DS, 70 + nq)
            Ds, Is = single.search(xq, k, params=faiss.SearchParameters(sel=sel))
            for r in (r0, r1):
                assert np.array_equal(r[f"{name}_I{nq}"], Is) and np.array_equal(r[f"{name}_D{nq}"], Ds), (name, nq)
