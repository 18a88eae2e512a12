"""Sharded range search on B200s: wb_range_search_dev against wb_range_search, wb_range_merge_dev against one index
holding all rows (several indices on one GPU, no transport), ShardedIndex with world 1, and a 2-GPU run of
ShardedIndex.range_search under both exchange modes (skipped with fewer than 2 GPUs)."""
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
from wise_b200.sharded import ShardedIndex, _cuda_local_range_search, _cuda_range_merge, shard_range

pytestmark = pytest.mark.gpu


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _bytes(*arrays):
    return b"".join(np.ascontiguousarray(a).tobytes() for a in arrays)


def _host_and_dev(index, xq, thresh, flt=None, nprobe=1):
    """wb_range_search and wb_range_search_dev on the same queries; each result read through both copy functions,
    which must agree.  Returns (host lims, D, I), (dev lims, D, I)."""
    L = _capi.lib()
    n = len(xq)
    st = torch.cuda.current_stream().cuda_stream
    q = torch.from_numpy(xq).cuda()
    out = []
    for dev in (False, True):
        lims = np.zeros(n + 1, np.int64)
        res = C.c_void_p()
        if dev:
            _capi.check(L.wb_range_search_dev(index._h, flt, n, q.data_ptr() if n else None, float(thresh), nprobe,
                                              _capi.ptr(lims), C.byref(res), st))
        else:
            _capi.check(L.wb_range_search(index._h, flt, n, _capi.ptr(xq) if n else None, float(thresh), nprobe,
                                          _capi.ptr(lims), C.byref(res)))
        try:
            total = int(lims[-1])
            Dh, Ih = np.empty(total, np.float32), np.empty(total, np.int64)
            _capi.check(L.wb_range_result_copy(res, _capi.ptr(Dh), _capi.ptr(Ih)))
            Dd = torch.empty(total, dtype=torch.float32, device="cuda")
            Id = torch.empty(total, dtype=torch.int64, device="cuda")
            _capi.check(L.wb_range_result_copy_dev(res, Dd.data_ptr(), Id.data_ptr(), st))
            torch.cuda.synchronize()
        finally:
            _capi.check(L.wb_range_result_free(res))
        assert _bytes(Dd.cpu().numpy(), Id.cpu().numpy()) == _bytes(Dh, Ih)
        out.append((lims, Dh, Ih))
    return out


N, D = 200_000, 126  # d = 126: the queries are re-strided on the device


@pytest.fixture(scope="module")
def flat():
    xb = O.unit_gaussian(N, D, 501)
    xb[150_001] = xb[1234]
    ids = np.random.default_rng(8).permutation(N).astype(np.int64) * 2 + 3
    index = faiss.IndexIDMap(faiss.IndexFlatIP(D))
    index.add_with_ids(xb, ids)
    return index, xb, ids


def _thresh(xb, xq, hits):
    s = (xq.astype(np.float64) @ xb.astype(np.float64).T).ravel()
    return float(np.quantile(s, 1 - hits / xb.shape[0]))


# (nq, WB_GEMM_FORCE, selector kind): K1, K1, K2 TS, K2 SS, the mask filter, the compact filter
FLAT_PATHS = [(1, False, None), (4, False, None), (16, True, None), (200, True, None), (4, False, 0.5),
              (200, True, 0.5), (4, False, 0.01)]


@pytest.mark.parametrize("nq,force,frac", FLAT_PATHS)
def test_dev_equals_host_flat(flat, monkeypatch, nq, force, frac):
    index, xb, ids = flat
    if force:
        monkeypatch.setenv("WB_GEMM_FORCE", "1")
    flt = None
    if frac is not None:
        sel = faiss.IDSelectorBatch(np.random.default_rng(21).choice(ids, int(frac * N), replace=False))
        _, flt = index._search_params(faiss.SearchParameters(sel=sel))
    xq = O.unit_gaussian(nq, D, 60 + nq)
    (lh, Dh, Ih), (ld, Dd, Id) = _host_and_dev(index, xq, _thresh(xb, xq, 3000), flt)
    assert lh[-1] > 0
    assert _bytes(lh, Dh, Ih) == _bytes(ld, Dd, Id)


def test_dev_equals_host_edge_cases(flat):
    index, xb, _ = flat
    xq = O.unit_gaussian(3, D, 11)
    for q, t in ((xq[:0], 0.0), (xq, 2.0)):  # nq = 0; no hits at all
        (lh, Dh, Ih), (ld, Dd, Id) = _host_and_dev(index, q, t)
        assert lh[-1] == 0 and _bytes(lh, Dh, Ih) == _bytes(ld, Dd, Id)
    # 64 queries x 200k rows = 12.8M hits: the first pool is too small and grows before the chunk runs again
    xb64 = O.unit_gaussian(N, 64, 9)
    big = faiss.IndexFlatIP(64)
    big.add(xb64)
    (lh, Dh, Ih), (ld, Dd, Id) = _host_and_dev(big, O.unit_gaussian(64, 64, 10), -2.0)
    assert lh[-1] == 64 * N and _bytes(lh, Dh, Ih) == _bytes(ld, Dd, Id)


def test_dev_equals_host_ivf():
    n, d, nlist = 60_000, 64, 32
    xb = O.clustered_unit(n, d, 64, 31)
    cent = O.unit_gaussian(nlist, d, 32)
    ids = np.arange(n, dtype=np.int64) * 5 + 1
    index = faiss.IndexIVFFlat(faiss.IndexFlatIP(d), d, nlist, faiss.METRIC_INNER_PRODUCT)
    index.set_centroids(cent)
    index.add_with_ids(xb, ids)
    xq = O.clustered_unit(8, d, 64, 41)
    t = _thresh(xb, xq, 300)
    params = faiss.SearchParametersIVF(sel=faiss.IDSelectorRange(1, 5 * (n // 2)), nprobe=8)  # owns the filter
    _, flt = index._search_params(params)
    for f in (None, flt):
        (lh, Dh, Ih), (ld, Dd, Id) = _host_and_dev(index, xq, t, f, nprobe=8)
        assert lh[-1] > 0 and _bytes(lh, Dh, Ih) == _bytes(ld, Dd, Id)


def test_dev_after_dev_add_on_a_side_stream():
    """Rows added with wb_add_with_ids_dev on a non-default stream, then at once wb_range_search_dev on that stream:
    the lists are grouped (on the index's own stream) only after the add has landed, so the result equals that of an
    index filled from the host."""
    n, d, nlist = 60_000, 64, 32
    xb = O.clustered_unit(n, d, 64, 31)
    cent = O.unit_gaussian(nlist, d, 32)
    ids = np.arange(n, dtype=np.int64) * 5 + 1
    xq = O.clustered_unit(8, d, 64, 43)
    t = _thresh(xb, xq, 300)

    def make():
        index = faiss.IndexIVFFlat(faiss.IndexFlatIP(d), d, nlist, faiss.METRIC_INNER_PRODUCT)
        index.set_centroids(cent)
        return index

    ref = make()
    ref.add_with_ids(xb, ids)
    want = _host_and_dev(ref, xq, t, nprobe=8)[0]
    L = _capi.lib()
    index = make()
    side = torch.cuda.Stream()
    x, i, q = (torch.from_numpy(a).cuda() for a in (xb, ids, xq))
    torch.cuda.synchronize()
    st = side.cuda_stream
    for rep in range(2):  # the first search groups the lists; the second reads the grouped store
        lims = np.zeros(len(xq) + 1, np.int64)
        res = C.c_void_p()
        if rep == 0:
            _capi.check(L.wb_add_with_ids_dev(index._h, n, x.data_ptr(), i.data_ptr(), st))
        _capi.check(L.wb_range_search_dev(index._h, None, len(xq), q.data_ptr(), float(t), 8, _capi.ptr(lims),
                                          C.byref(res), st))
        try:
            total = int(lims[-1])
            Dd = torch.empty(total, dtype=torch.float32, device="cuda")
            Id = torch.empty(total, dtype=torch.int64, device="cuda")
            _capi.check(L.wb_range_result_copy_dev(res, Dd.data_ptr(), Id.data_ptr(), st))
            side.synchronize()
        finally:
            _capi.check(L.wb_range_result_free(res))
        assert want[0][-1] > 0
        assert _bytes(lims, Dd.cpu().numpy(), Id.cpu().numpy()) == _bytes(*want)


def _merge_parts(parts, xq, t):
    """Local _dev range search on every part, packed into the padded all-gather layout, merged by wb_range_merge_dev."""
    q = torch.from_numpy(xq).cuda()
    local = [_cuda_local_range_search(p, q, t, 1) for p in parts]
    nq = len(xq)
    lims_parts = torch.stack([lims for lims, _, _ in local])
    stride = int(lims_parts[:, -1].max())
    Dp = torch.full((len(parts), stride), float("nan"), dtype=torch.float32, device="cuda")
    Ip = torch.full((len(parts), stride), -7, dtype=torch.int64, device="cuda")
    for p, (lims, Dl, Il) in enumerate(local):
        Dp[p, :Dl.shape[0]] = Dl
        Ip[p, :Il.shape[0]] = Il
    lims = lims_parts.sum(dim=0)
    if stride == 0:
        return lims.numpy(), np.zeros(0, np.float32), np.zeros(0, np.int64)
    D1, I1 = _cuda_range_merge(lims_parts, Dp, Ip, lims)
    D2, I2 = _cuda_range_merge(lims_parts, Dp, Ip, lims)
    torch.cuda.synchronize()
    assert _bytes(D1.cpu().numpy(), I1.cpu().numpy()) == _bytes(D2.cpu().numpy(), I2.cpu().numpy())
    assert nq == lims.shape[0] - 1
    return lims.numpy(), D1.cpu().numpy(), I1.cpu().numpy()


NM, DM = 120_000, 64


@pytest.fixture(scope="module")
def merge_data():
    xb = O.unit_gaussian(NM, DM, 71)
    xb[NM - 100:] = xb[:100]  # duplicates of the first slice's rows in the last slice
    ids = np.arange(NM, dtype=np.int64) * 3 + 2
    whole = faiss.IndexIDMap(faiss.IndexFlatIP(DM))
    whole.add_with_ids(xb, ids)
    return xb, ids, whole


@pytest.mark.parametrize("P", [1, 2, 3, 8])
@pytest.mark.parametrize("nq,force", [(4, False), (16, True)])  # K1 on every part; K2 on every part
def test_merge_equals_one_index(merge_data, monkeypatch, P, nq, force):
    xb, ids, whole = merge_data
    if force:
        monkeypatch.setenv("WB_GEMM_FORCE", "1")
    # contiguous slices in order; with P >= 3 slice 1 is empty
    bounds = [shard_range(NM, r, P) for r in range(P)]
    if P >= 3:
        bounds = [(0, bounds[1][1])] + [(bounds[1][1], bounds[1][1])] + bounds[2:]
    parts = []
    for lo, hi in bounds:
        idx = faiss.IndexIDMap(faiss.IndexFlatIP(DM))
        if hi > lo:
            idx.add_with_ids(xb[lo:hi], ids[lo:hi])
        parts.append(idx)
    xq = O.unit_gaussian(nq, DM, 72 + nq)
    xq[0] = xb[3]  # an exact tie across the first and the last slice
    xq[1] = 0.0  # no hits anywhere
    t = 0.05  # ~35k hits per query: more than kRangeRun (8192) on several parts
    got = _merge_parts(parts, xq, t)
    want = whole.range_search(xq, t)
    assert int(want[0][2]) > 30_000 and want[0][2] == want[0][1]
    assert _bytes(got[0].astype(np.uint64), got[1], got[2]) == _bytes(*want)
    a = int(want[0][0])
    assert want[2][a] == ids[3] and want[2][a + 1] == ids[NM - 100 + 3]


def test_merge_argument_checks():
    L = _capi.lib()
    st = torch.cuda.current_stream().cuda_stream
    for nq, parts, stride in ((-1, 1, 0), (1, 0, 0), (1, 1, -1)):
        assert L.wb_range_merge_dev(0, nq, parts, None, stride, None, None, None, None, None, st) != 0
    assert L.wb_range_merge_dev(0, 0, 2, None, 5, None, None, None, None, None, st) == 0  # nothing to merge
    assert L.wb_range_merge_dev(0, 3, 2, None, 5, None, None, None, None, None, st) != 0  # NULL buffers


def test_sharded_world1_equals_index(flat):
    index, xb, _ = flat
    sh = ShardedIndex(index)
    assert sh.world == 1
    xq = O.unit_gaussian(4, D, 5)
    t = _thresh(xb, xq, 2000)
    want = index.range_search(xq, t)
    got = sh.range_search(xq, t)
    assert got[0].dtype == np.uint64 and _bytes(*got) == _bytes(*want)
    lims, Dd, Id = sh.range_search_dev(torch.from_numpy(xq).cuda(), t)
    assert lims.device.type == "cpu" and Dd.is_cuda and Id.is_cuda
    assert _bytes(lims.numpy().astype(np.uint64), Dd.cpu().numpy(), Id.cpu().numpy()) == _bytes(*want)


# ---- two GPUs ------------------------------------------------------------------------------------------------------
N2, D2, NLIST2 = 60_000, 256, 32
BATCHES = [(1, False), (4, False), (16, True), (40, False)]  # K1, K1, K2 on both sides; 40: whichever each side takes


def _two_gpu_data():
    xb = O.unit_gaussian(N2, D2, 77)
    xb[N2 - 50:] = xb[:50]
    ids = np.arange(N2, dtype=np.int64) * 2 + 5
    cent = O.unit_gaussian(NLIST2, D2, 78)
    return xb, ids, cent


def _queries(xb, nq):
    xq = O.unit_gaussian(nq, D2, 90 + nq)
    xq[-1] = xb[3]
    return xq


def _two_gpu_searches(make, xb, ids, cent, res, tag, env):
    """Every (kind, batch) range search through `make(kind)` -> an object with range_search(x, t, params=...)."""
    sel = faiss.IDSelectorRange(int(ids[1000]), int(ids[N2 - 1000]))
    for kind in ("flat", "ivf", "filtered"):
        index = make(kind)
        for nq, force in BATCHES:
            env(force)
            xq = _queries(xb, nq)
            params = faiss.SearchParameters(sel=sel) if kind == "filtered" else None
            t = 0.12
            res[f"{tag}_{kind}_{nq}"] = np.concatenate([x.view(np.uint8) for x in index.range_search(xq, t, params=params)])
        env(False)


def _worker(rank, world, port, out, mode):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), WISE_B200_EXCHANGE=mode,
                      WISE_B200_DEVICE=str(rank))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))

    def env(force):
        if force:
            os.environ["WB_GEMM_FORCE"] = "1"
        else:
            os.environ.pop("WB_GEMM_FORCE", None)

    try:
        xb, ids, cent = _two_gpu_data()
        lo, hi = shard_range(N2, rank, world)

        def make_shard(kind):
            if kind == "ivf":
                idx = faiss.IndexIVFFlat(faiss.IndexFlatIP(D2, device=rank), D2, NLIST2, faiss.METRIC_INNER_PRODUCT)
                idx.set_centroids(cent)
                idx.nprobe = 8
            else:
                idx = faiss.IndexIDMap(faiss.IndexFlatIP(D2, device=rank))
            idx.add_with_ids(xb[lo:hi], ids[lo:hi])
            sh = ShardedIndex(idx)
            assert (sh.exchange is not None) == (mode == "peer")
            return sh

        res = {}
        shards = {}

        def make_and_check(kind):
            shards[kind] = make_shard(kind)
            return shards[kind]

        _two_gpu_searches(make_and_check, xb, ids, cent, res, "sh", env)
        # range_search_dev == range_search; a search between range searches still matches; no exchange time-out
        sh = shards["flat"]
        xq = _queries(xb, 4)
        D0, I0 = sh.search(xq, 100)
        want = sh.range_search(xq, 0.12)
        lims, Dd, Id = sh.range_search_dev(torch.from_numpy(xq).cuda(rank), 0.12)
        torch.cuda.synchronize()
        assert _bytes(lims.numpy().astype(np.uint64), Dd.cpu().numpy(), Id.cpu().numpy()) == _bytes(*want)
        D1, I1 = sh.search(xq, 100)
        assert _bytes(D0, I0) == _bytes(D1, I1)
        again = sh.range_search(xq, 0.12)
        assert _bytes(*again) == _bytes(*want)
        if sh.exchange is not None:
            assert not sh.exchange.timed_out()
        if rank == 0:  # the single index on GPU 0
            def make_single(kind):
                if kind == "ivf":
                    idx = faiss.IndexIVFFlat(faiss.IndexFlatIP(D2, device=0), D2, NLIST2, faiss.METRIC_INNER_PRODUCT)
                    idx.set_centroids(cent)
                    idx.nprobe = 8
                else:
                    idx = faiss.IndexIDMap(faiss.IndexFlatIP(D2, device=0))
                idx.add_with_ids(xb, ids)
                return idx

            _two_gpu_searches(make_single, xb, ids, cent, res, "one", env)
        np.savez(os.path.join(out, f"{mode}_r{rank}.npz"), **res)
    finally:
        dist.destroy_process_group()


def _unpack(buf, nq):
    lims = buf[:8 * (nq + 1)].view(np.uint64)
    total = int(lims[-1])
    D = buf[8 * (nq + 1):8 * (nq + 1) + 4 * total].view(np.float32)
    I = buf[8 * (nq + 1) + 4 * total:].view(np.int64)
    return lims, D, I


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("mode", ["peer", "nccl"])
def test_two_gpu_sharded_range(tmp_path, mode):
    mp.spawn(_worker, args=(2, _free_port(), str(tmp_path), mode), nprocs=2, join=True)
    xb, ids, cent = _two_gpu_data()
    r0, r1 = (np.load(tmp_path / f"{mode}_r{r}.npz") for r in (0, 1))
    keep = (ids >= ids[1000]) & (ids < ids[N2 - 1000])
    for kind in ("flat", "ivf", "filtered"):
        for nq, force in BATCHES:
            key = f"{kind}_{nq}"
            assert np.array_equal(r0["sh_" + key], r1["sh_" + key]), key  # identical on both ranks
            lims, D, I = _unpack(r0["sh_" + key], nq)
            assert lims[-1] > 0
            if kind != "filtered":  # (the selector drops row 3 and its copy)
                a = int(lims[nq - 1])
                assert I[a] == ids[3] and I[a + 1] == ids[N2 - 50 + 3]  # exact tie across the ranks: rank 0 first
            if nq <= 4 or force or kind == "ivf":  # the same kernel family on both sides: bit for bit
                assert np.array_equal(r0["sh_" + key], r0["one_" + key]), key
                continue
            # otherwise the single-GPU contract: fp64 membership outside the near-tie band, fp32 scores, the order
            xq = _queries(xb, nq)
            pos_of = {int(v): p for p, v in enumerate(ids)}
            for i in range(nq):
                a, b = int(lims[i]), int(lims[i + 1])
                d, p = D[a:b], np.array([pos_of[int(v)] for v in I[a:b]], np.int64)
                rows = np.nonzero(keep)[0] if kind == "filtered" else np.arange(N2)
                s = xb[rows].astype(np.float64) @ xq[i].astype(np.float64)
                assert np.all(d > np.float32(0.12)) and np.all(np.isin(p, rows))
                assert np.all(np.isin(rows[s > 0.12 + 4e-6], p))
                assert np.all(np.abs(d - xb[p].astype(np.float64) @ xq[i].astype(np.float64)) <= 1e-5)
                assert np.all(np.diff(d.astype(np.float64)) <= 0) and np.all(np.diff(p)[np.diff(d) == 0] > 0)
