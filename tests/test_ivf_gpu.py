"""GPU parity tests for IndexIVFFlat (coarse quantizer, list scan, add, k-means) vs the CPU oracle.
Search is compared on the oracle's own centroids so k-means randomness is out of the picture
(BASELINE.json north_star)."""
import ctypes as C

import numpy as np
import pytest

from oracle import oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def faiss():
    from wise_b200 import faiss_compat
    return faiss_compat


def _ivf(faiss, xb, ids, cent):
    q = faiss.IndexFlatIP(xb.shape[1])
    idx = faiss.IndexIVFFlat(q, xb.shape[1], cent.shape[0], faiss.METRIC_INNER_PRODUCT)
    assert not idx.is_trained
    idx.set_centroids(cent)
    assert idx.is_trained and q.ntotal == cent.shape[0]
    for s in range(0, xb.shape[0], 512):
        idx.add_with_ids(xb[s:s + 512], ids[s:s + 512])
    return idx


@pytest.mark.parametrize("n,d,nlist,k", [(20000, 64, 32, 10), (60000, 512, 300, 100), (30000, 768, 128, 100), (5000, 30, 7, 1000)])
def test_ivf_search_matches_oracle(faiss, n, d, nlist, k):
    xb = O.clustered_unit(n, d, 2 * nlist, 50)
    xq = O.clustered_unit(6, d, 2 * nlist, 51)
    cent = O.kmeans_init(xb, nlist)
    ids = np.arange(n, dtype=np.int64) * 5 + 2
    idx = _ivf(faiss, xb, ids, cent)
    assert idx.ntotal == n and idx.nprobe == 1
    a = O.ivf_assign(xb, cent)
    _, _, ga = idx._export(0, n, want_assign=True)
    assert (ga == a).mean() > 0.9999  # argmax ties / fp32 noise may move a handful of rows
    a = ga.astype(np.int64)  # compare search on identical lists
    for nprobe in (1, 8, 32, 4096):
        idx.nprobe = nprobe
        D, I = idx.search(xq, k)
        Dr, Ir = O.ivf_search(xb, ids, a, cent, xq, k, nprobe)
        O.compare_topk(D, I, Dr, Ir)
    Df, If = O.flat_search(xb, xq, k, ids)  # nprobe >= nlist is exhaustive
    O.compare_topk(D, I, Df, If)
    D1, I1 = idx.search(xq[:1], k)
    O.compare_topk(D1, I1, Df[:1], If[:1])


def test_ivf_untrained_and_surface(faiss):
    q = faiss.IndexFlatIP(16)
    idx = faiss.IndexIVFFlat(q, 16, 4, faiss.METRIC_INNER_PRODUCT)
    assert hasattr(idx, "nprobe") and hasattr(idx, "direct_map") and idx.direct_map.type == idx.direct_map.NoMap
    with pytest.raises(RuntimeError):
        idx.add_with_ids(O.unit_gaussian(3, 16, 0), np.arange(3))
    idx.parallel_mode = 1  # api/routes.py:901
    idx.set_centroids(O.unit_gaussian(4, 16, 1))
    xb = O.unit_gaussian(100, 16, 2)
    idx.add_with_ids(xb, np.arange(1, 101))  # WISE ids start at 1
    with pytest.raises(RuntimeError):
        idx.make_direct_map(True)  # faiss: "direct map supported only for seqential ids"
    with pytest.raises(RuntimeError):
        idx.reconstruct_batch([1])
    idx2 = faiss.IndexIVFFlat(faiss.IndexFlatIP(16), 16, 4, faiss.METRIC_INNER_PRODUCT)
    idx2.set_centroids(O.unit_gaussian(4, 16, 1))
    idx2.add_with_ids(xb, np.arange(100))
    idx2.make_direct_map(True)
    assert idx2.direct_map.type != idx2.direct_map.NoMap
    assert np.array_equal(idx2.reconstruct_batch([5, 99, 0]), xb[[5, 99, 0]])


def test_kmeans_one_iteration_matches_oracle(faiss):
    """From identical starting centroids, one GPU iteration == one oracle iteration."""
    import ctypes as C
    import torch
    from wise_b200 import _capi
    L = _capi.lib()
    n, d, k = 6000, 48, 40
    x = O.clustered_unit(n, d, 60, 9)
    c0 = O.kmeans_init(x, k)
    idx = faiss.IndexIVFFlat(faiss.IndexFlatIP(d), d, k, faiss.METRIC_INNER_PRODUCT)
    idx.set_centroids(c0)
    xd = torch.from_numpy(x).cuda()
    assign = torch.empty(n, dtype=torch.int32, device="cuda")
    sums = torch.empty(k, d, device="cuda"); counts = torch.empty(k, dtype=torch.int64, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    obj = C.c_double(0)
    _capi.check(L.wb_kmeans_assign_dev(idx._h, n, xd.data_ptr(), assign.data_ptr(), C.byref(obj), st))
    _capi.check(L.wb_kmeans_accumulate_dev(idx._h, n, xd.data_ptr(), assign.data_ptr(), sums.data_ptr(), counts.data_ptr(), st))
    nsplit = C.c_int64(0)
    _capi.check(L.wb_kmeans_update_dev(idx._h, sums.data_ptr(), counts.data_ptr(), n, 1234, C.byref(nsplit), st))
    torch.cuda.synchronize()
    c1_ref, a_ref, obj_ref, nsplit_ref = O.kmeans_iteration(x, c0)
    assert (assign.cpu().numpy() == a_ref).mean() > 0.9995
    assert abs(obj.value - obj_ref) < 1e-3 * n * 1e-2
    assert nsplit.value == nsplit_ref
    assert np.abs(idx.centroids() - c1_ref).max() < 1e-4


def test_kmeans_fast_assignment_within_tf32_band(faiss):
    """wb_kmeans_assign_fast_dev (training only): plain-TF32 scores on the 256-centroid SS kernel.  Every point must land
    on a centroid whose exact score is within 2e-3 |x||c| of the best one, and almost all on the best one itself."""
    import ctypes as C
    import torch
    from wise_b200 import _capi
    L = _capi.lib()
    n, d, k = 50000, 200, 700  # 3 centroid blocks (the last one partial), 7 k-chunks (the last one partial)
    x = O.clustered_unit(n, d, 900, 12)
    c0 = O.kmeans_init(x, k)
    idx = faiss.IndexIVFFlat(faiss.IndexFlatIP(d), d, k, faiss.METRIC_INNER_PRODUCT)
    idx.set_centroids(c0)
    xd = torch.from_numpy(x).cuda()
    assign = torch.empty(n, dtype=torch.int32, device="cuda")
    obj = C.c_double(0)
    st = torch.cuda.current_stream().cuda_stream
    _capi.check(L.wb_kmeans_assign_fast_dev(idx._h, n, xd.data_ptr(), assign.data_ptr(), C.byref(obj), st))
    torch.cuda.synchronize()
    a = assign.cpu().numpy().astype(np.int64)
    s = x.astype(np.float64) @ c0.astype(np.float64).T
    best = s.max(axis=1)
    got = s[np.arange(n), a]
    assert a.min() >= 0 and a.max() < k
    assert np.all(best - got <= 2e-3), float((best - got).max())
    assert (a == s.argmax(axis=1)).mean() > 0.995
    assert abs(obj.value - best.sum()) < 2e-3 * n


@pytest.mark.parametrize("spherical", [False, True])
def test_train_end_to_end_objective(faiss, spherical):
    """index.train (plain-TF32 assignment on the SS tensor-core kernel, device-side grouping): same clustering quality
    as the fp64 oracle run of the same algorithm; cp.spherical as in faiss (default False)."""
    n, d, k = 8000, 64, 50
    x = O.clustered_unit(n, d, 50, 21)
    idx = faiss.IndexIVFFlat(faiss.IndexFlatIP(d), d, k, faiss.METRIC_INNER_PRODUCT)
    assert idx.cp.spherical is False and idx.cp.niter == 10
    idx.cp.spherical = spherical
    idx.train(x)
    assert idx.is_trained and idx.quantizer.ntotal == k
    c = idx.centroids()
    if spherical:
        assert np.allclose(np.linalg.norm(c, axis=1), 1.0, atol=1e-4)
    else:
        assert np.all(np.linalg.norm(c, axis=1) <= 1.0 + 1e-4)
    c_ref, objs = O.kmeans_train(x, k, spherical=spherical)
    obj_gpu = float(np.max(x.astype(np.float64) @ c.astype(np.float64).T, axis=1).sum())
    obj_ref = float(np.max(x.astype(np.float64) @ c_ref.astype(np.float64).T, axis=1).sum())
    assert obj_gpu >= 0.995 * obj_ref, (obj_gpu, obj_ref)
    idx.add(x)
    idx.nprobe = 5
    D, I = idx.search(x[:4], 3)
    assert np.array_equal(I[:, 0], np.arange(4))


def test_ivf_ties_across_lists_and_regrouping(faiss):
    """Equal scores in DIFFERENT lists order by insertion position (the Flat rule; the oracle's rule), not by list
    number: the row store is regrouped list by list on the device (K8) but keys carry the original position.
    Also: storage-order export after the grouping, adds after a grouping, reconstruct on a grouped store."""
    from wise_b200 import _capi
    L = _capi.lib()
    n, d, nlist = 3000, 32, 8
    cent = O.unit_gaussian(nlist, d, 3)
    xb = O.unit_gaussian(n, d, 4)
    xb[1500] = xb[10]  # exact duplicate at a later insertion position
    assign = O.ivf_assign(xb, cent).astype(np.int32)
    assign[10], assign[1500] = 6, 2  # ... and the EARLIER row lives in the LATER list
    ids = np.arange(n, dtype=np.int64)
    idx = faiss.IndexIVFFlat(faiss.IndexFlatIP(d), d, nlist, faiss.METRIC_INNER_PRODUCT)
    idx.set_centroids(cent)
    _capi.check(L.wb_ivf_add_preassigned(idx._h, n, _capi.ptr(xb), _capi.ptr(ids), _capi.ptr(assign)))
    idx.nprobe = nlist
    xq = np.concatenate([xb[10:11], O.unit_gaussian(5, d, 5)])
    D, I = idx.search(xq, 20)
    assert I[0, 0] == 10 and I[0, 1] == 1500 and D[0, 0] == D[0, 1]
    Dr, Ir = O.ivf_search(xb, ids, assign.astype(np.int64), cent, xq, 20, nlist)
    O.compare_topk(D, I, Dr, Ir)
    # storage order after the grouping: list by list, insertion order inside a list, ids follow their rows
    x, i, a = idx._export(0, n, want_assign=True)
    assert np.all(np.diff(a) >= 0) and np.array_equal(x, xb[i]) and np.array_equal(a, assign[i])
    for l in range(nlist):
        assert np.all(np.diff(i[a == l]) > 0)
    # adds after a grouping: the next search regroups, old and new rows keep their insertion order
    x2 = O.unit_gaussian(500, d, 6)
    x2[7] = xb[10]
    a2 = O.ivf_assign(x2, cent).astype(np.int32)
    a2[7] = 0
    ids2 = np.arange(n, n + 500, dtype=np.int64)
    _capi.check(L.wb_ivf_add_preassigned(idx._h, 500, _capi.ptr(x2), _capi.ptr(ids2), _capi.ptr(a2)))
    D, I = idx.search(xq, 20)
    assert list(I[0, :3]) == [10, 1500, n + 7] and D[0, 0] == D[0, 2]
    xa, ia, aa = np.concatenate([xb, x2]), np.concatenate([ids, ids2]), np.concatenate([assign, a2]).astype(np.int64)
    Dr, Ir = O.ivf_search(xa, ia, aa, cent, xq, 20, nlist)
    O.compare_topk(D, I, Dr, Ir)
    idx.nprobe = 2
    D, I = idx.search(xq, 20)
    Dr, Ir = O.ivf_search(xa, ia, aa, cent, xq, 20, 2)
    O.compare_topk(D, I, Dr, Ir)
    # ids are 0..ntotal-1: the direct map exists and reconstruct finds rows in the grouped store
    idx.make_direct_map(True)
    assert np.array_equal(idx.reconstruct_batch([10, 1500, n + 7, 2999, 0]), xa[[10, 1500, n + 7, 2999, 0]])


def test_ivf_write_index_without_search_is_grouped(faiss, tmp_path):
    """create_index's order (train, add, write_index - no search): the writer finalizes the lists first, the file
    round-trips and searches like the original (/root/reference/src/index/feature_search_index.py:75-84)."""
    n, d, nlist = 20000, 48, 25
    xb = O.clustered_unit(n, d, 50, 8)
    ids = np.arange(n, dtype=np.int64) * 3 + 1
    cent = O.kmeans_init(xb, nlist)
    idx = _ivf(faiss, xb, ids, cent)
    fn = str(tmp_path / "image-IndexIVFFlat.faiss")
    faiss.write_index(idx, fn)
    idx2 = faiss.read_index(fn, faiss.IO_FLAG_READ_ONLY)
    assert idx2.ntotal == n and idx2.nlist == nlist
    xq = O.clustered_unit(4, d, 50, 9)
    for index in (idx, idx2):
        index.nprobe = 6
    D1, I1 = idx.search(xq, 10)
    D2, I2 = idx2.search(xq, 10)
    assert np.array_equal(I1, I2) and np.array_equal(D1, D2)


@pytest.mark.parametrize("n,d,nlist,k,nq", [(60000, 128, 64, 100, 96), (40000, 768, 200, 10, 33), (30000, 64, 16, 1000, 20)])
def test_ivf_batched_listmajor_matches_oracle(faiss, monkeypatch, n, d, nlist, k, nq):
    """Batches take the list-major kernel (ivf_lm.cuh): the probe table is inverted on the device, every probed list
    is streamed once per group of 8 queries, thresholds are shared across work items.  Same results as the oracle
    and as the query-major kernel, for few and many probes, including exact duplicates in different lists."""
    from wise_b200 import _capi
    L = _capi.lib()
    xb = O.clustered_unit(n, d, 3 * nlist, 60)
    xb[n - 7] = xb[11]
    cent = O.kmeans_init(xb, nlist)
    assign = O.ivf_assign(xb, cent).astype(np.int32)
    assign[n - 7] = (assign[11] + 1) % nlist  # the duplicate lives in another list
    ids = np.arange(n, dtype=np.int64) * 2 + 3
    idx = faiss.IndexIVFFlat(faiss.IndexFlatIP(d), d, nlist, faiss.METRIC_INNER_PRODUCT)
    idx.set_centroids(cent)
    _capi.check(L.wb_ivf_add_preassigned(idx._h, n, _capi.ptr(xb), _capi.ptr(ids), _capi.ptr(assign)))
    xq = np.concatenate([xb[11:12], O.clustered_unit(nq - 1, d, 3 * nlist, 61)])
    for nprobe in (1, 8, nlist):
        idx.nprobe = nprobe
        monkeypatch.setenv("WB_IVF_LISTMAJOR", "1")
        l0 = L.wb_launch_count(idx._h)
        D, I = idx.search(xq, k)
        assert L.wb_launch_count(idx._h) - l0 >= 6, "the list-major path launches its table-building kernels"
        monkeypatch.setenv("WB_IVF_LISTMAJOR", "0")
        Dq, Iq = idx.search(xq, k)
        Dr, Ir = O.ivf_search(xb, ids, assign.astype(np.int64), cent, xq, k, nprobe)
        O.compare_topk(D, I, Dr, Ir)
        O.compare_topk(Dq, Iq, Dr, Ir)
        if nprobe == nlist:
            assert I[0, 0] == ids[11] and I[0, 1] == ids[n - 7] and D[0, 0] == D[0, 1]
    monkeypatch.delenv("WB_IVF_LISTMAJOR")
    idx.nprobe = nlist  # nq * nprobe >= nlist: the automatic choice is list-major
    D, I = idx.search(xq, k)
    O.compare_topk(D, I, Dr, Ir)


def test_ivf_ungrouped_store_matches_grouped(faiss, monkeypatch, tmp_path):
    """When the second copy of the rows does not fit, the IVF store stays un-grouped: the list scan gathers rows through
    the CSR of row indices (`perm`).  WB_IVF_CONTIGUOUS=0 forces that.  An un-grouped index B returns the same bytes as
    a grouped twin A (selection keys carry the insertion position, not the storage row): in the fused coarse launch
    (1 and 4 queries) and in the query-major scan of a batch, where the list-major kernel refuses an un-grouped store.
    Then B is grouped once, takes more rows and is left un-grouped again (`perm` over a store described by `row_pos`).
    reconstruct_batch and a write_index / read_index round trip agree with A."""
    from wise_b200 import _capi
    L = _capi.lib()
    n, d, nlist, k = 20000, 128, 32, 50
    cent = O.unit_gaussian(nlist, d, 80)
    xs, ids, assigns = [], [], []

    def add(m, seed):  # the same rows into A and B, with an exact duplicate of row 11 in another list
        x = O.clustered_unit(m, d, 3 * nlist, seed)
        x[m - 7] = xs[0][11] if xs else x[11]
        a = O.ivf_assign(x, cent).astype(np.int32)
        a[m - 7] = (assigns[0][11] if assigns else a[11]) + 1
        a[m - 7] %= nlist
        i = np.arange(sum(len(v) for v in ids), sum(len(v) for v in ids) + m, dtype=np.int64)
        for index in (A, B):
            _capi.check(L.wb_ivf_add_preassigned(index._h, m, _capi.ptr(x), _capi.ptr(i), _capi.ptr(a)))
        xs.append(x)
        ids.append(i)
        assigns.append(a)

    def grouped(index):
        off = np.empty(nlist + 1, np.int64)
        g = C.c_int(-1)
        _capi.check(L.wb_ivf_list_offsets(index._h, _capi.ptr(off), C.byref(g)))
        return g.value

    def regroup(ungrouped_b):
        assert grouped(A) == 1
        if ungrouped_b:
            monkeypatch.setenv("WB_IVF_CONTIGUOUS", "0")
        assert grouped(B) == (0 if ungrouped_b else 1)
        monkeypatch.delenv("WB_IVF_CONTIGUOUS", raising=False)

    def same(D, I, D2, I2):
        return np.array_equal(I, I2) and np.array_equal(D.view(np.uint32), D2.view(np.uint32))

    def check_searches():
        xa, ia, aa = np.concatenate(xs), np.concatenate(ids), np.concatenate(assigns).astype(np.int64)
        xq = np.concatenate([xa[11:12], O.clustered_unit(63, d, 3 * nlist, 81)])
        for nq in (1, 4, 64):
            for nprobe in (1, 8, nlist):
                A.nprobe = B.nprobe = nprobe
                DA, IA = A.search(xq[:nq], k)
                f0 = L.wb_ivf_fused_searches(B._h)
                DB, IB = B.search(xq[:nq], k)
                Dr, Ir = O.ivf_search(xa, ia, aa, cent, xq[:nq], k, nprobe)
                O.compare_topk(DA, IA, Dr, Ir)
                O.compare_topk(DB, IB, Dr, Ir)
                if nq <= 4:  # both take the fused coarse launch
                    assert L.wb_ivf_fused_searches(B._h) - f0 == 1, "the fused path was not taken"
                else:  # A takes the list-major kernel by default; compare the same query-major kernel
                    monkeypatch.setenv("WB_IVF_LISTMAJOR", "0")
                    DA, IA = A.search(xq[:nq], k)
                    monkeypatch.delenv("WB_IVF_LISTMAJOR")
                assert same(DA, IA, DB, IB), (nq, nprobe)
                if nprobe == nlist:  # equal scores in different lists: insertion order
                    assert IB[0, 0] == 11 and IB[0, 1] == len(xs[0]) - 7 and DB[0, 0] == DB[0, 1]

    A = faiss.IndexIVFFlat(faiss.IndexFlatIP(d), d, nlist, faiss.METRIC_INNER_PRODUCT)
    B = faiss.IndexIVFFlat(faiss.IndexFlatIP(d), d, nlist, faiss.METRIC_INNER_PRODUCT)
    A.set_centroids(cent)
    B.set_centroids(cent)
    monkeypatch.delenv("WB_IVF_CONTIGUOUS", raising=False)
    add(n, 82)
    regroup(ungrouped_b=True)
    check_searches()
    # B grouped (row_pos set), then more rows and un-grouped again: perm over a store that row_pos describes
    add(3000, 83)
    regroup(ungrouped_b=False)
    add(2000, 84)
    regroup(ungrouped_b=True)
    check_searches()
    xa = np.concatenate(xs)
    A.make_direct_map(True)
    B.make_direct_map(True)
    keys = [11, n - 7, n + 2999, n + 3000, xa.shape[0] - 1, 0, 12345]
    assert np.array_equal(B.reconstruct_batch(keys), xa[keys])
    assert np.array_equal(B.reconstruct_batch(keys), A.reconstruct_batch(keys))
    fa, fb = str(tmp_path / "a.faiss"), str(tmp_path / "b.faiss")
    faiss.write_index(A, fa)
    faiss.write_index(B, fb)
    assert grouped(B) == 0  # writing did not regroup B
    with open(fa, "rb") as f1, open(fb, "rb") as f2:
        assert f1.read() == f2.read()
    B2 = faiss.read_index(fb, faiss.IO_FLAG_READ_ONLY)
    xq = O.clustered_unit(8, d, 3 * nlist, 85)
    A.nprobe = B2.nprobe = 8
    assert same(*A.search(xq, k), *B2.search(xq, k))
    assert np.array_equal(B2.reconstruct_batch(keys), xa[keys])


def test_kmeans_split_clusters_matches_oracle(faiss):
    """Empty lists: the host draws the (empty, donor) pairs from the list sizes with the faiss procedure (mt19937, same
    stream as the oracle), split_apply_kernel applies them on the device.  Several empties, one donor hit twice."""
    import ctypes as C
    import torch
    from wise_b200 import _capi
    L = _capi.lib()
    n, d, k = 3000, 32, 24
    x = O.clustered_unit(n, d, 6, 13)
    c0 = O.kmeans_init(x, k)
    for dead in (3, 9, 10, 20):
        c0[dead] = -c0[0] * (1.0 + 0.01 * dead)  # nobody's best centroid
    idx = faiss.IndexIVFFlat(faiss.IndexFlatIP(d), d, k, faiss.METRIC_INNER_PRODUCT)
    idx.set_centroids(c0)
    xd = torch.from_numpy(x).cuda()
    assign = torch.empty(n, dtype=torch.int32, device="cuda")
    sums = torch.empty(k, d, device="cuda"); counts = torch.empty(k, dtype=torch.int64, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    obj = C.c_double(0)
    _capi.check(L.wb_kmeans_assign_dev(idx._h, n, xd.data_ptr(), assign.data_ptr(), C.byref(obj), st))
    _capi.check(L.wb_kmeans_accumulate_dev(idx._h, n, xd.data_ptr(), assign.data_ptr(), sums.data_ptr(), counts.data_ptr(), st))
    nsplit = C.c_int64(0)
    _capi.check(L.wb_kmeans_update_dev(idx._h, sums.data_ptr(), counts.data_ptr(), n, 1234, C.byref(nsplit), st))
    torch.cuda.synchronize()
    c1_ref, a_ref, _, nsplit_ref = O.kmeans_iteration(x, c0)
    assert np.array_equal(assign.cpu().numpy(), a_ref)
    assert nsplit.value == nsplit_ref and nsplit.value >= 4
    assert np.abs(idx.centroids() - c1_ref).max() < 1e-5


@pytest.mark.parametrize("n,nlist,skew", [(300000, 5000, 1.5), (70001, 3, 0.0), (1000, 4096, 0.0), (200000, 64, 3.0)])
def test_k8_device_grouping_is_a_stable_counting_sort(faiss, n, nlist, skew):
    """K8 (csr.cuh: histogram, column scan, stable scatter): after wb_ivf_finalize the storage order is exactly
    numpy's stable argsort of the list numbers - skewed lists, empty lists, more lists than rows, several item blocks."""
    from wise_b200 import _capi
    L = _capi.lib()
    d = 8
    rng = np.random.default_rng(n + nlist)
    if skew > 0:
        w = 1.0 / np.arange(1, nlist + 1) ** skew
        assign = rng.choice(nlist, size=n, p=w / w.sum()).astype(np.int32)
    else:
        assign = rng.integers(0, nlist, size=n).astype(np.int32)
    x = rng.standard_normal((n, d)).astype(np.float32)
    ids = rng.permutation(n).astype(np.int64) + 7
    idx = faiss.IndexIVFFlat(faiss.IndexFlatIP(d), d, nlist, faiss.METRIC_INNER_PRODUCT)
    idx.set_centroids(O.unit_gaussian(nlist, d, 1))
    for s in range(0, n, 50000):  # several adds
        e = min(n, s + 50000)
        _capi.check(L.wb_ivf_add_preassigned(idx._h, e - s, _capi.ptr(x[s:e]), _capi.ptr(ids[s:e]), _capi.ptr(assign[s:e])))
    _capi.check(L.wb_ivf_finalize(idx._h))
    xs, is_, as_ = idx._export(0, n, want_assign=True)
    order = np.argsort(assign, kind="stable")
    assert np.array_equal(as_, assign[order]) and np.array_equal(is_, ids[order]) and np.array_equal(xs, x[order])
    off = np.empty(nlist + 1, np.int64)
    grouped = C.c_int(0)
    _capi.check(L.wb_ivf_list_offsets(idx._h, _capi.ptr(off), C.byref(grouped)))
    assert grouped.value == 1
    assert np.array_equal(off, np.concatenate([[0], np.cumsum(np.bincount(assign, minlength=nlist))]))
    bad = assign.copy()
    bad[5] = nlist  # an assignment outside [0, nlist) is reported, not scattered
    idx2 = faiss.IndexIVFFlat(faiss.IndexFlatIP(d), d, nlist, faiss.METRIC_INNER_PRODUCT)
    idx2.set_centroids(O.unit_gaussian(nlist, d, 1))
    _capi.check(L.wb_ivf_add_preassigned(idx2._h, 100, _capi.ptr(x[:100]), _capi.ptr(ids[:100]), _capi.ptr(bad[:100])))
    assert L.wb_ivf_finalize(idx2._h) != 0 and b"outside" in L.wb_last_error()


def test_misc_entry_points(faiss):
    """wb_tf32_peak (the roofline denominator), pinned buffers, slot bookkeeping of the asynchronous add."""
    from wise_b200 import _capi
    L = _capi.lib()
    tb, ts = C.c_double(), C.c_double()
    _capi.check(L.wb_tf32_peak(0, 2000, 4, C.byref(tb), C.byref(ts)))
    assert 300.0 < tb.value < 1400.0 and 300.0 < ts.value < 1400.0, (tb.value, ts.value)
    d, n = 40, 1000
    p_x, p_i = C.c_void_p(), C.c_void_p()
    _capi.check(L.wb_pinned_alloc(n * d * 4, C.byref(p_x)))
    _capi.check(L.wb_pinned_alloc(n * 8, C.byref(p_i)))
    x = np.ctypeslib.as_array((C.c_float * (n * d)).from_address(p_x.value)).reshape(n, d)
    ids = np.ctypeslib.as_array((C.c_int64 * n).from_address(p_i.value))
    x[:] = O.unit_gaussian(n, d, 3)
    ids[:] = np.arange(n) * 2
    idx = faiss.IndexIDMap(faiss.IndexFlatIP(d))
    assert L.wb_add_with_ids_pinned(idx._h, n, p_x, p_i, 8) != 0  # slot out of range
    _capi.check(L.wb_add_with_ids_pinned(idx._h, n, p_x, p_i, 3))
    _capi.check(L.wb_add_slot_wait(idx._h, 3))
    _capi.check(L.wb_add_slot_wait(idx._h, 5))  # nothing pending: returns at once
    _capi.check(L.wb_sync(idx._h))
    D, I = idx.search(x[:3].copy(), 1)
    assert I[:, 0].tolist() == [0, 2, 4]
    _capi.check(L.wb_pinned_free(p_x))
    _capi.check(L.wb_pinned_free(p_i))


@pytest.mark.parametrize("nq", [1, 40])
def test_ivf_nan_rows_are_stored_but_never_returned(faiss, nq):
    """Same float-compare rule as the flat index (faiss heaps never insert a NaN score).  faiss's add_core drops a row
    whose coarse label is -1 while still counting it in ntotal; here such a row lands in list 0 and no search can
    return it - the observable behaviour (ntotal, results) is the same."""
    n, d, nlist, k = 30000, 128, 64, 20
    xb = O.clustered_unit(n, d, 2 * nlist, 60)
    xq = O.clustered_unit(nq, d, 2 * nlist, 61)
    cent = O.kmeans_init(xb, nlist)
    bad = np.array([3, 700, 15000, n - 2])
    xb[bad, 9] = np.nan
    ids = np.arange(n, dtype=np.int64) * 7
    idx = _ivf(faiss, xb, ids, cent)
    assert idx.ntotal == n
    _, _, ga = idx._export(0, n, want_assign=True)
    clean = np.setdiff1d(np.arange(n), bad)
    for nprobe in (4, 64):
        idx.nprobe = nprobe
        D, I = idx.search(xq, k)
        Dr, Ir = O.ivf_search(xb[clean], ids[clean], ga[clean].astype(np.int64), cent, xq, k, nprobe)
        O.compare_topk(D, I, Dr, Ir)
        assert not np.isin(I, ids[bad]).any() and np.isfinite(D).all()
        xq2 = xq.copy()
        xq2[-1, 0] = np.nan  # a NaN query has no best centroid: it probes nothing and returns the empty row
        D2, I2 = idx.search(xq2, k)
        assert np.all(I2[-1] == -1) and np.all(D2[-1] == O.NEG_FLT_MAX)
        if nq > 1:
            O.compare_topk(D2[:-1], I2[:-1], Dr[:-1], Ir[:-1])
    # faiss Clustering::train refuses a training set with NaN / Inf [faiss-upstream]
    fresh = faiss.IndexIVFFlat(faiss.IndexFlatIP(d), d, nlist, faiss.METRIC_INNER_PRODUCT)
    with pytest.raises(RuntimeError, match="NaN"):
        fresh.train(xb[:10000])  # rows 3 and 700 are corrupt (no subsampling below 256 points per centroid)
    assert not fresh.is_trained
    fresh.train(xb[clean][:10000])
    assert fresh.is_trained


@pytest.mark.parametrize("n,d,nlist,k", [(40000, 512, 300, 100), (30000, 64, 7, 10), (120000, 128, 20000, 100),
                                          (20000, 768, 1024, 1000)])
def test_ivf_fused_coarse_matches_two_launch_path(faiss, monkeypatch, n, d, nlist, k):
    """Up to 4 queries: the coarse quantizer runs as the prologue of the list-scan kernel (coarse.cuh) - ONE cooperative
    launch per search.  Same (D, I) bytes as the two-launch path (coarse scan + merge, then the list scan) and parity
    with the oracle, for one and many probes, fewer lists than CTAs, more lists than one histogram pass separates,
    a zero query (every coarse score ties: the LOWER list ids are probed) and a NaN query (no list is probed)."""
    from wise_b200 import _capi
    L = _capi.lib()
    xb = O.clustered_unit(n, d, min(2 * nlist, 4000), 70)
    cent = O.kmeans_init(xb, nlist)
    ids = np.arange(n, dtype=np.int64) * 3 + 1
    idx = _ivf(faiss, xb, ids, cent)
    _, _, ga = idx._export(0, n, want_assign=True)
    a = ga.astype(np.int64)
    xq = O.clustered_unit(4, d, min(2 * nlist, 4000), 71)
    idx.search(xq, 1)  # groups the rows by list (K8) - not part of the launch counts below
    for nq in (1, 2, 3, 4):
        for nprobe in sorted({1, 5, 32, 128, nlist} & set(range(1, nlist + 1))):
            idx.nprobe = nprobe
            monkeypatch.setenv("WB_IVF_FUSE_COARSE", "1")
            f0, l0 = L.wb_ivf_fused_searches(idx._h), L.wb_launch_count(idx._h)
            D, I = idx.search(xq[:nq], k)
            assert L.wb_ivf_fused_searches(idx._h) - f0 == 1, "the fused path was not taken"
            assert L.wb_launch_count(idx._h) - l0 == 1, "a fused search is one launch"
            monkeypatch.setenv("WB_IVF_FUSE_COARSE", "0")
            f0 = L.wb_ivf_fused_searches(idx._h)
            D2, I2 = idx.search(xq[:nq], k)
            assert L.wb_ivf_fused_searches(idx._h) == f0
            assert np.array_equal(I, I2) and np.array_equal(D.view(np.uint32), D2.view(np.uint32)), (nq, nprobe)
            if nprobe in (1, 32, nlist) and nq in (1, 4) and nlist <= 1024:
                Dr, Ir = O.ivf_search(xb, ids, a, cent, xq[:nq], k, nprobe)
                O.compare_topk(D, I, Dr, Ir)
    # degenerate coarse scores
    idx.nprobe = min(5, nlist)
    for q in (np.zeros((1, d), np.float32), np.full((1, d), np.nan, np.float32)):
        monkeypatch.setenv("WB_IVF_FUSE_COARSE", "1")
        D, I = idx.search(q, k)
        monkeypatch.setenv("WB_IVF_FUSE_COARSE", "0")
        D2, I2 = idx.search(q, k)
        assert np.array_equal(I, I2) and np.array_equal(D.view(np.uint32), D2.view(np.uint32))
    monkeypatch.setenv("WB_IVF_FUSE_COARSE", "1")
    D, I = idx.search(np.zeros((1, d), np.float32), k)
    in_first = np.isin(a, np.arange(idx.nprobe))  # rows of the lists 0 .. nprobe-1, lowest insertion positions first
    want = ids[np.nonzero(in_first)[0][:k]]
    assert np.array_equal(I[0, :want.size], want) and (I[0, want.size:] == -1).all()
    D, I = idx.search(np.full((1, d), np.nan, np.float32), k)
    assert (I == -1).all()
