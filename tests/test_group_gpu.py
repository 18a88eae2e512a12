"""One index over several GPUs of one process (wb_group, faiss_compat devices= / WISE_B200_DEVICES): every search,
filtered search, range search and index file must be byte-identical to one single-GPU index holding all the rows in
the same insertion order.

The stores are integer-valued (small integers times a power of two, as in test_exact_ties_gpu.py), so every score is
exact in fp32 whatever the kernel and the order of accumulation: any difference is a routing, exchange or merge bug,
never rounding.  Ties are frequent, and duplicates of one row are planted on both sides of every shard boundary.
The tests skip with fewer than 2 GPUs; they run on 2 GPUs and, where the box has more, on all of them (up to 8)."""
import numpy as np
import pytest
import torch

from wise_b200 import _capi
from wise_b200 import faiss_compat as faiss

pytestmark = pytest.mark.gpu


def _ngpu():
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


DEVSETS = [[0, 1]] + ([list(range(min(_ngpu(), 8)))] if _ngpu() > 2 else [])
need2 = pytest.mark.skipif(_ngpu() < 2, reason="needs at least 2 GPUs")


def int_store(n, d, seed, L=3, e=2, dup_every=None):
    rng = np.random.default_rng(seed)
    x = rng.integers(-L, L + 1, size=(n, d), dtype=np.int8).astype(np.float32) * np.float32(2.0 ** -e)
    if dup_every:  # copies of row 0 on both sides of every boundary of every device set
        for w in (2, 3, 4, 5, 6, 7, 8):
            for s in range(1, w):
                b = n * s // w
                x[max(b - 1, 0)] = x[0]
                x[min(b, n - 1)] = x[0]
    return x


def queries(nq, d, seed, L=3, e=2):
    return int_store(nq, d, seed + 1000, L, e)


def same(a, b):
    for u, v in zip(a, b):
        assert u.dtype == v.dtype and u.shape == v.shape
        assert np.array_equal(u.view(np.uint8), v.view(np.uint8))


def flat_pair(x, devices, ids=None, reserve=True):
    single = faiss.IndexIDMap(faiss.IndexFlatIP(x.shape[1], device=devices[0]))
    group = faiss.IndexIDMap(faiss.IndexFlatIP(x.shape[1], devices=devices))
    ids = np.arange(x.shape[0], dtype=np.int64) * 3 + 1 if ids is None else ids
    for idx in (single, group):
        if reserve:
            idx.reserve(x.shape[0])
        for a in range(0, x.shape[0], 700000):  # several adds: some straddle a shard boundary
            idx.add_with_ids(x[a:a + 700000], ids[a:a + 700000])
    return single, group


def ivf_pair(x, devices, nlist, seed=5):
    cent = int_store(nlist, x.shape[1], seed, L=2, e=1)
    out = []
    for devs in ([devices[0]], devices):
        idx = faiss.IndexIVFFlat(faiss.IndexFlatIP(x.shape[1], devices=devs), x.shape[1], nlist)
        idx.set_centroids(cent)
        idx.reserve(x.shape[0])
        idx.add_with_ids(x, np.arange(x.shape[0], dtype=np.int64) * 7 + 2)
        out.append(idx)
    return out


@pytest.fixture(scope="module")
def big_flat():
    # 2 x 2.5M rows: each shard of a 2-GPU group is large enough for the bf16 image of 1-2 query searches
    return int_store(5_000_000, 64, 11, dup_every=True)


@need2
@pytest.mark.parametrize("devices", DEVSETS)
def test_flat_search_matches_single_index(big_flat, devices, monkeypatch):
    single, group = flat_pair(big_flat, devices)
    assert [sh.ntotal for sh in group._shards] == [hi - lo for lo, hi in
                                                   (faiss.routing.shard_range(big_flat.shape[0], s, len(devices))
                                                    for s in range(len(devices)))]
    for force in ("0", "1"):  # K1 / bf16 image / K2 as the dispatch picks them, then K2 forced (TS and SS)
        monkeypatch.setenv("WB_GEMM_FORCE", force)
        for nq in (1, 3, 16, 300):
            q = queries(nq, 64, nq)
            for k in (1, 100, 2048):
                same(group.search(q, k), single.search(q, k))


@need2
@pytest.mark.parametrize("devices", DEVSETS)
def test_flat_search_dev_matches_single_index(big_flat, devices):
    single, group = flat_pair(big_flat[:400000], devices)
    L = _capi.lib()
    root = torch.device("cuda", devices[0])
    for nq, k in ((1, 100), (4, 2048), (16, 100), (300, 10)):
        q = torch.from_numpy(queries(nq, 64, nq)).to(root)
        D = torch.empty((nq, k), dtype=torch.float32, device=root)
        I = torch.empty((nq, k), dtype=torch.int64, device=root)
        st = torch.cuda.current_stream(root)
        _capi.check(L.wb_group_search_dev(group._group().g, None, nq, q.data_ptr(), k, 1, D.data_ptr(), I.data_ptr(),
                                          st.cuda_stream))
        st.synchronize()
        same((D.cpu().numpy(), I.cpu().numpy()), single.search(q.cpu().numpy(), k))


@need2
@pytest.mark.parametrize("devices", DEVSETS)
def test_ivf_search_and_assignment_match_single_index(devices, monkeypatch):
    nlist = 128
    x = int_store(300_000, 64, 21, dup_every=True)
    single, group = ivf_pair(x, devices, nlist)
    a1 = single._export(0, single.ntotal, want_assign=True, want_x=False)[2]  # before any search: insertion order
    a2 = np.concatenate([sh._export(0, sh.ntotal, want_assign=True, want_x=False)[2] for sh in group._shards])
    assert np.array_equal(a1, a2)
    for fuse in ("1", "0"):  # one fused launch for 1-4 queries, then the coarse + list-scan launches
        monkeypatch.setenv("WB_IVF_FUSE_COARSE", fuse)
        for nprobe in (1, 8, nlist):
            single.nprobe = group.nprobe = nprobe
            for nq in (1, 3, 64):  # 64: list-major batches
                q = queries(nq, 64, 100 + nq)
                for k in (1, 100):
                    same(group.search(q, k), single.search(q, k))


def _selectors(n, ids_of):
    return {
        "none_of_shard0": faiss.IDSelectorRange(int(ids_of(n // 2 + 1)), int(ids_of(n))),
        "shard0_only": faiss.IDSelectorBatch(ids_of(np.arange(0, n // 4, 3))),
        "zero_rows": faiss.IDSelectorBatch(np.zeros(0, np.int64)),
        "not_sparse": faiss.IDSelectorNot(faiss.IDSelectorRange(int(ids_of(10)), int(ids_of(n - 10)))),
    }


@need2
@pytest.mark.parametrize("devices", DEVSETS)
@pytest.mark.parametrize("kind", ["flat", "ivf"])
def test_filtered_and_range_search_match_single_index(devices, kind):
    n = 200_000
    x = int_store(n, 32, 31, dup_every=True)
    if kind == "flat":
        single, group = flat_pair(x, devices)
        params = lambda sel: faiss.SearchParameters(sel=sel)
        sels = _selectors(n, lambda pos: np.asarray(pos, np.int64) * 3 + 1)
    else:
        single, group = ivf_pair(x, devices, 64)
        single.nprobe = group.nprobe = 8
        params = lambda sel: faiss.SearchParametersIVF(sel=sel, nprobe=8)
        sels = _selectors(n, lambda pos: np.asarray(pos, np.int64) * 7 + 2)
    q = queries(5, 32, 7)
    for sel in sels.values():
        for k in (1, 100):
            same(group.search(q, k, params=params(sel)), single.search(q, k, params=params(sel)))
        for thresh in (0.5, 1e9):  # hits / zero hits
            same(group.range_search(q, thresh, params=params(sel)), single.range_search(q, thresh, params=params(sel)))
    for thresh in (0.5, 1e9):
        same(group.range_search(q, thresh), single.range_search(q, thresh))


@need2
def test_a_shard_without_rows():
    # without a reservation rows fill the first GPU: shard 1 stays empty
    x = int_store(50_000, 32, 41)
    single, group = flat_pair(x, [0, 1], reserve=False)
    assert [sh.ntotal for sh in group._shards] == [50_000, 0]
    q = queries(3, 32, 3)
    for k in (1, 100):
        same(group.search(q, k), single.search(q, k))
    sel = faiss.IDSelectorRange(1, 3000)
    same(group.search(q, 100, params=faiss.SearchParameters(sel=sel)),
         single.search(q, 100, params=faiss.SearchParameters(sel=sel)))
    same(group.range_search(q, 0.5), single.range_search(q, 0.5))
    same(group.reconstruct_batch(np.array([1, 4, 3 * 49_999 + 1])), single.reconstruct_batch(np.array([1, 4, 3 * 49_999 + 1])))


@need2
def test_fallback_merge_gives_the_same_bytes():
    x = int_store(300_000, 64, 51, dup_every=True)
    single, group = flat_pair(x, [0, 1])
    group.index._grp = faiss._Group(group._shards, max_queries=4, max_entries=64)  # every batch below is too big
    for nq, k in ((1, 100), (3, 100), (16, 10), (300, 100)):
        q = queries(nq, 64, 60 + nq)
        same(group.search(q, k), single.search(q, k))


@need2
@pytest.mark.parametrize("path", ["exchange", "fallback"])
def test_dev_search_on_a_busy_side_stream(path):
    x = int_store(400_000, 64, 61, dup_every=True)
    single, group = flat_pair(x, [0, 1])
    if path == "fallback":  # local searches, peer copies of the results and the merge on the caller's stream
        group.index._grp = faiss._Group(group._shards, max_queries=4, max_entries=64)
    L = _capi.lib()
    root = torch.device("cuda", 0)
    side = torch.cuda.Stream(root)
    for nq, k in ((1, 100), (3, 100), (16, 100)):
        qh = queries(nq, 64, 70 + nq)
        q = torch.zeros((nq, 64), dtype=torch.float32, device=root)
        D = torch.empty((nq, k), dtype=torch.float32, device=root)
        I = torch.empty((nq, k), dtype=torch.int64, device=root)
        src = torch.from_numpy(qh).to(root)
        torch.cuda.synchronize(root)
        with torch.cuda.stream(side):
            torch.cuda._sleep(200_000_000)  # keeps `side` busy: the queries below are written after the sleep
            q.copy_(src)
            _capi.check(L.wb_group_search_dev(group._group().g, None, nq, q.data_ptr(), k, 1, D.data_ptr(), I.data_ptr(),
                                              side.cuda_stream))
            q.zero_()  # a later write of the queries on the same stream must not reach the shards' copies
        side.synchronize()
        same((D.cpu().numpy(), I.cpu().numpy()), single.search(qh, k))


@need2
@pytest.mark.parametrize("kind", ["flat", "ivf"])
def test_index_files_are_identical_and_read_back_balanced(tmp_path, kind, monkeypatch):
    x = int_store(120_001, 32, 71, dup_every=True)
    if kind == "flat":
        single, group = flat_pair(x, [0, 1])
    else:
        single, group = ivf_pair(x, [0, 1], 64)
        single.nprobe = group.nprobe = 8
        single.make_direct_map()  # ids are not 0..n-1: the map is refused the same way on both
    f1, f2 = tmp_path / "single.faiss", tmp_path / "group.faiss"
    faiss.write_index(single, str(f1))
    faiss.write_index(group, str(f2))
    assert f1.read_bytes() == f2.read_bytes()
    monkeypatch.setenv("WISE_B200_DEVICES", "0,1")
    back = faiss.read_index(str(f2))
    counts = [sh.ntotal for sh in back._shards]
    assert sum(counts) == x.shape[0] and max(counts) - min(counts) <= 1
    monkeypatch.delenv("WISE_B200_DEVICES")
    ref = faiss.read_index(str(f1))
    if kind == "ivf":
        back.nprobe = ref.nprobe = 8
    q = queries(4, 32, 80)
    for k in (1, 100):
        same(back.search(q, k), ref.search(q, k))


@need2
def test_ivf_train_copies_the_root_centroids():
    x = int_store(60_000, 32, 81)
    idx = faiss.IndexIVFFlat(faiss.IndexFlatIP(32, devices=[0, 1]), 32, 64)
    idx.train(x)
    ref = faiss.IndexIVFFlat(faiss.IndexFlatIP(32, device=0), 32, 64)
    ref.train(x)
    assert np.array_equal(idx.centroids().view(np.uint32), ref.centroids().view(np.uint32))
    c1 = np.empty((64, 32), np.float32)
    _capi.check(_capi.lib().wb_ivf_get_centroids(idx._shards[1]._h, _capi.ptr(c1)))
    assert np.array_equal(c1.view(np.uint32), ref.centroids().view(np.uint32))
    idx.add(x)
    ref.add(x)
    idx.nprobe = ref.nprobe = 4
    q = queries(3, 32, 90)
    same(idx.search(q, 50), ref.search(q, 50))


@need2
def test_errors():
    with pytest.raises(RuntimeError):
        faiss.IndexFlatIP(16, devices=[0, 0])
    a, b = faiss.IndexFlatIP(16, device=0), faiss.IndexFlatIP(32, device=1)
    with pytest.raises(RuntimeError):
        faiss._Group([a, b])
    _, group = flat_pair(int_store(1000, 16, 91), [0, 1])
    with pytest.raises(RuntimeError):
        group.reconstruct_batch(np.array([1, 5]))  # 5 is no id (ids are 3 * position + 1)


@pytest.mark.skipif(_ngpu() < 1, reason="needs a GPU")
def test_one_device_takes_the_single_index_path(monkeypatch):
    monkeypatch.setenv("WISE_B200_DEVICES", "0")
    x = int_store(20_000, 32, 95)
    a = faiss.IndexIDMap(faiss.IndexFlatIP(32))
    assert a._shards is None and a._grp is None
    monkeypatch.delenv("WISE_B200_DEVICES")
    b = faiss.IndexIDMap(faiss.IndexFlatIP(32, device=0))
    ids = np.arange(20_000, dtype=np.int64)
    L = _capi.lib()
    for idx in (a, b):
        idx.reserve(20_000)
        idx.add_with_ids(x, ids)
    q = queries(3, 32, 96)
    same(a.search(q, 10), b.search(q, 10))
    assert L.wb_launch_count(a._h) == L.wb_launch_count(b._h)
