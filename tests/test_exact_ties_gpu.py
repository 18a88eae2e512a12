"""The tie rule, tested exactly: rows come back by score descending and equal scores by lowest insertion position, on
every search path (include/wise_b200.h, DESIGN.md section 5).

The float tests elsewhere excuse any id swap inside a near-tie band, and their data almost never ties.  Here every
entry of every row, query and centroid is a small integer times a power of two, m * 2^-e with |m| <= L and
d * L^2 < 2^22.  Every product and every partial sum is then an integer multiple of 2^-2e below 2^22 in magnitude,
so it is exact in fp32 in any order of accumulation; TF32 holds such an operand exactly (11 significant bits), so
the 3xTF32 lo terms are zero and the one-term filter scores, the exact re-scoring, the CUDA-core FMAs and the fp64
oracle all produce the same float.  The expected (D, I) is unique and every check below is an exact equality with the
oracle (ids, lims, counts, assignments, D by value), while ties are as frequent as the data makes them: at L = 1 a
query's 100th score is shared by 50-100 rows.

Ids are a random permutation of a sparse range, so "lowest id" and "lowest position" pick different rows.

The GPU tests are marked `gpu`; the CPU tests at the end check the data's own claims and the oracle's tie order."""
import ctypes as C
import os
import socket
from contextlib import contextmanager

import numpy as np
import pytest
import torch

from oracle import oracle as O
import range_oracle as R
from wise_b200 import _capi
from wise_b200 import faiss_compat as faiss

gpu = pytest.mark.gpu
MAX_EXACT = 1 << 22  # |integer score| bound below which every fp32 partial sum is exact (24-bit significand)


# ---- data ---------------------------------------------------------------------------------------------------------
def exact_store(n, d, L, e, seed, dup=0, zeros=0, ortho=None):
    """[n, d] float32 rows m * 2^-e, m uniform in [-L, L].  Planted structures (positions returned in a dict):
    dup: one vector copied to that many positions spread over the whole store, position 0 and n - 1 included;
    zeros: that many all-zero rows at random positions;
    ortho: (q, count): `count` random rows made orthogonal to the query q (zero on q's support)."""
    assert 1 <= L <= 2047 and d * L * L < MAX_EXACT, (d, L)
    rng = np.random.default_rng(seed)
    x = np.empty((n, d), np.float32)
    scale = np.float32(2.0 ** -e)
    for r0 in range(0, n, 1 << 16):
        r1 = min(n, r0 + (1 << 16))
        x[r0:r1] = rng.integers(-L, L + 1, size=(r1 - r0, d), dtype=np.int16).astype(np.float32) * scale
    planted = {}
    if dup:
        pos = np.unique(np.linspace(0, n - 1, dup).round().astype(np.int64))
        assert pos[0] == 0 and pos[-1] == n - 1 and pos.size == dup
        x[pos] = x[pos[0]]
        planted["dup"] = pos
    free = np.setdiff1d(np.arange(n), planted.get("dup", []))
    if zeros:
        pos = np.sort(rng.choice(free, zeros, replace=False))
        x[pos] = 0
        planted["zeros"] = pos
    if ortho is not None:
        q, count = ortho
        pos = np.sort(rng.choice(free, count, replace=False))
        x[np.ix_(pos, np.nonzero(q)[0])] = 0
        planted["ortho"] = pos
    return x, planted


def perm_ids(n, seed):
    """A random permutation of the sparse range 3, 10, 17, ...: ids never rise with position."""
    return np.random.default_rng(seed).permutation(n).astype(np.int64) * 7 + 3


def positions_of(ids):
    """id -> insertion position (for messages and for the CPU checks)."""
    ids = np.asarray(ids, np.int64)
    pos = np.full(int(ids.max()) + 1, -1, np.int64)
    pos[ids] = np.arange(ids.size)
    return lambda i: int(pos[i]) if 0 <= i < pos.size else -1


# ---- exact comparisons ----------------------------------------------------------------------------------------------
def assert_exact_topk(D, I, Dr, Ir, ids=None, what=""):
    """I equal and D equal by value (-0.0 == +0.0: order_f32 folds the sign).  The message names the first differing
    (query, rank), both ids, their insertion positions and their scores."""
    D, I, Dr, Ir = (np.asarray(a) for a in (D, I, Dr, Ir))
    assert D.shape == Dr.shape and I.shape == Ir.shape, (D.shape, Dr.shape, I.shape, Ir.shape)
    bad = (I != Ir) | (D != Dr)
    if bad.any():
        q, r = (int(v) for v in np.argwhere(bad)[0])
        pos = positions_of(ids) if ids is not None else (lambda i: int(i))
        raise AssertionError(
            f"{what}: {int(bad.sum())} entries differ in {int(bad.any(1).sum())} queries; first at query {q} rank {r}: "
            f"got id {I[q, r]} (position {pos(I[q, r])}, score {D[q, r]!r}), "
            f"want id {Ir[q, r]} (position {pos(Ir[q, r])}, score {Dr[q, r]!r}); k-th score wanted {Dr[q, -1]!r}")


def assert_exact_range(lims, D, I, ref, ids=None, what=""):
    """lims equal to the fp64 hit counts (scores strictly above thresh), then D (by value) and I entry by entry."""
    lr, Dr, Ir = ref
    lims = np.asarray(lims).astype(np.int64)
    lr = np.asarray(lr).astype(np.int64)
    assert lims.shape == lr.shape, (lims.shape, lr.shape)
    if not np.array_equal(lims, lr):
        q = int(np.nonzero(np.diff(lims) != np.diff(lr))[0][0])
        raise AssertionError(f"{what}: query {q} has {lims[q + 1] - lims[q]} hits, want {lr[q + 1] - lr[q]}")
    D, I = np.asarray(D), np.asarray(I)
    assert D.shape == Dr.shape and I.shape == Ir.shape
    bad = (I != Ir) | (D != Dr)
    if bad.any():
        j = int(np.nonzero(bad)[0][0])
        q = int(np.searchsorted(lims, j, side="right") - 1)
        pos = positions_of(ids) if ids is not None else (lambda i: int(i))
        raise AssertionError(
            f"{what}: {int(bad.sum())} entries differ; first at query {q} entry {j - lims[q]}: got id {I[j]} "
            f"(position {pos(I[j])}, score {D[j]!r}), want id {Ir[j]} (position {pos(Ir[j])}, score {Dr[j]!r})")


# ---- witnesses and device helpers -----------------------------------------------------------------------------------
def gemm_stats(idx):
    a, b = C.c_int64(), C.c_int64()
    _capi.check(_capi.lib().wb_gemm_stats(idx._h, C.byref(a), C.byref(b)))
    return a.value, b.value


def fused(idx):
    return int(_capi.lib().wb_ivf_fused_searches(idx._h))


def launches(idx):
    return int(_capi.lib().wb_launch_count(idx._h))


def scan_plan(idx, nq, k):
    out = (C.c_int32 * 5)()
    _capi.check(_capi.lib().wb_scan_plan(idx._h, nq, k, 0, 0, out))
    return dict(zip(("NQ", "RW", "ck", "nchunks", "stages"), list(out)))


@contextmanager
def env(**kv):
    """Environment switches of the C API (read at every call) for the duration of a block."""
    old = {k: os.environ.get(k) for k in kv}
    os.environ.update({k: str(v) for k, v in kv.items()})
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def k2_search(idx, xq, k, filt=1, params=None):
    """A forced tensor-core search; returns (D, I, epochs, fallbacks) of this call."""
    e0, f0 = gemm_stats(idx)
    with env(WB_GEMM_FORCE=1, WB_GEMM_FILTER=filt):
        D, I = idx.search(xq, k, params=params)
    e1, f1 = gemm_stats(idx)
    return D, I, e1 - e0, f1 - f0


def range_host_and_dev(idx, xq, thresh, flt=None, nprobe=1):
    """wb_range_search and wb_range_search_dev of the same queries: [(lims uint64, D, I)] x 2."""
    L = _capi.lib()
    st = torch.cuda.current_stream().cuda_stream
    q = torch.from_numpy(np.ascontiguousarray(xq)).cuda()
    out = []
    for dev in (False, True):
        lims = np.zeros(len(xq) + 1, np.int64)
        res = C.c_void_p()
        if dev:
            _capi.check(L.wb_range_search_dev(idx._h, flt, len(xq), q.data_ptr(), float(thresh), nprobe,
                                              _capi.ptr(lims), C.byref(res), st))
        else:
            _capi.check(L.wb_range_search(idx._h, flt, len(xq), _capi.ptr(np.ascontiguousarray(xq)), float(thresh),
                                          nprobe, _capi.ptr(lims), C.byref(res)))
        try:
            n = int(lims[-1])
            D, I = np.empty(n, np.float32), np.empty(n, np.int64)
            _capi.check(L.wb_range_result_copy(res, _capi.ptr(D), _capi.ptr(I)))
        finally:
            _capi.check(L.wb_range_result_free(res))
        out.append((lims.astype(np.uint64), D, I))
    return out


def first_k_hits_are_search(lims, Dg, Ig, D, I, k):
    """For every query with at least k hits, its first k hits are search(x, k) exactly; returns how many queries."""
    lims = lims.astype(np.int64)
    big = np.nonzero(np.diff(lims) >= k)[0]
    for i in big:
        a = int(lims[i])
        assert np.array_equal(Ig[a:a + k], I[i]) and np.array_equal(Dg[a:a + k], D[i]), f"query {i}"
    return big.size


def gpu_assign(idx, n):
    """The lists the library assigned rows [0, n) to, read before a search regroups the store."""
    _, _, a = idx._export(0, n, want_assign=True, want_ids=False, want_x=False)
    return a.astype(np.int64)


def ivf_index(cent):
    idx = faiss.IndexIVFFlat(faiss.IndexFlatIP(cent.shape[1]), cent.shape[1], cent.shape[0],
                             faiss.METRIC_INNER_PRODUCT)
    idx.set_centroids(cent)
    return idx


def add_dev(idx, x, ids):
    """wb_add_with_ids_dev from torch-owned device memory."""
    st = torch.cuda.current_stream()
    xd, idd = torch.from_numpy(x).cuda(), torch.from_numpy(ids).cuda()
    _capi.check(_capi.lib().wb_add_with_ids_dev(idx._h, len(x), xd.data_ptr(), idd.data_ptr(), st.cuda_stream))
    st.synchronize()


def add_pinned(idx, x, ids, batch=8192):
    """wb_add_with_ids_pinned in batches over two slots."""
    L = _capi.lib()
    n, d = x.shape
    bufs = []
    try:
        for _ in range(2):
            px, pi = C.c_void_p(), C.c_void_p()
            _capi.check(L.wb_pinned_alloc(batch * d * 4, C.byref(px)))
            bufs.append(px)
            _capi.check(L.wb_pinned_alloc(batch * 8, C.byref(pi)))
            bufs.append(pi)
        for b, r0 in enumerate(range(0, n, batch)):
            r1 = min(n, r0 + batch)
            slot = b % 2
            px, pi = bufs[2 * slot], bufs[2 * slot + 1]
            _capi.check(L.wb_add_slot_wait(idx._h, slot))
            np.ctypeslib.as_array((C.c_float * ((r1 - r0) * d)).from_address(px.value))[:] = x[r0:r1].ravel()
            np.ctypeslib.as_array((C.c_int64 * (r1 - r0)).from_address(pi.value))[:] = ids[r0:r1]
            _capi.check(L.wb_add_with_ids_pinned(idx._h, r1 - r0, px, pi, slot))
        _capi.check(L.wb_sync(idx._h))
    finally:
        for p in bufs:
            _capi.check(L.wb_pinned_free(p))


# ---- flat stores --------------------------------------------------------------------------------------------------
N = 300_000
DUP = 64  # copies of one vector, spread over the store


def _queries(xb, planted, nq, d, L, e, seed):
    """Query 0 is the planted duplicate (its copies tie at the top, so k = 8 / 9 cut through the group), query 3 is
    zero (every row ties at 0: the answer is the first k positions), the others are drawn like the rows."""
    xq = exact_store(nq, d, L, e, seed)[0]
    xq[0] = xb[planted["dup"][0]]
    if nq > 3:
        xq[3] = 0
    return xq


@pytest.fixture(scope="module")
def flat_stores():
    """d -> (index, xb, ids, planted, xq [4], oracle top-2048 of xq): tie-dense L = 1 data, 300000 rows at d = 16, 64
    and 768 (every CTA draws many row groups), 60000 rows at d = 4096 (the chunked scan plan: at d = 2560 only
    batches of 8 or more queries are chunked)."""
    cache = {}

    def get(d):
        if d not in cache:
            n = 60_000 if d == 4096 else N
            xb, planted = exact_store(n, d, 1, 3, 10 + d, dup=DUP, zeros=500)
            ids = perm_ids(n, 20 + d)
            idx = faiss.IndexIDMap(faiss.IndexFlatIP(d))
            idx.add_with_ids(xb, ids)
            xq = _queries(xb, planted, 4, d, 1, 3, 30 + d)
            cache[d] = (idx, xb, ids, planted, xq, O.flat_search(xb, xq, 2048, ids))
        return cache[d]

    yield get
    cache.clear()


# ---- 1. the exactness premise on the tensor cores ------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("filt", [0, 1])
def test_k2_is_exact_on_integer_data(filt):
    """d = 768, L = 7, e = 8 (d * L^2 = 37632): forced K2, with the one-term filter epochs (WB_GEMM_FILTER=1) and with
    3xTF32 in every epoch (0), returns scores equal to the fp64 oracle's, not merely close.  Every other K2 case below
    rests on this."""
    n, d, nq, k = 100_000, 768, 16, 100
    xb, planted = exact_store(n, d, 7, 8, 1, dup=20)
    ids = perm_ids(n, 2)
    idx = faiss.IndexIDMap(faiss.IndexFlatIP(d))
    idx.add_with_ids(xb, ids)
    xq = exact_store(nq, d, 7, 8, 3)[0]
    xq[0] = xb[0]
    D, I, ep, fb = k2_search(idx, xq, k, filt)
    assert ep >= 2 and fb == 0, (ep, fb)
    Dr, Ir = O.flat_search(xb, xq, k, ids)
    assert np.array_equal(D, Dr), f"K2 scores are not exact: max |dD| {float(np.abs(D - Dr).max())}"
    assert_exact_topk(D, I, Dr, Ir, ids, f"K2 d=768 L=7 filter={filt}")


# ---- 2. K1 ----------------------------------------------------------------------------------------------------------
K1_K = [1, 8, 9, 100, 128, 129, 1000, 2048]


@gpu
@pytest.mark.parametrize("d", [16, 64, 768, 4096])
def test_k1_exact(flat_stores, d):
    """nq 1-4 (each NQ instantiation) x k on both sides of the heads merge (k <= 128) and of its sort fallback."""
    idx, xb, ids, planted, xq, (Dr, Ir) = flat_stores(d)
    if d == 4096:
        assert all(scan_plan(idx, nq, k)["nchunks"] > 1 for nq in (1, 4) for k in (1, 2048))
    e0 = gemm_stats(idx)
    for nq in (1, 2, 3, 4):
        for k in K1_K:
            D, I = idx.search(xq[:nq], k)
            assert_exact_topk(D, I, Dr[:nq, :k], Ir[:nq, :k], ids, f"K1 d={d} nq={nq} k={k}")
    assert gemm_stats(idx) == e0
    top = Ir[0][np.isin(Ir[0], ids[planted["dup"]])]  # the data plants what it claims
    assert np.array_equal(top, ids[planted["dup"]]) and Dr[0, 0] == Dr[0, DUP - 1]
    assert np.array_equal(Ir[3], ids[:2048])


@gpu
def test_every_row_identical():
    """300000 copies of one vector: every score ties, so the answer is positions 0..k-1 with one score, on K1 and on
    forced K2 (whose candidate lists overflow and are repaired on K1)."""
    n, d = N, 64
    v = exact_store(1, d, 1, 3, 5)[0][0]
    xb = np.ascontiguousarray(np.broadcast_to(v, (n, d)))
    ids = perm_ids(n, 6)
    idx = faiss.IndexIDMap(faiss.IndexFlatIP(d))
    idx.add_with_ids(xb, ids)
    xq = exact_store(16, d, 1, 3, 7)[0]
    s = (xq.astype(np.float64) @ v.astype(np.float64)).astype(np.float32)

    def check(D, I, k, what):
        Dr = np.broadcast_to(s[:len(D), None], (len(D), k))
        Ir = np.broadcast_to(ids[:k], (len(D), k))
        assert_exact_topk(D, I, Dr, Ir, ids, what)

    for nq in (1, 2, 3, 4):
        for k in (1, 100, 128, 129, 2048):
            check(*idx.search(xq[:nq], k), k, f"identical rows K1 nq={nq} k={k}")
    for k in (100, 2048):
        D, I, ep, fb = k2_search(idx, xq, k)
        print(f"\nidentical rows K2 k={k}: {ep} epochs, {fb} fallbacks")
        assert ep >= 1
        check(D, I, k, f"identical rows K2 k={k}")


# ---- 4. K2 ----------------------------------------------------------------------------------------------------------
K2_NQ = [5, 16, 33, 64, 65, 128, 129, 300, 1024]


@pytest.fixture(scope="module")
def sparse_tie_store():
    """d = 256, L = 3, e = 6: ~500 score levels per query, 7-12 rows tied with the 100th score."""
    n, d = 200_000, 256
    xb, planted = exact_store(n, d, 3, 6, 40, dup=12)
    ids = perm_ids(n, 41)
    idx = faiss.IndexIDMap(faiss.IndexFlatIP(d))
    idx.add_with_ids(xb, ids)
    xq = exact_store(max(K2_NQ), d, 3, 6, 42)[0]
    xq[0] = xb[0]
    return idx, xb, ids, xq, O.flat_search(xb, xq, 100, ids)


@gpu
@pytest.mark.parametrize("filt", [1, 0])
@pytest.mark.parametrize("nq", K2_NQ)
def test_k2_exact(sparse_tie_store, nq, filt):
    """The BN 32/64/128 fold variants, the pair kernel, SS single-block and SS multi-block: K2 itself resolves the ties
    (three or more epochs, no repair)."""
    idx, xb, ids, xq, (Dr, Ir) = sparse_tie_store
    D, I, ep, fb = k2_search(idx, xq[:nq], 100, filt)
    assert ep >= 3 and fb == 0, (ep, fb)
    assert_exact_topk(D, I, Dr[:nq], Ir[:nq], ids, f"K2 nq={nq} filter={filt}")


@pytest.fixture(scope="module")
def big_dup_store():
    """20000 copies of one vector (more than the 4096-row candidate cap) spread over 300000 tie-dense rows."""
    n, d = N, 64
    xb, planted = exact_store(n, d, 1, 3, 50, dup=20_000)
    ids = perm_ids(n, 51)
    idx = faiss.IndexIDMap(faiss.IndexFlatIP(d))
    idx.add_with_ids(xb, ids)
    xq = exact_store(16, d, 1, 3, 52)[0]
    xq[0] = xb[0]
    return idx, xb, ids, planted, xq, O.flat_search(xb, xq, 1000, ids)


@gpu
@pytest.mark.parametrize("filt", [1, 0])
@pytest.mark.parametrize("k", [100, 1000])
def test_k2_overflow_repair_exact(big_dup_store, k, filt):
    """Query 0 ties with 20000 rows.  With the one-term filter epochs every copy passes `score > thr - margin`, an
    epoch collects more candidates than the 4096-row cap and the batch is repaired on K1, exactly: the first k copies
    in position order.  With 3xTF32 in every epoch (WB_GEMM_FILTER=0) the strict `score > thr` drops the later copies
    (they lose the tie to the earlier ones), so K2 resolves the group itself."""
    idx, xb, ids, planted, xq, (Dr, Ir) = big_dup_store
    D, I, ep, fb = k2_search(idx, xq, k, filt)
    assert ep >= 1 and (fb >= 1 if filt else fb == 0), (ep, fb)
    assert_exact_topk(D, I, Dr[:, :k], Ir[:, :k], ids, f"K2 repair k={k} filter={filt}")
    assert np.array_equal(I[0], ids[planted["dup"][:k]])


# ---- 5. incremental adds --------------------------------------------------------------------------------------------
@gpu
def test_incremental_adds_exact():
    """512-row adds (the reference's add loop) into a store that grows: positions run on across the batches."""
    n, d = 60_000, 64
    xb, planted = exact_store(n, d, 1, 3, 60, dup=200, zeros=100)
    ids = perm_ids(n, 61)
    idx = faiss.IndexIDMap(faiss.IndexFlatIP(d))
    for r0 in range(0, n, 512):
        idx.add_with_ids(xb[r0:r0 + 512], ids[r0:r0 + 512])
    assert idx.ntotal == n
    xq = exact_store(64, d, 1, 3, 62)[0]
    xq[0] = xb[0]
    k = 300
    Dr, Ir = O.flat_search(xb, xq, k, ids)
    D, I = idx.search(xq[:4], k)
    assert_exact_topk(D, I, Dr[:4], Ir[:4], ids, "incremental adds K1")
    D, I, ep, fb = k2_search(idx, xq, k)
    assert ep >= 2 and fb == 0, (ep, fb)
    assert_exact_topk(D, I, Dr, Ir, ids, "incremental adds K2")
    assert np.array_equal(I[0, :200], ids[planted["dup"]])


# ---- 6. zero rows and rows orthogonal to the query ------------------------------------------------------------------
@gpu
def test_zero_scores_at_the_boundary():
    """Queries supported on 8 coordinates over a store in which all but 3000 rows are orthogonal to them (and 1000 are
    zero): ~1200 rows score above 0, ~299000 score exactly 0 (+0.0 or -0.0), so the k = 2048 boundary falls among the
    zeros, which must come in position order."""
    n, d, k = N, 64, 2048
    q = np.zeros(d, np.float32)
    q[:8] = 0.125
    q2 = q.copy()
    q2[1:8:2] = -0.125
    xb, planted = exact_store(n, d, 1, 3, 70, zeros=1000, ortho=(q, n - 3000))
    ids = perm_ids(n, 71)
    idx = faiss.IndexIDMap(faiss.IndexFlatIP(d))
    idx.add_with_ids(xb, ids)
    xq = np.concatenate([np.stack([q, q2]), exact_store(14, d, 1, 3, 72)[0]])
    s = xq[:2].astype(np.float64) @ xb.astype(np.float64).T
    assert np.all((s > 0).sum(1) < k - 200) and np.all((s >= 0).sum(1) > k + 200)
    Dr, Ir = O.flat_search(xb, xq, k, ids)
    D, I = idx.search(xq[:2], k)
    assert_exact_topk(D, I, Dr[:2], Ir[:2], ids, "zero boundary K1")
    D, I, ep, fb = k2_search(idx, xq, k)
    print(f"\nzero boundary K2: {ep} epochs, {fb} fallbacks")
    assert ep >= 1
    assert_exact_topk(D, I, Dr, Ir, ids, "zero boundary K2")


# ---- IVF ------------------------------------------------------------------------------------------------------------
def exact_centroids(nlist, d, seed):
    """Integer centroids (L = 1, e = 3) with a duplicated pair (9, 41) and two zero centroids (62, 63): rows and queries
    tie between the lists of each pair for every query."""
    c = exact_store(nlist, d, 1, 3, seed)[0]
    if nlist >= 64:
        c[41] = c[9]
        c[62:64] = 0
    return c


NI, DI, NLIST = 200_000, 64, 64


@pytest.fixture(scope="module")
def ivf_data():
    xb, planted = exact_store(NI, DI, 1, 3, 80, dup=50, zeros=200)
    ids = perm_ids(NI, 81)
    cent = exact_centroids(NLIST, DI, 82)
    xq = exact_store(64, DI, 1, 3, 83)[0]
    xq[0] = xb[0]
    sc = np.sort(xq.astype(np.float64) @ cent.astype(np.float64).T, axis=1)[:, ::-1]
    # the smallest nprobe >= 4 at which the boundary centroid of query 0 is tied with the next one
    np_tie = next(p for p in range(4, NLIST) if sc[0, p - 1] == sc[0, p])
    return xb, ids, cent, xq, np_tie, O.ivf_assign(xb, cent)


@pytest.fixture(scope="module")
def ivf_indices(ivf_data):
    """contiguous -> index: the store regrouped list by list (1) or left in place behind a slot permutation (0)."""
    xb, ids, cent, xq, np_tie, assign = ivf_data
    out = {}
    for contiguous in (1, 0):
        idx = ivf_index(cent)
        idx.add_with_ids(xb, ids)
        with env(WB_IVF_CONTIGUOUS=contiguous):
            _capi.check(_capi.lib().wb_ivf_finalize(idx._h))
        out[contiguous] = idx
    return out


def _ties_in_assignment(x, cent):
    s = x.astype(np.float64) @ cent.astype(np.float64).T
    return float(((s == s.max(1, keepdims=True)).sum(1) >= 2).mean())


# ---- 7. add-time assignment -----------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("how", ["host", "dev", "pinned"])
@pytest.mark.parametrize("n,nlist,force", [(200_000, 64, False),  # assignment GEMM (n >= 1024, nlist >= 64)
                                           (50_000, 32, False),   # K1 over the centroids (nlist < 64)
                                           (1000, 64, False),     # K1 (n < 1024)
                                           (1000, 2048, True)])   # K2 over the centroids (3xTF32 every epoch)
def test_add_assignment_exact(n, nlist, force, how):
    """Each row goes to its max-inner-product list, ties to the lowest list, on every assignment kernel add picks
    (assign_rows in capi.cu): the ARGMAX epilogue of the assignment GEMM, or the k = 1 search over the centroids."""
    d = DI
    x = exact_store(n, d, 1, 3, 90 + nlist)[0]
    cent = exact_centroids(nlist, d, 91 + nlist)
    if nlist == 2048:
        cent[1000:1100] = cent[:100]
    ids = perm_ids(n, 92)
    want = O.ivf_assign(x, cent)
    tied = _ties_in_assignment(x, cent)
    assert tied > 0.01, tied
    idx = ivf_index(cent)
    e0 = gemm_stats(idx)
    with env(WB_GEMM_FORCE=int(force)):
        if how == "host":
            idx.add_with_ids(x, ids)
        elif how == "dev":
            add_dev(idx, x, ids)
        else:
            add_pinned(idx, x, ids)
    e1 = gemm_stats(idx)
    assert (e1[0] > e0[0]) == (force or (n >= 1024 and nlist >= 64)), (e0, e1)  # K2 or the assignment GEMM
    got = gpu_assign(idx, n)
    bad = np.nonzero(got != want)[0]
    assert bad.size == 0, (f"{bad.size} rows ({tied:.0%} of rows tie): row {bad[0]} in list {got[bad[0]]}, "
                           f"want {want[bad[0]]}")


# ---- 8. IVF search --------------------------------------------------------------------------------------------------
def _ivf_oracle(ivf_data, nq, nprobe, k, xb=None, ids=None, assign=None):
    xb0, ids0, cent, xq, _, assign0 = ivf_data
    xb = xb0 if xb is None else xb
    return O.ivf_search(xb, ids0 if ids is None else ids, assign0 if assign is None else assign, cent, xq[:nq], k,
                        nprobe)


@gpu
@pytest.mark.parametrize("contiguous", [1, 0])
@pytest.mark.parametrize("fuse", [1, 0])
def test_ivf_small_batches_exact(ivf_data, ivf_indices, contiguous, fuse):
    """nq 1-4: the coarse step fused into the list scan (radix selection of (score, ~list)) or as its own launch;
    nprobe 1, one whose boundary centroid ties, and every list; k 10, 100, 1000."""
    xb, ids, cent, xq, np_tie, assign = ivf_data
    idx = ivf_indices[contiguous]
    nfused = {10: 0, 100: 0, 1000: 0}
    for nprobe in (1, np_tie, NLIST):
        Dr, Ir = _ivf_oracle(ivf_data, 4, nprobe, 1000)
        for nq in (1, 2, 3, 4):
            for k in (10, 100, 1000):
                f0 = fused(idx)
                with env(WB_IVF_FUSE_COARSE=fuse, WB_IVF_LISTMAJOR=0):
                    D, I = idx.search(xq[:nq], k, params=faiss.SearchParametersIVF(nprobe=nprobe))
                nfused[k] += fused(idx) - f0
                assert_exact_topk(D, I, Dr[:nq, :k], Ir[:nq, :k], ids,
                                  f"IVF contiguous={contiguous} fuse={fuse} nprobe={nprobe} nq={nq} k={k}")
    print(f"\nIVF nq 1-4 contiguous={contiguous} fuse={fuse}: fused searches by k {nfused}")
    # every k = 10 search takes the fused launch when allowed (larger k may not fit the fused tail's scratch)
    assert nfused[10] == (12 if fuse else 0) and (fuse or sum(nfused.values()) == 0), nfused


@gpu
@pytest.mark.parametrize("contiguous,listmajor", [(1, 1), (1, 0), (0, 0)])
def test_ivf_batches_exact(ivf_data, ivf_indices, contiguous, listmajor):
    """64 queries: list-major K5b (the shared atomicMax threshold keeps rows that tie with it) and query-major K5; the
    list-major scan needs the store grouped by list."""
    xb, ids, cent, xq, np_tie, assign = ivf_data
    idx = ivf_indices[contiguous]
    nq = len(xq)
    for nprobe in (1, np_tie, NLIST):
        Dr, Ir = _ivf_oracle(ivf_data, nq, nprobe, 1000)
        for k in (10, 100, 1000):
            l0 = launches(idx)
            with env(WB_IVF_LISTMAJOR=listmajor):
                D, I = idx.search(xq, k, params=faiss.SearchParametersIVF(nprobe=nprobe))
            lm = launches(idx) - l0
            if listmajor:  # the witness: list-major makes more launches than query-major (test_limits_gpu.py)
                l0 = launches(idx)
                with env(WB_IVF_LISTMAJOR=0):
                    idx.search(xq, k, params=faiss.SearchParametersIVF(nprobe=nprobe))
                qm = launches(idx) - l0
                print(f"\nIVF batch nprobe={nprobe} k={k}: launches list-major {lm}, query-major {qm}")
                assert k > 100 or lm > qm, (lm, qm)  # (k = 1000 may not fit the list-major plan)
            assert_exact_topk(D, I, Dr[:, :k], Ir[:, :k], ids,
                              f"IVF batch contiguous={contiguous} listmajor={listmajor} nprobe={nprobe} k={k}")


@gpu
def test_ivf_add_after_search_exact(ivf_data):
    """Rows added after the first search (which regrouped the store) keep their insertion positions."""
    xb, ids, cent, xq, np_tie, assign = ivf_data
    idx = ivf_index(cent)
    idx.add_with_ids(xb, ids)
    idx.search(xq[:1], 10)
    more, _ = exact_store(20_000, DI, 1, 3, 84)
    more[::997] = xb[:21]  # copies of early rows: they tie with them and must come after them
    ids2 = np.concatenate([ids, perm_ids(20_000, 85) + 7 * NI])
    xb2 = np.concatenate([xb, more])
    idx.add_with_ids(more, ids2[NI:])
    a2 = np.concatenate([assign, O.ivf_assign(more, cent)])
    for nq, listmajor in ((4, 0), (64, 1)):
        for nprobe in (np_tie, NLIST):
            Dr, Ir = _ivf_oracle(ivf_data, nq, nprobe, 100, xb2, ids2, a2)
            with env(WB_IVF_LISTMAJOR=listmajor):
                D, I = idx.search(xq[:nq], 100, params=faiss.SearchParametersIVF(nprobe=nprobe))
            assert_exact_topk(D, I, Dr, Ir, ids2, f"IVF after add nq={nq} nprobe={nprobe}")


@gpu
def test_ivf_k2_coarse_exact():
    """20000 lists: the coarse step of a 256-query batch runs on K2 (3xTF32 over the centroids, exact here)."""
    n, d, nlist, nq, nprobe, k = 100_000, DI, 20_000, 256, 16, 10
    xb = exact_store(n, d, 1, 3, 100, dup=30)[0]
    ids = perm_ids(n, 101)
    cent = exact_store(nlist, d, 1, 3, 102)[0]
    cent[10_000:10_500] = cent[:500]
    xq = exact_store(nq, d, 1, 3, 103)[0]
    idx = ivf_index(cent)
    idx.add_with_ids(xb, ids)
    assign = gpu_assign(idx, n)
    assert np.array_equal(assign, O.ivf_assign(xb, cent))
    e0 = gemm_stats(idx)
    with env(WB_GEMM_FORCE=1):
        D, I = idx.search(xq, k, params=faiss.SearchParametersIVF(nprobe=nprobe))
    e1 = gemm_stats(idx)
    assert e1[0] > e0[0] and e1[1] == e0[1], (e0, e1)
    Dr, Ir = O.ivf_search(xb, ids, assign, cent, xq, k, nprobe)
    assert_exact_topk(D, I, Dr, Ir, ids, "IVF K2 coarse")


# ---- 9. filtered search ---------------------------------------------------------------------------------------------
def _selectors(ids, seed):
    """name -> (selector, kept positions): Batch, Range and Not of each, selecting 1/2 (mask path) and 1/64 (the
    compact path of a flat store: under 1/8)."""
    n = ids.size
    rng = np.random.default_rng(seed)
    srt = np.sort(ids)
    half = rng.choice(ids, n // 2, replace=False)
    most = rng.choice(ids, n - n // 64, replace=False)
    few = rng.choice(ids, n // 64, replace=False)
    r_half = (int(srt[n // 4]), int(srt[3 * n // 4]))
    r_few = (int(srt[n // 3]), int(srt[n // 3 + n // 64]))
    sels = {
        "batch_half": (faiss.IDSelectorBatch(half), np.isin(ids, half)),
        "batch_few": (faiss.IDSelectorBatch(few), np.isin(ids, few)),
        "range_half": (faiss.IDSelectorRange(*r_half), (ids >= r_half[0]) & (ids < r_half[1])),
        "range_few": (faiss.IDSelectorRange(*r_few), (ids >= r_few[0]) & (ids < r_few[1])),
        "not_batch_few": (faiss.IDSelectorNot(faiss.IDSelectorBatch(most)), ~np.isin(ids, most)),
        "not_range_half": (faiss.IDSelectorNot(faiss.IDSelectorRange(*r_half)), ~((ids >= r_half[0]) & (ids < r_half[1]))),
    }
    out = {}
    for name, (sel, keep) in sels.items():
        keep = np.nonzero(keep)[0]
        if name.endswith("few"):
            assert keep.size * 8 < n, name
        else:
            assert abs(keep.size - n // 2) <= 1, name
        out[name] = (sel, keep)
    return out


SEL_NAMES = ["batch_half", "batch_few", "range_half", "range_few", "not_batch_few", "not_range_half"]


@gpu
@pytest.mark.parametrize("sel", SEL_NAMES)
def test_filtered_flat_exact(flat_stores, sel):
    """K1 (4 queries) and forced K2 (64 queries) over the selected rows: the oracle over xb[keep] (ties by original
    position, since keep is in position order)."""
    idx, xb, ids, planted, xq4, _ = flat_stores(64)
    s, keep = _selectors(ids, 110)[sel]
    xq = np.concatenate([xq4, exact_store(60, 64, 1, 3, 111)[0]])
    k = 100
    Dr, Ir = O.flat_search(xb[keep], xq, k, ids[keep])
    params = faiss.SearchParameters(sel=s)
    D, I = idx.search(xq[:4], k, params=params)
    assert_exact_topk(D, I, Dr[:4], Ir[:4], ids, f"filtered K1 {sel}")
    D, I, ep, fb = k2_search(idx, xq, k, params=params)
    assert ep >= 1, ep
    assert_exact_topk(D, I, Dr, Ir, ids, f"filtered K2 {sel}")


@gpu
@pytest.mark.parametrize("sel", ["batch_half", "range_few", "not_range_half"])
def test_filtered_ivf_exact(ivf_data, ivf_indices, sel):
    xb, ids, cent, xq, np_tie, assign = ivf_data
    idx = ivf_indices[1]
    s, keep = _selectors(ids, 112)[sel]
    k = 100
    for nq, listmajor in ((4, 0), (64, 1)):
        Dr, Ir = O.ivf_search(xb[keep], ids[keep], assign[keep], cent, xq[:nq], k, np_tie)
        with env(WB_IVF_LISTMAJOR=listmajor):
            D, I = idx.search(xq[:nq], k, params=faiss.SearchParametersIVF(sel=s, nprobe=np_tie))
        assert_exact_topk(D, I, Dr, Ir, ids, f"filtered IVF {sel} nq={nq}")


# ---- 10. range search -----------------------------------------------------------------------------------------------
def _levels(s, lo, hi):
    """A score level present in row 0 of `s` with between lo and hi scores strictly above it, and the next lower
    level present."""
    lv = np.unique(s[0])[::-1]
    above = np.array([(s[0] > v).sum() for v in lv])
    i = int(np.nonzero((above >= lo) & (above <= hi))[0][0])
    return np.float32(lv[i]), np.float32(lv[i + 1])


def _check_range(idx, xq, ref_fn, thresh, ids, what, nprobe=1, k=100):
    """Host and device range results equal the oracle's; the first k hits of a query with at least k are search(x, k).
    Returns the number of hits."""
    ref = ref_fn(thresh)
    out = range_host_and_dev(idx, xq, thresh, nprobe=nprobe)
    for (lims, Dg, Ig), via in zip(out, ("host", "dev")):
        assert_exact_range(lims, Dg, Ig, ref, ids, f"{what} thresh={thresh!r} {via}")
    D, I = idx.search(xq, k) if nprobe == 1 else idx.search(xq, k, params=faiss.SearchParametersIVF(nprobe=nprobe))
    assert first_k_hits_are_search(*out[0], D, I, k) >= 1
    return int(ref[0][-1])


@gpu
@pytest.mark.parametrize("path", ["k1", "k2"])
def test_range_flat_exact(flat_stores, path):
    """thresh equal to a score level present in the data (the strict > drops the rows at it) and one level below."""
    idx, xb, ids, planted, xq4, _ = flat_stores(64)
    xq = xq4[:3] if path == "k1" else np.concatenate([xq4[:3], exact_store(61, 64, 1, 3, 120)[0]])
    s = xq[:1].astype(np.float64) @ xb.astype(np.float64).T
    levels = _levels(s, 1000, 4000)
    with env(WB_GEMM_FORCE=int(path == "k2")):
        for t in levels:
            e0 = gemm_stats(idx)
            hits = _check_range(idx, xq, lambda t: R.range_search(xb, xq, t, ids), t, ids, f"range {path}")
            assert (gemm_stats(idx)[0] > e0[0]) == (path == "k2")
            print(f"\nrange {path} thresh={t}: {hits} hits")


@gpu
def test_range_ivf_exact(ivf_data, ivf_indices):
    xb, ids, cent, xq, np_tie, assign = ivf_data
    idx = ivf_indices[1]
    xq = xq[:4]
    s = xq[:1].astype(np.float64) @ xb.astype(np.float64).T
    for t in _levels(s, 300, 2000):
        _check_range(idx, xq, lambda t: R.ivf_range_search(xb, ids, assign, cent, xq, t, np_tie), t, ids,
                     "range IVF", nprobe=np_tie, k=10)


# ---- 11. sharded merges ---------------------------------------------------------------------------------------------
def _cuts(n, P):
    """P contiguous parts of [0, n), one empty and one of a single row."""
    return {2: [0, n - 1, n], 3: [0, 1, 1, n],
            8: [0, 37_000, 37_000, 37_001, 100_000, 150_000, 200_000, 250_000, n]}[P]


@gpu
@pytest.mark.parametrize("P", [2, 3, 8])
def test_sharded_merges_exact(flat_stores, P):
    """wb_merge_topk_dev of the parts' wb_search_dev results (K1 and forced K2 on every part) and wb_range_merge_dev of
    their range results equal the oracle over the whole store."""
    from wise_b200.sharded import _cuda_local_range_search, _cuda_range_merge
    idx, xb, ids, planted, xq4, _ = flat_stores(64)
    n = xb.shape[0]
    cuts = _cuts(n, P)
    parts = []
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        p = faiss.IndexIDMap(faiss.IndexFlatIP(64))
        if hi > lo:
            p.add_with_ids(xb[lo:hi], ids[lo:hi])
        parts.append(p)
    L = _capi.lib()
    st = torch.cuda.current_stream().cuda_stream
    xq = np.concatenate([xq4, exact_store(12, 64, 1, 3, 130)[0]])
    k = 1000
    Dr, Ir = O.flat_search(xb, xq, k, ids)
    for nq, force in ((4, 0), (16, 1)):
        q = torch.from_numpy(xq[:nq]).cuda()
        Dp = torch.empty(P, nq, k, device="cuda")
        Ip = torch.empty(P, nq, k, dtype=torch.int64, device="cuda")
        with env(WB_GEMM_FORCE=force):
            for r, p in enumerate(parts):
                _capi.check(L.wb_search_dev(p._h, nq, q.data_ptr(), k, 1, Dp[r].data_ptr(), Ip[r].data_ptr(), st))
        Dm = torch.empty(nq, k, device="cuda")
        Im = torch.empty(nq, k, dtype=torch.int64, device="cuda")
        _capi.check(L.wb_merge_topk_dev(0, nq, k, P, Dp.data_ptr(), Ip.data_ptr(), Dm.data_ptr(), Im.data_ptr(), st))
        torch.cuda.synchronize()
        assert_exact_topk(Dm.cpu().numpy(), Im.cpu().numpy(), Dr[:nq], Ir[:nq], ids, f"merge_topk P={P} nq={nq}")
    xq = xq[:3]
    s = xq[:1].astype(np.float64) @ xb.astype(np.float64).T
    q = torch.from_numpy(xq).cuda()
    for t in _levels(s, 1000, 4000):
        local = [_cuda_local_range_search(p, q, float(t), 1) for p in parts]
        lims_parts = torch.stack([lm for lm, _, _ in local])
        stride = max(1, int(lims_parts[:, -1].max()))
        Dp = torch.full((P, stride), float("nan"), device="cuda")
        Ip = torch.full((P, stride), -7, dtype=torch.int64, device="cuda")
        for r, (lm, Dl, Il) in enumerate(local):
            Dp[r, :Dl.shape[0]] = Dl
            Ip[r, :Il.shape[0]] = Il
        lims = lims_parts.sum(dim=0)
        Dm, Im = _cuda_range_merge(lims_parts, Dp, Ip, lims)
        torch.cuda.synchronize()
        assert_exact_range(lims.numpy(), Dm.cpu().numpy(), Im.cpu().numpy(), R.range_search(xb, xq, t, ids), ids,
                           f"range merge P={P} thresh={t!r}")


def _two_gpu_data():
    xb, planted = exact_store(120_000, 64, 1, 3, 140, dup=DUP, zeros=300)
    ids = perm_ids(len(xb), 141)
    xq = exact_store(16, 64, 1, 3, 142)[0]
    xq[0] = xb[0]
    s = xq[:1].astype(np.float64) @ xb.astype(np.float64).T
    return xb, ids, xq, _levels(s, 1000, 4000)[0]


def _two_gpu_worker(rank, world, port, out, mode):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), WISE_B200_EXCHANGE=mode,
                      WISE_B200_DEVICE=str(rank))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from wise_b200.sharded import ShardedIndex, shard_range
        xb, ids, xq, t = _two_gpu_data()
        lo, hi = shard_range(len(xb), rank, world)
        idx = faiss.IndexIDMap(faiss.IndexFlatIP(64, device=rank))
        idx.add_with_ids(xb[lo:hi], ids[lo:hi])
        sh = ShardedIndex(idx)
        res = {}
        for nq, k in ((4, 100), (4, 2048), (16, 100)):
            res[f"D{nq}_{k}"], res[f"I{nq}_{k}"] = sh.search(xq[:nq], k)
        res["lims"], res["rD"], res["rI"] = sh.range_search(xq[:4], t)
        np.savez(os.path.join(out, f"{mode}_r{rank}.npz"), **res)
    finally:
        dist.destroy_process_group()


@gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("mode", ["peer", "nccl"])
def test_two_gpu_sharded_exact(tmp_path, mode):
    import torch.multiprocessing as mp
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_two_gpu_worker, args=(2, port, str(tmp_path), mode), nprocs=2, join=True)
    xb, ids, xq, t = _two_gpu_data()
    Dr, Ir = O.flat_search(xb, xq, 2048, ids)
    for r in (0, 1):
        res = np.load(tmp_path / f"{mode}_r{r}.npz")
        for nq, k in ((4, 100), (4, 2048), (16, 100)):
            assert_exact_topk(res[f"D{nq}_{k}"], res[f"I{nq}_{k}"], Dr[:nq, :k], Ir[:nq, :k], ids,
                              f"sharded {mode} rank {r} nq={nq} k={k}")
        assert_exact_range(res["lims"], res["rD"], res["rI"], R.range_search(xb, xq[:4], t, ids), ids,
                           f"sharded range {mode} rank {r}")


# ---- 12. k-means pieces ---------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("n", [50_000, 1000])
def test_kmeans_pieces_exact(n):
    """Assignment (3xTF32 and plain TF32 at n >= 1024, the CUDA-core scan below) equals the fp64 argmax with ties to
    the lowest list; the objective is the fp64 sum; the per-list sums and counts are the fp64 ones.  TF32 holds these
    operands exactly, so the fast assignment's 2e-3 band does not apply."""
    d, nlist = DI, 300
    x = exact_store(n, d, 1, 3, 150)[0]
    cent = exact_centroids(nlist, d, 151)
    cent[200:260] = cent[100:160]
    want = O.ivf_assign(x, cent)
    assert _ties_in_assignment(x, cent) > 0.01
    best = (x.astype(np.float64) * cent[want].astype(np.float64)).sum(1)
    idx = ivf_index(cent)
    L = _capi.lib()
    st = torch.cuda.current_stream().cuda_stream
    xd = torch.from_numpy(x).cuda()
    for fn in (L.wb_kmeans_assign_dev, L.wb_kmeans_assign_fast_dev):
        assign = torch.full((n,), -1, dtype=torch.int32, device="cuda")
        obj = C.c_double(0)
        _capi.check(fn(idx._h, n, xd.data_ptr(), assign.data_ptr(), C.byref(obj), st))
        torch.cuda.synchronize()
        got = assign.cpu().numpy().astype(np.int64)
        bad = np.nonzero(got != want)[0]
        assert bad.size == 0, f"{fn.__name__}: {bad.size} rows; row {bad[0]} in {got[bad[0]]}, want {want[bad[0]]}"
        assert obj.value == best.sum(), (fn.__name__, obj.value, best.sum())
    sums = torch.empty(nlist, d, device="cuda")
    counts = torch.empty(nlist, dtype=torch.int64, device="cuda")
    _capi.check(L.wb_kmeans_accumulate_dev(idx._h, n, xd.data_ptr(), assign.data_ptr(), sums.data_ptr(),
                                           counts.data_ptr(), st))
    torch.cuda.synchronize()
    ref = np.zeros((nlist, d), np.float64)
    np.add.at(ref, want, x.astype(np.float64))
    assert np.array_equal(counts.cpu().numpy(), np.bincount(want, minlength=nlist))
    assert np.array_equal(sums.cpu().numpy().astype(np.float64), ref)


# ---- CPU: the data's claims and the oracle's tie order ---------------------------------------------------------------
REGIMES = [(16, 1, 3), (64, 1, 3), (256, 3, 6), (768, 7, 8), (768, 1, 3), (4096, 1, 3)]


@pytest.mark.parametrize("d,L,e", REGIMES)
def test_exact_store_products_are_exact(d, L, e):
    """Every regime the GPU tests use: entries are m * 2^-e with |m| <= L, and fp32 xq @ xb.T (any BLAS order) equals
    the fp64 product rounded once."""
    xb, planted = exact_store(3000, d, L, e, 1, dup=10, zeros=5)
    m = xb * np.float32(2.0 ** e)
    assert np.array_equal(m, np.round(m)) and np.abs(m).max() == L
    assert np.all(xb[planted["dup"]] == xb[0]) and not xb[planted["zeros"]].any()
    xq = exact_store(40, d, L, e, 2)[0]
    s32 = xq @ xb.T
    s64 = (xq.astype(np.float64) @ xb.astype(np.float64).T)
    assert np.array_equal(s32, s64.astype(np.float32)) and np.array_equal(s64, s64.astype(np.float32))
    with pytest.raises(AssertionError):
        exact_store(10, 4096, 33, 0, 1)  # d * L^2 >= 2^22


def test_exact_store_orthogonal_rows():
    q = np.zeros(64, np.float32)
    q[:8] = 0.125
    xb, planted = exact_store(5000, 64, 1, 3, 3, ortho=(q, 4000))
    assert np.all(xb[planted["ortho"]] @ q == 0)


def test_oracle_orders_a_tie_group_by_position_at_the_boundary():
    """A planted group of 64 copies with permuted ids: O.flat_search returns them in position order, and the k = 9
    boundary cuts the group after its 9 lowest positions, not its 9 lowest ids."""
    n = 20_000
    xb, planted = exact_store(n, 64, 1, 3, 4, dup=64)
    ids = perm_ids(n, 5)
    xq = xb[:1].copy()
    D, I = O.flat_search(xb, xq, 9, ids, chunk=777)
    grp = planted["dup"]
    assert np.array_equal(I[0], ids[grp[:9]]) and np.all(D[0] == D[0, 0])
    assert not np.array_equal(np.sort(ids[grp])[:9], I[0])  # lowest ids would pick other rows
    D2, I2 = O.flat_search(xb, xq, 100, ids)
    assert np.array_equal(I2[0, :64], ids[grp])
    with pytest.raises(AssertionError, match="position"):
        assert_exact_topk(D, I[:, ::-1], D, I, ids, "swap")
