"""Search and range search at the C API's internal size limits (wise_b200/csrc/capi.cu): the scan launch split at
kMaxGridY query groups, the K2 query chunks of 65536, the range chunks of kRangeMaxQ queries and the 2^28-hit budget,
the chunked scan plan of very wide rows, the tensor-core coarse quantizer of large IVF indices and the bound of the
list-major IVF scan.  Every case compares every query with an fp64 reference, re-searches the queries on both sides of
each boundary alone (bit for bit), and asserts a witness that it took the path it targets (launch counts, K2 epochs,
fused coarse searches, the scan plan).

The large batches use `topk_fp64` / `ivf_topk_fp64`: fp64 matmul + topk in torch on the GPU (cuBLAS, independent of
this library), with the oracle's rule - the fp64 score rounded once to fp32, ties by insertion position."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import oracle as O
from range_oracle import check as range_check
from wise_b200 import _capi
from wise_b200 import faiss_compat as faiss

pytestmark = pytest.mark.gpu

GRID_Y = 32768      # kMaxGridY: query groups per scan launch
K2_MAX_Q = 65536    # queries per K2 call (run_flat_any)
RANGE_MAX_Q = 32768  # kRangeMaxQ: queries per range chunk
BUDGET = 1 << 28    # kRangeBudgetHits: hits per range chunk
BAND = {False: O.NEAR_TIE_BAND, True: 4e-6}  # scan path, tensor-core path


# ---- fp64 references ------------------------------------------------------------------------------------------------
def _order(v, i):
    """Rows of (score, position) pairs sorted by score descending, then position ascending."""
    i, o = torch.sort(i, dim=1)
    v = torch.gather(v, 1, o)
    v, o = torch.sort(v, dim=1, descending=True, stable=True)
    return v, torch.gather(i, 1, o)


def topk_fp64(xb, xq, k, ids=None, device="cuda"):
    """IndexFlatIP(+IndexIDMap).search in fp64, query chunk by query chunk: what O.flat_search computes."""
    xb_t = torch.as_tensor(np.ascontiguousarray(xb, np.float32), device=device).double()
    N, n = xb_t.shape[0], len(xq)
    D = np.full((n, k), O.NEG_FLT_MAX, np.float32)
    I = np.full((n, k), -1, np.int64)
    kk = min(k, N)
    if kk == 0:
        return D, I
    chunk = max(1, min(8192, (1 << 27) // N))
    for q0 in range(0, n, chunk):
        q = torch.as_tensor(np.ascontiguousarray(xq[q0:q0 + chunk], np.float32), device=device).double()
        s = (q @ xb_t.T).float()
        v, i = torch.topk(s, kk, dim=1)
        # a row tied with the k-th score may have lost to a later one: take every tied row, then cut by position
        extra = int((s >= v[:, -1:]).sum(1).max()) - kk
        if extra > 0:
            v, i = torch.topk(s, min(N, kk + extra), dim=1)
        v, i = _order(v, i)
        D[q0:q0 + len(q), :kk] = v[:, :kk].cpu().numpy()
        I[q0:q0 + len(q), :kk] = i[:, :kk].cpu().numpy()
    if ids is not None:
        I[:, :kk] = np.asarray(ids, np.int64)[I[:, :kk]]
    return D, I


def coarse_fp64(cent, xq, nprobe, device="cuda"):
    """The fp64 coarse quantizer: probes [n, nprobe] and the gap between the nprobe-th and (nprobe+1)-th centroid
    score of each query (inf when every list is probed)."""
    c = torch.as_tensor(cent, device=device).double()
    q = torch.as_tensor(np.ascontiguousarray(xq, np.float32), device=device).double()
    probes, gaps = [], []
    for q0 in range(0, len(xq), 4096):
        s = q[q0:q0 + 4096] @ c.T
        m = min(nprobe + 1, c.shape[0])
        v, i = torch.topk(s, m, dim=1)
        v, i = _order(v, i)
        probes.append(i[:, :nprobe].cpu().numpy())
        gaps.append((v[:, nprobe - 1] - v[:, nprobe]).cpu().numpy() if m > nprobe else np.full(len(s), np.inf))
    return np.concatenate(probes), np.concatenate(gaps)


def ivf_topk_fp64(xb, ids, assign, probes, xq, k, device="cuda"):
    """IndexIVFFlat.search in fp64 over the rows of the given probed lists (one row of `probes` per query)."""
    xb_t = torch.as_tensor(np.ascontiguousarray(xb, np.float32), device=device).double()
    a = torch.as_tensor(np.asarray(assign, np.int64), device=device)
    nlist = int(max(int(assign.max()), int(probes.max()))) + 1
    N, n = xb_t.shape[0], len(xq)
    D = np.full((n, k), O.NEG_FLT_MAX, np.float32)
    I = np.full((n, k), -1, np.int64)
    kk = min(k, N)
    chunk = max(1, min(4096, (1 << 26) // N))
    for q0 in range(0, n, chunk):
        q = torch.as_tensor(np.ascontiguousarray(xq[q0:q0 + chunk], np.float32), device=device).double()
        pr = torch.as_tensor(probes[q0:q0 + chunk], device=device)
        probed = torch.zeros(len(q), nlist, dtype=torch.bool, device=device).scatter_(1, pr, True)
        ok = probed[:, a]
        s = (q @ xb_t.T).float().masked_fill(~ok, float("-inf"))
        v, i = torch.topk(s, kk, dim=1)
        kth = v[:, -1:]
        extra = int(((s >= kth) & ok).sum(1).max()) - kk
        if extra > 0:
            v, i = torch.topk(s, min(N, kk + extra), dim=1)
        v, i = _order(v, i)
        v, i = v[:, :kk], i[:, :kk]
        pad = ~torch.isfinite(v)
        D[q0:q0 + len(q), :kk] = v.masked_fill(pad, float(O.NEG_FLT_MAX)).cpu().numpy()
        I[q0:q0 + len(q), :kk] = np.where(pad.cpu().numpy(), -1, np.asarray(ids, np.int64)[i.cpu().numpy()])
    return D, I


# ---- witnesses and helpers ------------------------------------------------------------------------------------------
def scan_plan(idx, nq, k, gather=False, nprobe=0):
    """plan_scan's choice (wb_scan_plan): NQ, RW, ck, nchunks, stages."""
    out = (C.c_int32 * 5)()
    _capi.check(_capi.lib().wb_scan_plan(idx._h, nq, k, int(gather), nprobe, out))
    return dict(zip(("NQ", "RW", "ck", "nchunks", "stages"), list(out)))


def launches(idx):
    return int(_capi.lib().wb_launch_count(idx._h))


def gemm_stats(idx):
    a, b = C.c_int64(), C.c_int64()
    _capi.check(_capi.lib().wb_gemm_stats(idx._h, C.byref(a), C.byref(b)))
    return a.value, b.value


def fused(idx):
    return int(_capi.lib().wb_ivf_fused_searches(idx._h))


def grouped(idx):
    off = np.zeros(int(_capi.lib().wb_nlist(idx._h)) + 1, np.int64)
    g = C.c_int()
    _capi.check(_capi.lib().wb_ivf_list_offsets(idx._h, _capi.ptr(off), C.byref(g)))
    return bool(g.value)


def counted(idx, fn):
    """(fn(), launches it made)."""
    l0 = launches(idx)
    r = fn()
    return r, launches(idx) - l0


def same_alone(idx, xq, D, I, k, qs):
    """The queries `qs` (both sides of a boundary) searched again on their own: bit for bit the same rows."""
    qs = np.asarray(qs)
    D2, I2 = idx.search(xq[qs], k)
    assert np.array_equal(I[qs], I2), f"queries {qs.tolist()}: ids differ from a search of them alone"
    assert np.array_equal(D[qs].view(np.uint32), D2.view(np.uint32)), f"queries {qs.tolist()}: scores differ"


def range_dev(idx, xq, thresh, nprobe=1):
    """wb_range_search_dev + wb_range_result_copy_dev: (lims uint64, D, I) as device tensors."""
    L = _capi.lib()
    q = torch.as_tensor(np.ascontiguousarray(xq, np.float32), device="cuda")
    st = torch.cuda.current_stream()
    lims = np.zeros(len(xq) + 1, np.int64)
    res = C.c_void_p()
    _capi.check(L.wb_range_search_dev(idx._h, None, len(xq), q.data_ptr(), float(thresh), nprobe, _capi.ptr(lims),
                                      C.byref(res), st.cuda_stream))
    try:
        n = int(lims[-1])
        Dt = torch.empty(n, dtype=torch.float32, device="cuda")
        It = torch.empty(n, dtype=torch.int64, device="cuda")
        _capi.check(L.wb_range_result_copy_dev(res, Dt.data_ptr(), It.data_ptr(), st.cuda_stream))
        st.synchronize()
    finally:
        _capi.check(L.wb_range_result_free(res))
    return lims.astype(np.uint64), Dt, It


def range_subset(lims, Dg, Ig, qs):
    """The results of the queries `qs` as a range result of its own."""
    l = lims.astype(np.int64)
    seg = [np.arange(l[q], l[q + 1]) for q in qs]
    sub = np.zeros(len(qs) + 1, np.uint64)
    sub[1:] = np.cumsum([s.size for s in seg])
    at = np.concatenate(seg) if seg else np.zeros(0, np.int64)
    return sub, Dg[at], Ig[at]


def same_range_alone(idx, xq, lims, Dg, Ig, thresh, qs):
    """Range results of the queries `qs` searched alone: the same entries, bit for bit (so lims run on continuously
    across the chunk boundaries between them)."""
    l2, D2, I2 = idx.range_search(xq[np.asarray(qs)], thresh)
    l1, D1, I1 = range_subset(lims, Dg, Ig, qs)
    assert np.array_equal(l1, l2), f"queries {list(qs)}: hit counts differ from a search of them alone"
    assert np.array_equal(I1, I2) and np.array_equal(D1.view(np.uint32), D2.view(np.uint32))


def ivf_index(xb, ids, cent):
    idx = faiss.IndexIVFFlat(faiss.IndexFlatIP(xb.shape[1]), xb.shape[1], cent.shape[0], faiss.METRIC_INNER_PRODUCT)
    idx.set_centroids(cent)
    idx.add_with_ids(xb, ids)
    return idx


def candidates(assign, probes):
    """The rows of each query's probed lists (rows of `probes`), as index arrays."""
    order = np.argsort(assign, kind="stable")
    off = np.searchsorted(assign[order], np.arange(int(assign.max()) + 2))
    return [np.sort(np.concatenate([order[off[l]:off[l + 1]] for l in pr])) for pr in probes]


def gpu_assign(idx, n):
    """The lists the library assigned rows [0, n) to, read before the first search regroups the store; then one search
    builds the inverted lists, so that the launch counts of later searches are theirs alone."""
    _, _, a = idx._export(0, n, want_assign=True, want_ids=True, want_x=False)
    idx.search(np.zeros((1, idx.d), np.float32), 1)
    return a.astype(np.int64)


# ---- 1. K1 / K5 launch split at kMaxGridY query groups -------------------------------------------------------------
@pytest.mark.parametrize("rows,d,k,fuse_tail", [(1000, 37, 10, True), (3000, 5, 400, False)])
def test_k1_grid_split(rows, d, k, fuse_tail):
    """8 * 32768 + 9 queries = 32769 groups of 8: two K1 launches, the second offset by 262144 queries.  K2 does not
    take these stores (fewer than 4 * cap rows, or k > cap / 2)."""
    xb = O.unit_gaussian(rows, d, 100 + d)
    ids = np.arange(rows, dtype=np.int64) * 3 + 7
    idx = faiss.IndexIDMap(faiss.IndexFlatIP(d))
    idx.add_with_ids(xb, ids)
    nq = 8 * GRID_Y + 9
    assert scan_plan(idx, nq, k)["NQ"] == 8 and scan_plan(idx, nq, k)["nchunks"] == 1
    xq = O.unit_gaussian(nq, d, 200 + d)
    _, small = counted(idx, lambda: idx.search(xq[:9], k))  # one scan launch (+ the query padding, + K3 if unfused)
    (D, I), big = counted(idx, lambda: idx.search(xq, k))
    pad = 1 if d % 4 else 0
    assert small == pad + 1 + (0 if fuse_tail else 1), small
    assert big == small + 1, (big, small)  # one more scan launch, one merge either way
    assert gemm_stats(idx) == (0, 0)
    print(f"\nK1 split rows={rows} d={d} k={k}: launches {big} (9 queries: {small}), fused tail {fuse_tail}")
    O.compare_topk(D, I, *topk_fp64(xb, xq, k, ids))
    same_alone(idx, xq, D, I, k, [0, 1, 8 * GRID_Y - 1, 8 * GRID_Y, 8 * GRID_Y + 1, nq - 1])


NI, DI, NLIST = 20_000, 37, 64


@pytest.fixture(scope="module")
def ivf_data():
    xb = O.clustered_unit(NI, DI, 64, 31)
    cent = O.unit_gaussian(NLIST, DI, 32)
    ids = np.arange(NI, dtype=np.int64) * 5 + 1
    return xb, ids, cent


@pytest.mark.parametrize("contiguous", [1, 0])
def test_ivf_query_major_grid_split(ivf_data, monkeypatch, contiguous):
    """32768 + 7 queries, one query per K5 group: two list-scan launches, on a store grouped by list and on one that is
    not (WB_IVF_CONTIGUOUS=0: the scan reads rows through the slot permutation)."""
    monkeypatch.setenv("WB_IVF_LISTMAJOR", "0")
    monkeypatch.setenv("WB_IVF_CONTIGUOUS", str(contiguous))
    xb, ids, cent = ivf_data
    idx = ivf_index(xb, ids, cent)
    assign = gpu_assign(idx, NI)
    idx.nprobe = nprobe = 4
    k, nq = 20, GRID_Y + 7
    xq = O.clustered_unit(nq, DI, 64, 41)
    e0 = gemm_stats(idx)
    _, small = counted(idx, lambda: idx.search(xq[:8], k))
    assert grouped(idx) == bool(contiguous)
    (D, I), big = counted(idx, lambda: idx.search(xq, k))
    assert big == small + 1, (big, small)
    assert gemm_stats(idx) == e0  # the coarse step of 64 lists stays on K1 (exact fp32)
    print(f"\nK5 split contiguous={contiguous}: launches {big} (8 queries: {small})")
    probes, gaps = coarse_fp64(cent, xq, nprobe)
    clear = gaps > 1e-5
    assert clear.sum() >= nq - 50
    Dr, Ir = ivf_topk_fp64(xb, ids, assign, probes, xq, k)
    O.compare_topk(D[clear], I[clear], Dr[clear], Ir[clear])
    same_alone(idx, xq, D, I, k, [0, GRID_Y - 1, GRID_Y, GRID_Y + 1, nq - 1])


# ---- 2. K2 query chunks of 65536 ------------------------------------------------------------------------------------
def test_k2_query_chunks(monkeypatch):
    """2 * 65536 + 129 queries over 20000 x 64: three K2 calls, the last a 129-query block."""
    n, d, k = 20_000, 64, 100
    xb = O.unit_gaussian(n, d, 300)
    idx = faiss.IndexFlatIP(d)
    idx.add(xb)
    nq = 2 * K2_MAX_Q + 129
    xq = O.unit_gaussian(nq, d, 301)
    D, I = idx.search(xq, k)
    epochs, fallbacks = gemm_stats(idx)
    assert epochs > 0 and fallbacks == 0, (epochs, fallbacks)
    print(f"\nK2 chunks: {epochs} epochs, {fallbacks} fallbacks")
    O.compare_topk(D, I, *topk_fp64(xb, xq, k), band=BAND[True])
    monkeypatch.setenv("WB_GEMM_FORCE", "1")  # the boundary queries alone on K2 as well
    qs = [0, K2_MAX_Q - 2, K2_MAX_Q - 1, K2_MAX_Q, K2_MAX_Q + 1, 2 * K2_MAX_Q - 1, 2 * K2_MAX_Q, 2 * K2_MAX_Q + 1, nq - 1]
    same_alone(idx, xq, D, I, k, qs)
    assert gemm_stats(idx)[0] > epochs


def test_k2_overflow_repair_past_one_chunk(monkeypatch):
    """Adversarial order (every row beats the running threshold) in a batch of 65536 + 40 queries: both K2 calls
    overflow and the whole batch is repaired by the CUDA-core scan."""
    monkeypatch.setenv("WB_GEMM_FORCE", "1")
    n, d, k = 120_000, 64, 10
    rng = np.random.default_rng(0)
    base = O.unit_gaussian(1, d, 1)[0]
    t = np.linspace(-0.9, 0.9, n).astype(np.float32)  # score of row i against `base` grows with i
    noise = O.unit_gaussian(n, d, 2)
    noise -= (noise @ base)[:, None] * base[None, :]
    noise /= np.linalg.norm(noise, axis=1, keepdims=True)
    xb = (t[:, None] * base[None, :] + np.sqrt(1 - t[:, None] ** 2) * noise).astype(np.float32)
    nq = K2_MAX_Q + 40
    xq = np.repeat(base[None, :], nq, axis=0) + 1e-3 * rng.standard_normal((nq, d)).astype(np.float32)
    xq = (xq / np.linalg.norm(xq, axis=1, keepdims=True)).astype(np.float32)
    idx = faiss.IndexFlatIP(d)
    idx.add(xb)
    D, I = idx.search(xq, k)
    epochs, fallbacks = gemm_stats(idx)
    assert epochs > 0 and fallbacks == 1, (epochs, fallbacks)
    print(f"\nK2 overflow repair: {epochs} epochs, {fallbacks} fallback")
    O.compare_topk(D, I, *topk_fp64(xb, xq, k))


# ---- 3. range chunks of 32768 queries ------------------------------------------------------------------------------
def _range_store(kind):
    if kind == "ivf":
        xb = O.clustered_unit(NI, DI, 64, 31)
        cent = O.unit_gaussian(NLIST, DI, 32)
        ids = np.arange(NI, dtype=np.int64) * 5 + 1
        idx = ivf_index(xb, ids, cent)
        return idx, xb, ids, cent, gpu_assign(idx, NI)
    n = 1000 if kind == "k1" else 3000  # K2 takes no store below 4 * 256 rows
    xb = O.unit_gaussian(n, DI, 400)
    ids = np.arange(n, dtype=np.int64) * 2 + 11
    idx = faiss.IndexIDMap(faiss.IndexFlatIP(DI))
    idx.add_with_ids(xb, ids)
    return idx, xb, ids, None, None


@pytest.mark.parametrize("kind", ["k1", "k2", "ivf"])
def test_range_chunks(monkeypatch, kind):
    """2 * 32768 + 3 queries: three range chunks; lims run on across them, through the host entry point and as a device
    result of one part per chunk."""
    if kind == "k2":
        monkeypatch.setenv("WB_GEMM_FORCE", "1")
    idx, xb, ids, cent, assign = _range_store(kind)
    nprobe = 4
    idx.nprobe = nprobe
    nq = 2 * RANGE_MAX_Q + 3
    xq = O.clustered_unit(nq, DI, 64, 42) if kind == "ivf" else O.unit_gaussian(nq, DI, 401)
    s = xq[:64].astype(np.float64) @ xb.astype(np.float64).T
    thresh = np.float32(np.quantile(s, 1 - 20 / xb.shape[0]))  # about 20 hits per query
    e0 = gemm_stats(idx)
    (lims, Dg, Ig), small = counted(idx, lambda: idx.range_search(xq[:3], thresh))
    (lims, Dg, Ig), big = counted(idx, lambda: idx.range_search(xq, thresh))
    e1 = gemm_stats(idx)
    pad = 1  # d = 37: the queries are padded to the row stride
    if kind == "k2":
        assert e1[0] > e0[0] and e1[1] == e0[1], (e0, e1)
    else:
        assert e1 == e0
        assert big - pad == 3 * (small - pad), (big, small)  # every chunk: the same launches as one small batch
    print(f"\nrange chunks {kind}: launches {big} (3 queries: {small}), K2 epochs {e1[0] - e0[0]}")
    assert int(lims[-1]) > nq
    if kind == "ivf":
        probes, gaps = coarse_fp64(cent, xq, nprobe)
        clear = np.nonzero(gaps > 1e-5)[0]
        assert clear.size >= nq - 50
        cand = candidates(assign, probes[clear])
        range_check(*range_subset(lims, Dg, Ig, clear), xb, xq[clear], thresh, ids, cand=cand, band=BAND[False])
    else:
        range_check(lims, Dg, Ig, xb, xq, thresh, ids, band=BAND[kind == "k2"])
    qs = [0, RANGE_MAX_Q - 1, RANGE_MAX_Q, RANGE_MAX_Q + 1, 2 * RANGE_MAX_Q - 1, 2 * RANGE_MAX_Q, nq - 1]
    same_range_alone(idx, xq, lims, Dg, Ig, thresh, qs)
    ld, Dd, Id = range_dev(idx, xq, thresh, nprobe)
    assert np.array_equal(ld, lims)
    assert np.array_equal(Id.cpu().numpy(), Ig) and np.array_equal(Dd.cpu().numpy().view(np.uint32), Dg.view(np.uint32))


# ---- 4. the range hit budget ---------------------------------------------------------------------------------------
def _check_everything(lims, Dt, It, xb_t, xq, N):
    """Every query returned every row once, by score descending then position, scores within 1e-5 of fp64."""
    n = len(xq)
    assert np.array_equal(lims, np.arange(n + 1, dtype=np.uint64) * N)
    ar = torch.arange(N, device="cuda")
    for q0 in range(0, n, 16):
        q1 = min(n, q0 + 16)
        d, p = Dt(q0, q1).view(q1 - q0, N), It(q0, q1).view(q1 - q0, N)
        assert torch.equal(torch.sort(p, dim=1).values, ar.expand(q1 - q0, N)), f"queries {q0}..{q1}: not every row"
        s = torch.as_tensor(xq[q0:q1], device="cuda").double() @ xb_t.T
        assert float((d.double() - torch.gather(s, 1, p)).abs().max()) <= 1e-5
        dd = torch.diff(d, dim=1)
        assert bool((dd <= 0).all()), "scores must be descending"
        assert bool((torch.diff(p, dim=1)[dd == 0] > 0).all()), "equal scores must come in insertion order"


def test_range_budget_splits_a_chunk():
    """2^20 rows, 300 queries, every row a hit: 3.1e8 hits do not fit the 2^28 budget of one chunk, which shrinks to
    the 256 queries that do (2^28 exactly) and runs the other 44 next."""
    N, d, nq = 1 << 20, 4, 300
    xb = O.unit_gaussian(N, d, 500)
    idx = faiss.IndexFlatIP(d)
    idx.add(xb)
    xq = O.unit_gaussian(nq, d, 501)
    xb_t = torch.as_tensor(xb, device="cuda").double()
    lims, Dg, Ig = idx.range_search(xq, -2.0)
    assert int(lims[256]) == BUDGET and int(lims[-1]) > BUDGET
    print(f"\nrange budget: {int(lims[-1])} hits, first chunk {int(lims[256])}")
    _check_everything(lims, lambda a, b: torch.as_tensor(Dg[a * N:b * N], device="cuda"),
                      lambda a, b: torch.as_tensor(Ig[a * N:b * N], device="cuda"), xb_t, xq, N)
    del Dg, Ig
    ld, Dd, Id = range_dev(idx, xq, -2.0)
    _check_everything(ld, lambda a, b: Dd[a * N:b * N], lambda a, b: Id[a * N:b * N], xb_t, xq, N)


def test_range_single_query_over_budget():
    """One query with 2^28 + 2^20 hits is an error; the index then still answers search and range search."""
    L = _capi.lib()
    n = BUDGET + (1 << 20)
    idx = faiss.IndexFlatIP(1)
    idx.reserve(n)
    g = torch.Generator(device="cuda").manual_seed(7)
    x = torch.rand(n, 1, device="cuda", generator=g) * 2 - 1  # scores against q = 1 are the values themselves
    _capi.check(L.wb_add_with_ids_dev(idx._h, n, x.data_ptr(), None, torch.cuda.current_stream().cuda_stream))
    torch.cuda.current_stream().synchronize()
    assert idx.ntotal == n
    q = np.ones((1, 1), np.float32)
    with pytest.raises(RuntimeError, match="more than the 268435456 one call can hold"):
        idx.range_search(q, -2.0)
    print("\nrange over budget: raised")
    v = x[:, 0]
    k = 100
    top = torch.topk(v, 4 * k).values
    D, I = idx.search(q, k)
    cand = torch.nonzero(v >= top[k - 1])[:, 0]  # every row tied with the k-th value too
    order = np.lexsort((cand.cpu().numpy(), -v[cand].double().cpu().numpy()))[:k]
    assert np.array_equal(I[0], cand.cpu().numpy()[order])
    assert np.array_equal(D[0], v[cand].cpu().numpy()[order])
    t = float(top[3 * k])
    lims, Dg, Ig = idx.range_search(q, t)
    hit = torch.nonzero(v > t)[:, 0]
    order = np.lexsort((hit.cpu().numpy(), -v[hit].double().cpu().numpy()))
    assert int(lims[1]) == hit.numel() and np.array_equal(Ig, hit.cpu().numpy()[order])
    assert np.array_equal(Dg, v[hit].cpu().numpy()[order])


# ---- 5. wide rows: the chunked scan plan -----------------------------------------------------------------------------
WIDE_N = 60_000


@pytest.fixture(scope="module")
def wide():
    """60000 rows at d = 2560 and 4096: about 13 row groups per CTA, so the static row partition of the chunked plan
    loops."""
    out = {}
    for d in (2560, 4096):
        xb = O.unit_gaussian(WIDE_N, d, d)
        ids = np.arange(WIDE_N, dtype=np.int64) * 7 + 3
        idx = faiss.IndexIDMap(faiss.IndexFlatIP(d))
        idx.add_with_ids(xb, ids)
        out[d] = (idx, xb, ids)
    return out


@pytest.mark.parametrize("d,nq,k", [(2560, 8, 10), (2560, 9, 100)] + [(4096, nq, k) for nq in (1, 2, 4)
                                                                    for k in (1, 100, 2048)])
def test_wide_rows_search(wide, d, nq, k):
    idx, xb, ids = wide[d]
    p = scan_plan(idx, nq, k)
    assert p["nchunks"] > 1 and (d != 2560 or p["NQ"] == 8), p
    xq = O.unit_gaussian(nq, d, 600 + nq)
    e0 = gemm_stats(idx)
    (D, I), n = counted(idx, lambda: idx.search(xq, k))
    assert gemm_stats(idx) == e0
    print(f"\nwide d={d} nq={nq} k={k}: plan {p}, launches {n}")
    O.compare_topk(D, I, *topk_fp64(xb, xq, k, ids))
    if nq > 1:
        same_alone(idx, xq, D, I, k, [nq - 1])


def test_wide_rows_range(wide):
    idx, xb, ids = wide[2560]
    nq = 9
    p = scan_plan(idx, nq, 0)
    assert p["nchunks"] > 1 and p["NQ"] == 8, p
    xq = O.unit_gaussian(nq, 2560, 610)
    s = xq.astype(np.float64) @ xb.astype(np.float64).T
    thresh = np.float32(np.quantile(s, 1 - 300 / WIDE_N))
    e0 = gemm_stats(idx)
    lims, Dg, Ig = idx.range_search(xq, thresh)
    assert gemm_stats(idx) == e0 and int(lims[-1]) > 100 * nq
    print(f"\nwide range: plan {p}, {int(lims[-1])} hits")
    range_check(lims, Dg, Ig, xb, xq, thresh, ids, band=BAND[False])


@pytest.mark.parametrize("nq", [4, 8])  # (from 9 queries K2 takes the masked store)
def test_wide_rows_filtered(wide, nq):
    """The mask path (half of the rows selected) under the chunked plan."""
    idx, xb, ids = wide[4096]
    k = 100
    assert scan_plan(idx, nq, k)["nchunks"] > 1
    sel = faiss.IDSelectorRange(int(ids[WIDE_N // 4]), int(ids[3 * WIDE_N // 4]))
    keep = np.nonzero((ids >= sel.imin) & (ids < sel.imax))[0]
    xq = O.unit_gaussian(nq, 4096, 620 + nq)
    e0 = gemm_stats(idx)
    D, I = idx.search(xq, k, params=faiss.SearchParameters(sel=sel))
    assert gemm_stats(idx) == e0
    Dr, Ir = topk_fp64(xb[keep], xq, k, ids[keep])
    O.compare_topk(D, I, Dr, Ir)


@pytest.fixture(scope="module")
def wide_ivf():
    d, nlist = 4096, 32
    xb = O.clustered_unit(WIDE_N // 2, d, 64, 630)
    cent = O.unit_gaussian(nlist, d, 631)
    ids = np.arange(xb.shape[0], dtype=np.int64) + 5
    idx = ivf_index(xb, ids, cent)
    return idx, xb, ids, cent, gpu_assign(idx, xb.shape[0])


@pytest.mark.parametrize("nq,fuse", [(1, True), (4, True), (4, False), (9, False)])
def test_wide_rows_ivf(wide_ivf, monkeypatch, nq, fuse):
    """The K5 gather scan with chunked stages: coarse step fused into the launch, and as its own launch."""
    idx, xb, ids, cent, assign = wide_ivf
    nprobe, k = 4, 50
    idx.nprobe = nprobe
    p = scan_plan(idx, 1, k, gather=True, nprobe=nprobe)
    assert p["nchunks"] > 1, p
    if not fuse:
        monkeypatch.setenv("WB_IVF_FUSE_COARSE", "0")
    xq = O.clustered_unit(nq, 4096, 64, 640 + nq)
    f0 = fused(idx)
    D, I = idx.search(xq, k)
    assert fused(idx) - f0 == (1 if fuse else 0)
    print(f"\nwide IVF nq={nq} fused={fuse}: plan {p}")
    O.compare_topk(D, I, *O.ivf_search(xb, ids, assign, cent, xq, k, nprobe))


@pytest.mark.parametrize("d", [4096, 8192])
def test_wide_rows_k2(monkeypatch, d):
    monkeypatch.setenv("WB_GEMM_FORCE", "1")
    n, nq, k = 20_000, 16, 100
    xb = O.unit_gaussian(n, d, 650 + d)
    idx = faiss.IndexFlatIP(d)
    idx.add(xb)
    xq = O.unit_gaussian(nq, d, 651)
    D, I = idx.search(xq, k)
    epochs, fallbacks = gemm_stats(idx)
    assert epochs > 0 and fallbacks == 0, (epochs, fallbacks)
    print(f"\nwide K2 d={d}: {epochs} epochs")
    O.compare_topk(D, I, *topk_fp64(xb, xq, k), band=BAND[True])


def test_widest_rows():
    """d = 16384 still plans (chunked); d = 65536 is accepted by create but no scan fits shared memory: search fails
    with the planner's message, and a later search on another index is unaffected."""
    d, n = 16384, 8000
    xb = O.unit_gaussian(n, d, 660)
    idx = faiss.IndexFlatIP(d)
    idx.add(xb)
    p = scan_plan(idx, 4, 10)
    assert p["nchunks"] > 1, p
    xq = O.unit_gaussian(4, d, 661)
    D, I = idx.search(xq, 10)
    O.compare_topk(D, I, *topk_fp64(xb, xq, 10))
    huge = faiss.IndexFlatIP(65536)
    huge.add(O.unit_gaussian(100, 65536, 662))
    with pytest.raises(RuntimeError, match="scan does not fit shared memory"):
        scan_plan(huge, 1, 10)
    with pytest.raises(RuntimeError, match="scan does not fit shared memory"):
        huge.search(O.unit_gaussian(1, 65536, 663), 10)
    print(f"\nwidest: d=16384 plan {p}; d=65536 refused")
    D2, I2 = idx.search(xq, 10)
    assert np.array_equal(I, I2) and np.array_equal(D.view(np.uint32), D2.view(np.uint32))


# ---- 6. the tensor-core coarse quantizer ----------------------------------------------------------------------------
@pytest.fixture(scope="module")
def big_ivf():
    """nlist = 20000 at d = 768 (WISE's IVF sizes): a batch's coarse step runs on K2 in 3xTF32."""
    d, nlist, n = 768, 20_000, 200_000
    cent = O.unit_gaussian(nlist, d, 700)
    xb = O.unit_gaussian(n, d, 701)
    ids = np.arange(n, dtype=np.int64) * 3 + 2
    idx = ivf_index(xb, ids, cent)
    return idx, xb, ids, cent, gpu_assign(idx, n)


def _ivf_superset_ok(I, D, xb, ids, assign, cent, xq, nprobe):
    """A query whose nprobe-th centroid is a near tie: every returned row lies in a list within 1e-5 of the fp64
    nprobe-th centroid score and its score is within 1e-5 of fp64."""
    pos = {int(v): i for i, v in enumerate(ids)}
    s = xq.astype(np.float64) @ cent.astype(np.float64).T
    kth = np.sort(s)[::-1][nprobe - 1]
    ok_lists = np.nonzero(s >= kth - 1e-5)[0]
    p = np.array([pos[int(v)] for v in I if v >= 0])
    assert np.all(np.isin(assign[p], ok_lists))
    assert np.all(np.abs(D[: p.size] - xb[p].astype(np.float64) @ xq.astype(np.float64)) <= 1e-5)


def test_tensor_core_coarse_search(big_ivf):
    idx, xb, ids, cent, assign = big_ivf
    nq, nprobe, k = 256, 16, 10
    idx.nprobe = nprobe
    xq = O.unit_gaussian(nq, 768, 710)
    e0 = gemm_stats(idx)
    D, I = idx.search(xq, k)
    e1 = gemm_stats(idx)
    assert e1[0] > e0[0] and e1[1] == e0[1], (e0, e1)  # no WB_GEMM_FORCE: the cost model picks K2
    _, gaps = coarse_fp64(cent, xq, nprobe)
    clear = np.nonzero(gaps > 1e-5)[0]
    print(f"\nK2 coarse: {e1[0] - e0[0]} epochs, {clear.size} / {nq} queries clear of a coarse near tie")
    assert clear.size >= nq * 3 // 4
    Dr, Ir = O.ivf_search(xb, ids, assign, cent, xq[clear], k, nprobe)
    O.compare_topk(D[clear], I[clear], Dr, Ir)
    is_clear = np.isin(np.arange(nq), clear)
    for i in range(nq):
        f0 = fused(idx)
        Da, Ia = idx.search(xq[i:i + 1], k)  # one query: the exact fp32 coarse step fused into the list scan
        assert fused(idx) - f0 == 1
        if is_clear[i]:
            assert np.array_equal(Ia[0], I[i]) and np.array_equal(Da[0].view(np.uint32), D[i].view(np.uint32)), i
        else:
            _ivf_superset_ok(I[i], D[i], xb, ids, assign, cent, xq[i], nprobe)


def test_tensor_core_coarse_range(big_ivf):
    idx, xb, ids, cent, assign = big_ivf
    nq, nprobe = 256, 16
    idx.nprobe = nprobe
    xq = O.unit_gaussian(nq, 768, 720)
    thresh = np.float32(0.05)
    e0 = gemm_stats(idx)
    lims, Dg, Ig = idx.range_search(xq, thresh)
    e1 = gemm_stats(idx)
    assert e1[0] > e0[0] and e1[1] == e0[1], (e0, e1)
    probes, gaps = coarse_fp64(cent, xq, nprobe)
    clear = np.nonzero(gaps > 1e-5)[0]
    print(f"\nK2 coarse range: {int(lims[-1])} hits, {clear.size} / {nq} queries clear")
    cand = candidates(assign, probes[clear])
    range_check(*range_subset(lims, Dg, Ig, clear), xb, xq[clear], thresh, ids, cand=cand, band=BAND[False])
    for i in np.setdiff1d(np.arange(nq), clear):
        a, b = int(lims[i]), int(lims[i + 1])
        _ivf_superset_ok(Ig[a:b], Dg[a:b], xb, ids, assign, cent, xq[i], nprobe)
    # the first k hits of a query with at least k of them are search(x, k) (the same probes: the same K2 coarse step)
    k = 5
    D, I = idx.search(xq, k)
    cnt = np.diff(lims.astype(np.int64))
    big = np.nonzero(cnt >= k)[0]
    assert big.size >= nq // 2
    Dr = np.stack([Dg[int(lims[i]):int(lims[i]) + k] for i in big])
    Ir = np.stack([Ig[int(lims[i]):int(lims[i]) + k] for i in big])
    assert np.array_equal(Ir, I[big]) and np.array_equal(Dr.view(np.uint32), D[big].view(np.uint32))


# ---- 7. the list-major bound ----------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lm_ivf():
    d, nlist, n = 64, 256, 40_000
    xb = O.clustered_unit(n, d, 64, 800)
    cent = O.unit_gaussian(nlist, d, 801)
    ids = np.arange(n, dtype=np.int64) + 100
    idx = ivf_index(xb, ids, cent)
    return idx, xb, ids, cent, gpu_assign(idx, n)


@pytest.mark.parametrize("nq,k", [(1024, 2048), (4096, 512)])
def test_listmajor_parts_bound(lm_ivf, monkeypatch, nq, k):
    """nq x 128 probes x k x 8 bytes of list-major parts above 2e9: the batch goes query-major even with
    WB_IVF_LISTMAJOR=1.  At k = 512 the list-major plan itself fits (8 queries per CTA), so only the bound keeps the
    batch off it; half the batch (1.07e9 bytes) does take it."""
    idx, xb, ids, cent, assign = lm_ivf
    nprobe = 128
    idx.nprobe = nprobe
    assert nq * nprobe * k * 8 > 2e9
    xq = O.clustered_unit(nq, xb.shape[1], 64, 802)
    monkeypatch.setenv("WB_IVF_LISTMAJOR", "1")
    (D, I), bound = counted(idx, lambda: idx.search(xq, k))
    if k == 512:
        assert scan_plan(idx, 8, k)["NQ"] == 8
        _, lm = counted(idx, lambda: idx.search(xq[:nq // 2], k))
    monkeypatch.setenv("WB_IVF_LISTMAJOR", "0")
    (Dq, Iq), qm = counted(idx, lambda: idx.search(xq, k))
    assert bound == qm, (bound, qm)
    if k == 512:
        _, qm_half = counted(idx, lambda: idx.search(xq[:nq // 2], k))
        assert lm > qm_half, (lm, qm_half)  # the witness tells the two paths apart
    print(f"\nlist-major bound nq={nq} k={k}: launches {bound}, query-major {qm}")
    assert np.array_equal(I, Iq) and np.array_equal(D.view(np.uint32), Dq.view(np.uint32))
    probes, gaps = coarse_fp64(cent, xq, nprobe)
    clear = gaps > 1e-5
    assert clear.sum() >= 0.95 * nq  # 128 of 256 lists: near ties at the cut are common
    Dr, Ir = ivf_topk_fp64(xb, ids, assign, probes, xq, k)
    O.compare_topk(D[clear], I[clear], Dr[clear], Ir[clear])
