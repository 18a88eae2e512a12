"""Range search on a B200: every path (K1, K2 TS and SS, K5 gather; mask and compact filters) against the fp64
reference of tests/range_oracle.py.  Membership may differ from fp64 only for rows within the near-tie band of the
threshold; every returned score is within 1e-5 of fp64 and strictly above the threshold."""
import ctypes as C

import numpy as np
import pytest

from oracle import oracle as O
from range_oracle import check as _check, ivf_range_search, range_search
from wise_b200 import _capi
from wise_b200 import faiss_compat as faiss

pytestmark = pytest.mark.gpu

N, D = 200_000, 126
BAND = {False: 2e-6, True: 4e-6}  # scan path, tensor-core path


@pytest.fixture(scope="module")
def flat():
    xb = O.unit_gaussian(N, D, 501)
    xb[150_001] = xb[1234]  # a planted duplicate
    ids = np.random.default_rng(8).permutation(N).astype(np.int64) * 2 + 3
    index = faiss.IndexIDMap(faiss.IndexFlatIP(D))
    index.add_with_ids(xb, ids)
    return index, xb, ids


def _thresholds(xb, xq):
    s = (xq.astype(np.float64) @ xb.astype(np.float64).T).ravel()
    return {"none": float(s.max()) + 0.01, "50": float(np.quantile(s, 1 - 50 / N)),
            "5000": float(np.quantile(s, 1 - 5000 / N))}


PATHS = [(1, False), (4, False), (16, True), (200, True)]  # (nq, WB_GEMM_FORCE): K1, K1, K2 TS, K2 SS


@pytest.mark.parametrize("nq,force", PATHS)
@pytest.mark.parametrize("which", ["none", "50", "5000"])
def test_flat_matches_fp64(flat, monkeypatch, nq, force, which):
    index, xb, ids = flat
    if force:
        monkeypatch.setenv("WB_GEMM_FORCE", "1")
    xq = O.unit_gaussian(nq, D, 60 + nq)
    t = _thresholds(xb, xq)[which]
    lims, Dg, Ig = index.range_search(xq, t)
    _check(lims, Dg, Ig, xb, xq, np.float32(t), ids, band=BAND[force])
    if which == "none":
        assert lims[-1] == 0
    # agreement with search: the first 100 hits of a query with >= 100 hits are search(x, 100)
    cnt = np.diff(lims.astype(np.int64))
    big = np.nonzero(cnt >= 100)[0]
    if big.size:
        Ds, Is = index.search(xq, 100)
        Dr = np.stack([Dg[int(lims[i]):int(lims[i]) + 100] for i in big])
        Ir = np.stack([Ig[int(lims[i]):int(lims[i]) + 100] for i in big])
        O.compare_topk(Dr, Ir, Ds[big], Is[big], band=BAND[force])


@pytest.mark.parametrize("nq,force", [(1, False), (16, True)])
def test_strict_threshold_and_duplicates(flat, monkeypatch, nq, force):
    index, xb, ids = flat
    if force:
        monkeypatch.setenv("WB_GEMM_FORCE", "1")
    xq = O.unit_gaussian(nq, D, 70)
    xq[0] = xb[1234]
    lims, Dg, Ig = index.range_search(xq, 0.3)
    a, b = int(lims[0]), int(lims[1])
    assert Ig[a] == ids[1234] and Ig[a + 1] == ids[150_001] and Dg[a] == Dg[a + 1]  # both copies, insertion order
    j = a + (b - a) // 2
    s = Dg[j]
    l2, D2, I2 = index.range_search(xq, s)
    assert np.all(D2 > s)
    assert Ig[j] not in set(I2[int(l2[0]):int(l2[1])].tolist())
    assert int(l2[1]) == int(np.sum(Dg[a:b] > s))
    l3, D3, I3 = index.range_search(xq, np.nextafter(s, -np.inf))
    assert Ig[j] in set(I3[int(l3[0]):int(l3[1])].tolist())
    assert int(l3[1]) == int(np.sum(Dg[a:b] >= s))
    l4, _, I4 = index.range_search(xq, Dg[a])  # the duplicated best score: both copies leave together
    assert ids[1234] not in set(I4[: int(l4[1])].tolist()) and ids[150_001] not in set(I4[: int(l4[1])].tolist())


@pytest.mark.parametrize("force", [False, True])
def test_everything(monkeypatch, force):
    """thresh = -2 on unit rows: all 200k rows for 64 queries (12.8M hits) - overflows the first pool and every K2
    epoch's candidate list; the results stay exact."""
    if force:
        monkeypatch.setenv("WB_GEMM_FORCE", "1")
    xb = O.unit_gaussian(N, 64, 9)
    index = faiss.IndexFlatIP(64)
    index.add(xb)
    xq = O.unit_gaussian(64, 64, 10)
    lims, Dg, Ig = index.range_search(xq, -2.0)
    assert np.array_equal(lims, np.arange(65, dtype=np.uint64) * N)
    for i in range(64):
        d, p = Dg[i * N:(i + 1) * N], Ig[i * N:(i + 1) * N]
        assert np.array_equal(np.sort(p), np.arange(N))
        s = xb[p].astype(np.float64) @ xq[i].astype(np.float64)
        assert np.all(np.abs(d - s) <= 1e-5)
        assert np.all(np.diff(d.astype(np.float64)) <= 0)
        assert np.all(np.diff(p)[np.diff(d) == 0] > 0)


def test_nothing_and_edge_cases(flat):
    index, xb, ids = flat
    xq = O.unit_gaussian(3, D, 11)
    for t in (np.inf, np.nan):
        lims, Dg, Ig = index.range_search(xq, t)
        assert lims.tolist() == [0, 0, 0, 0] and Dg.size == 0 and Ig.size == 0
    lims, Dg, Ig = index.range_search(xq[:0], 0.0)
    assert lims.tolist() == [0] and lims.dtype == np.uint64
    empty = faiss.IndexFlatIP(D)
    lims, Dg, _ = empty.range_search(xq, -1.0)
    assert lims.tolist() == [0, 0, 0, 0]
    # rows containing NaN are never returned
    xn = O.unit_gaussian(5000, D, 12)
    xn[[7, 4000]] = np.nan
    nan_index = faiss.IndexFlatIP(D)
    nan_index.add(xn)
    lims, Dg, Ig = nan_index.range_search(xq, -2.0)
    assert int(lims[-1]) == 3 * 4998 and not np.any(np.isin(Ig, [7, 4000]))


def _keep(sel, ids):
    if isinstance(sel, faiss.IDSelectorNot):
        return ~_keep(sel.sel, ids)
    if isinstance(sel, faiss.IDSelectorRange):
        return (ids >= sel.imin) & (ids < sel.imax)
    return np.isin(ids, sel.ids)


def _selector(kind, frac, ids):
    rng = np.random.default_rng(21)
    n = ids.size
    if kind == "batch":
        return faiss.IDSelectorBatch(rng.choice(ids, int(frac * n), replace=False))
    if kind == "not_batch":
        return faiss.IDSelectorNot(faiss.IDSelectorBatch(rng.choice(ids, n - int(frac * n), replace=False)))
    lo = int(np.sort(ids)[n // 3])
    return faiss.IDSelectorRange(lo, lo + 2 * int(frac * n))


@pytest.mark.parametrize("nq,force", [(4, False), (200, True)])
@pytest.mark.parametrize("frac", [0.5, 0.01])  # mask path, compact copy
@pytest.mark.parametrize("kind", ["batch", "range", "not_batch"])
def test_filtered(flat, monkeypatch, nq, force, frac, kind):
    index, xb, ids = flat
    if force:
        monkeypatch.setenv("WB_GEMM_FORCE", "1")
    sel = _selector(kind, frac, ids)
    keep = np.nonzero(_keep(sel, ids))[0]
    xq = O.unit_gaussian(nq, D, 80 + nq)
    t = _thresholds(xb, xq)["5000"]
    lims, Dg, Ig = index.range_search(xq, t, params=faiss.SearchParameters(sel=sel))
    _check(lims, Dg, Ig, xb, xq, np.float32(t), ids, cand=[keep] * nq, band=BAND[force])
    assert lims[-1] > 0
    none = faiss.IDSelectorRange(5, 5)
    lims, Dg, _ = index.range_search(xq, -2.0, params=faiss.SearchParameters(sel=none))
    assert np.all(lims == 0) and Dg.size == 0


NI, DI, NLIST = 60_000, 64, 32


@pytest.fixture(scope="module")
def ivf():
    xb = O.clustered_unit(NI, DI, 64, 31)
    cent = O.unit_gaussian(NLIST, DI, 32)
    ids = np.arange(NI, dtype=np.int64) * 5 + 1
    index = faiss.IndexIVFFlat(faiss.IndexFlatIP(DI), DI, NLIST, faiss.METRIC_INNER_PRODUCT)
    index.set_centroids(cent)
    index.add_with_ids(xb, ids)
    return index, xb, ids, cent


@pytest.mark.parametrize("nq", [1, 4, 64])
@pytest.mark.parametrize("nprobe", [1, 8, NLIST])
@pytest.mark.parametrize("with_params", [False, True])
def test_ivf(ivf, nq, nprobe, with_params):
    index, xb, ids, cent = ivf
    xq = O.clustered_unit(nq, DI, 64, 40 + nq)
    s = (xq.astype(np.float64) @ xb.astype(np.float64).T).ravel()
    t = float(np.quantile(s, 1 - 300 / NI))
    assign = O.ivf_assign(xb, cent)
    _, probes = O.ivf_coarse(xq, cent, nprobe)
    if with_params:
        sel = faiss.IDSelectorRange(1, 5 * (NI // 2))  # the first half of the rows
        index.nprobe = 1
        lims, Dg, Ig = index.range_search(xq, t, params=faiss.SearchParametersIVF(sel=sel, nprobe=nprobe))
        keep = np.arange(NI) < NI // 2
    else:
        index.nprobe = nprobe
        lims, Dg, Ig = index.range_search(xq, t)
        keep = np.ones(NI, bool)
    cand = [np.nonzero(np.isin(assign, probes[i]) & keep)[0] for i in range(nq)]
    _check(lims, Dg, Ig, xb, xq, np.float32(t), ids, cand=cand, band=BAND[False])
    if not with_params:
        lr, Dr, Ir = ivf_range_search(xb, ids, assign, cent, xq, t, nprobe)
        assert abs(int(lims[-1]) - int(lr[-1])) <= max(2, int(lr[-1]) // 1000)
    if nprobe == NLIST and not with_params:  # every list: the same rows as a flat range search
        flat = faiss.IndexIDMap(faiss.IndexFlatIP(DI))
        flat.add_with_ids(xb, ids)
        lf, Df, If = flat.range_search(xq, t)
        assert np.array_equal(lf, lims) or abs(int(lf[-1]) - int(lims[-1])) <= 2
        if np.array_equal(lf, lims):
            assert np.all(np.abs(Df - Dg) <= 1e-5)
            for i in range(nq):
                a, b = int(lims[i]), int(lims[i + 1])
                assert set(If[a:b].tolist()) == set(Ig[a:b].tolist())


def test_ivf_regrouped_after_add(ivf):
    _, _, _, cent = ivf
    xb = O.clustered_unit(30_000, DI, 64, 50)
    ids = np.arange(30_000, dtype=np.int64) + 10
    index = faiss.IndexIVFFlat(faiss.IndexFlatIP(DI), DI, NLIST, faiss.METRIC_INNER_PRODUCT)
    index.set_centroids(cent)
    index.nprobe = 8
    xq = O.clustered_unit(8, DI, 64, 51)
    t = float(np.quantile(xq.astype(np.float64) @ xb.astype(np.float64).T, 1 - 500 / 30_000))
    index.add_with_ids(xb[:20_000], ids[:20_000])
    index.range_search(xq, t)
    index.add_with_ids(xb[20_000:], ids[20_000:])
    lims, Dg, Ig = index.range_search(xq, t)
    assign = O.ivf_assign(xb, cent)
    _, probes = O.ivf_coarse(xq, cent, 8)
    cand = [np.nonzero(np.isin(assign, probes[i]))[0] for i in range(8)]
    _check(lims, Dg, Ig, xb, xq, np.float32(t), ids, cand=cand, band=BAND[False])
    assert np.any(Ig >= 20_010)  # rows of the second add are found


def test_untrained_ivf_raises():
    index = faiss.IndexIVFFlat(faiss.IndexFlatIP(16), 16, 4, faiss.METRIC_INNER_PRODUCT)
    with pytest.raises(RuntimeError, match="not trained"):
        index.range_search(O.unit_gaussian(2, 16, 1), 0.0)
    with pytest.raises(RuntimeError, match="incorrect type"):
        index.range_search(O.unit_gaussian(2, 16, 1), 0.0, params=faiss.SearchParameters())


@pytest.mark.parametrize("nq,force", [(4, False), (200, True)])
def test_deterministic_and_search_unchanged(flat, monkeypatch, nq, force):
    index, xb, ids = flat
    if force:
        monkeypatch.setenv("WB_GEMM_FORCE", "1")
    xq = O.unit_gaussian(nq, D, 90)
    t = _thresholds(xb, xq)["5000"]
    D0, I0 = index.search(xq, 50)
    a = index.range_search(xq, t)
    b = index.range_search(xq, t)
    for x, y in zip(a, b):
        assert x.tobytes() == y.tobytes()
    D1, I1 = index.search(xq, 50)
    assert D0.tobytes() == D1.tobytes() and I0.tobytes() == I1.tobytes()


def test_result_outlives_index():
    L = _capi.lib()
    xb = O.unit_gaussian(1000, 32, 3)
    xq = O.unit_gaussian(2, 32, 4)
    h = C.c_void_p()
    _capi.check(L.wb_flat_create(32, 0, C.byref(h)))
    _capi.check(L.wb_add_with_ids(h, 1000, _capi.ptr(xb), None))
    lims = np.zeros(3, np.int64)
    res = C.c_void_p()
    _capi.check(L.wb_range_search(h, None, 2, _capi.ptr(xq), 0.1, 1, _capi.ptr(lims), C.byref(res)))
    _capi.check(L.wb_free(h))
    Dg = np.empty(int(lims[-1]), np.float32)
    Ig = np.empty(int(lims[-1]), np.int64)
    _capi.check(L.wb_range_result_copy(res, _capi.ptr(Dg), _capi.ptr(Ig)))
    _capi.check(L.wb_range_result_free(res))
    lr, Dr, Ir = range_search(xb, xq, np.float32(0.1))
    assert abs(int(lims[-1]) - int(lr[-1])) <= 2 and lims[-1] > 0
    for i in range(2):
        a, b = int(lims[i]), int(lims[i + 1])
        assert np.all(np.abs(Dg[a:b] - xb[Ig[a:b]].astype(np.float64) @ xq[i].astype(np.float64)) <= 1e-5)
        assert np.all(Dg[a:b] > np.float32(0.1))
