"""fp64 reference of range search (faiss Index::range_search, METRIC_INNER_PRODUCT [faiss-upstream]), built on the
same scoring and tie rule as oracle.flat_search / oracle.ivf_search: every candidate row whose fp64 inner product with
the query is strictly greater than `thresh`, by score descending, then insertion position ascending.
Returns (lims uint64[n+1], D float32 (the fp64 score rounded), I int64)."""
import numpy as np

from oracle import oracle as O


def _one(xb64, q64, rows, thresh, ids):
    s = xb64[rows] @ q64
    hit = s > np.float64(thresh)  # NaN never qualifies
    r, sc = rows[hit], s[hit]
    order = np.lexsort((r, -sc))
    r, sc = r[order], sc[order]
    return sc.astype(np.float32), (r if ids is None else np.asarray(ids, np.int64)[r])


def _assemble(parts, n):
    lims = np.zeros(n + 1, np.uint64)
    lims[1:] = np.cumsum([p[0].size for p in parts], dtype=np.uint64)
    D = np.concatenate([p[0] for p in parts]) if parts else np.zeros(0, np.float32)
    I = np.concatenate([p[1] for p in parts]) if parts else np.zeros(0, np.int64)
    return lims, D.astype(np.float32), I.astype(np.int64)


def range_search(xb, xq, thresh, ids=None):
    """IndexFlatIP(+IndexIDMap).range_search: every row is a candidate."""
    xb64 = np.asarray(xb, np.float64)
    rows = np.arange(xb64.shape[0])
    return _assemble([_one(xb64, np.asarray(q, np.float64), rows, thresh, ids) for q in xq], len(xq))


def check(lims, Dg, Ig, xb, xq, thresh, ids, cand=None, band=4e-6):
    """Every query's results against fp64 over its candidate rows (cand[i]: row indices; None: all rows).  Membership
    may differ from fp64 only for rows within `band` of the threshold; every returned score is within 1e-5 of fp64 and
    strictly above the threshold; equal scores come in insertion order.  Queries are checked in blocks of one score
    matrix each, so large batches stay affordable."""
    n, N = len(xq), xb.shape[0]
    assert lims.dtype == np.uint64 and lims.shape == (n + 1,) and lims[0] == 0
    assert Dg.dtype == np.float32 and Ig.dtype == np.int64 and Dg.size == Ig.size == int(lims[-1])
    lims = lims.astype(np.int64)
    assert np.all(np.diff(lims) >= 0)
    pos_of = np.full(int(ids.max()) + 1, -1, np.int64)
    pos_of[ids] = np.arange(ids.size)
    assert np.all((Ig >= 0) & (Ig < pos_of.size)) and np.all(pos_of[Ig] >= 0), "an id that is not in the index"
    P = pos_of[Ig]
    assert np.all(Dg > np.float32(thresh))
    qid = np.repeat(np.arange(n), np.diff(lims))
    same = qid[1:] == qid[:-1]
    assert np.all(np.diff(Dg.astype(np.float64))[same] <= 0), "scores must be descending"
    tie = same & (np.diff(Dg) == 0)
    assert np.all(np.diff(P)[tie] > 0), "equal scores must come in insertion order"
    xb64 = xb.astype(np.float64)
    block = max(1, min(1024, (1 << 24) // max(N, 1)))
    for b0 in range(0, n, block):
        b1 = min(n, b0 + block)
        S = np.asarray(xq[b0:b1], np.float64) @ xb64.T
        a, e = lims[b0], lims[b1]
        lq, p, d = qid[a:e] - b0, P[a:e], Dg[a:e]
        got = np.bincount(lq * N + p, minlength=(b1 - b0) * N).reshape(b1 - b0, N)
        assert got.max(initial=0) <= 1, "a row returned twice"
        if cand is None:
            ok = np.ones_like(got, bool)
        else:
            ok = np.zeros_like(got, bool)
            for i in range(b0, b1):
                ok[i - b0, cand[i]] = True
            assert not np.any((got > 0) & ~ok), "a row that is not a candidate"
        s_ret = S[lq, p]
        assert np.all(np.abs(d - s_ret) <= 1e-5)
        miss = ok & (S > thresh + band) & (got == 0)
        assert not miss.any(), f"query {b0 + int(np.nonzero(miss.any(1))[0][0])}: {int(miss.sum())} rows missing"
        assert np.all(s_ret > thresh - band)


def ivf_range_search(xb, ids, assign, centroids, xq, thresh, nprobe):
    """IndexIVFFlat.range_search: the candidates of a query are the rows of its nprobe lists (oracle.ivf_coarse)."""
    xb64 = np.asarray(xb, np.float64)
    _, probes = O.ivf_coarse(xq, centroids, nprobe)
    parts = []
    for i, q in enumerate(xq):
        rows = np.nonzero(np.isin(assign, probes[i][probes[i] >= 0]))[0]
        parts.append(_one(xb64, np.asarray(q, np.float64), rows, thresh, ids))
    return _assemble(parts, len(xq))
