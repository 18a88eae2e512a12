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


def ivf_range_search(xb, ids, assign, centroids, xq, thresh, nprobe):
    """IndexIVFFlat.range_search: the candidates of a query are the rows of its nprobe lists (oracle.ivf_coarse)."""
    xb64 = np.asarray(xb, np.float64)
    _, probes = O.ivf_coarse(xq, centroids, nprobe)
    parts = []
    for i, q in enumerate(xq):
        rows = np.nonzero(np.isin(assign, probes[i][probes[i] >= 0]))[0]
        parts.append(_one(xb64, np.asarray(q, np.float64), rows, thresh, ids))
    return _assemble(parts, len(xq))
