"""The fp64 range-search reference against oracle.flat_search with k = n cut at the threshold (no GPU)."""
import numpy as np
import pytest

from oracle import oracle as O
from range_oracle import ivf_range_search, range_search
from wise_b200 import _capi


def _cut(xb, xq, thresh, ids=None):
    """flat_search(k = n) keeps every row in (score desc, position asc) order; keep the fp64 scores > thresh."""
    D, I = O.flat_search(xb, xq, xb.shape[0], ids)
    pos = np.argsort(ids) if ids is not None else None
    out = []
    for i in range(len(xq)):
        p = I[i] if ids is None else pos[np.searchsorted(ids[pos], I[i])]
        s64 = xb[p].astype(np.float64) @ xq[i].astype(np.float64)
        out.append((D[i][s64 > thresh], I[i][s64 > thresh]))
    return out


@pytest.mark.parametrize("thresh", [-2.0, 0.0, 0.1, 0.3, 5.0])
def test_reference_matches_flat_search_cut(thresh):
    xb = O.unit_gaussian(500, 24, 1)
    xb[77] = xb[12]  # an exact duplicate: both rows, adjacent, lower position first
    xq = O.unit_gaussian(6, 24, 2)
    xq[0] = xb[12]
    ids = np.arange(500, dtype=np.int64)[::-1] * 3 + 5
    lims, D, I = range_search(xb, xq, thresh, ids)
    assert lims.dtype == np.uint64 and lims.shape == (7,) and lims[0] == 0
    for i, (Dc, Ic) in enumerate(_cut(xb, xq, thresh, ids)):
        a, b = int(lims[i]), int(lims[i + 1])
        np.testing.assert_array_equal(I[a:b], Ic)
        np.testing.assert_array_equal(D[a:b], Dc)
    if thresh < 1:
        a, b = int(lims[0]), int(lims[1])
        j = list(I[a:b]).index(ids[12])
        assert I[a + j + 1] == ids[77]  # the duplicate follows its original


def test_empty_results_and_nan():
    xb = O.unit_gaussian(50, 8, 3)
    xq = O.unit_gaussian(3, 8, 4)
    for t in (np.inf, np.nan, 1.5):
        lims, D, I = range_search(xb, xq, t)
        assert lims.tolist() == [0, 0, 0, 0] and D.size == 0 and I.size == 0
    lims, D, I = range_search(xb, xq[:0], 0.0)
    assert lims.tolist() == [0]


def test_ivf_reference_with_every_list_is_flat():
    xb = O.unit_gaussian(400, 16, 5)
    cent = O.unit_gaussian(8, 16, 6)
    xq = O.unit_gaussian(4, 16, 7)
    assign = O.ivf_assign(xb, cent)
    a = ivf_range_search(xb, None, assign, cent, xq, 0.1, 8)
    b = range_search(xb, xq, 0.1)
    for x, y in zip(a, b):
        np.testing.assert_array_equal(x, y)
    l1, _, I1 = ivf_range_search(xb, None, assign, cent, xq, 0.1, 1)
    assert l1[-1] < b[0][-1]
    _, probes = O.ivf_coarse(xq, cent, 1)
    for i in range(4):
        assert np.all(assign[I1[int(l1[i]):int(l1[i + 1])]] == probes[i][0])


def test_range_search_is_declared():
    for name in ("wb_range_search", "wb_range_result_copy", "wb_range_result_free"):
        assert name in _capi.SIGNATURES
