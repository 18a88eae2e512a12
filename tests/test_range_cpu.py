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


def test_check_accepts_the_reference_and_rejects_errors():
    """range_oracle.check, the rule every GPU range test applies: it accepts the fp64 reference's own output and
    rejects a missing row, a row of another query, a wrong score and a broken tie order."""
    from range_oracle import check
    xb = O.unit_gaussian(3000, 16, 1)
    xb[2500] = xb[7]
    xq = np.concatenate([O.unit_gaussian(5, 16, 2), xb[7:8]])
    ids = np.arange(3000, dtype=np.int64) * 2 + 1
    t = np.float32(0.3)
    lims, D, I = range_search(xb, xq, t, ids)
    assert lims[-1] > 50
    check(lims, D, I, xb, xq, t, ids)
    check(lims, D, I, xb, xq, t, ids, cand=[np.arange(3000)] * len(xq))
    a = int(lims[-2])  # the query equal to row 7: rows 7 and 2500 lead, tied
    assert I[a] == ids[7] and I[a + 1] == ids[2500]
    bad = [(lims, D, np.roll(I, 1)), (lims, D + np.float32(1e-3) * (np.arange(D.size) == 3), I)]
    I2 = I.copy()
    I2[a], I2[a + 1] = I[a + 1], I[a]
    bad.append((lims, D, I2))
    l3 = lims.copy()
    l3[1:] -= 1
    l3[0] = 0
    bad.append((l3, D[1:], I[1:]))  # query 0 loses its best row
    for lb, Db, Ib in bad:
        with pytest.raises(AssertionError):
            check(lb, Db, Ib, xb, xq, t, ids)
