"""Selector construction and validation of the filtered-search API (no GPU: nothing here reaches the device)."""
import numpy as np
import pytest

from wise_b200 import faiss_compat as faiss


def test_batch_forms_sort_and_deduplicate():
    a = faiss.IDSelectorBatch([7, 3, 3, 11, 7])
    assert a.ids.dtype == np.int64 and a.ids.tolist() == [3, 7, 11]
    b = faiss.IDSelectorBatch(2, np.array([9, 4, 100], np.int32))  # faiss's (n, ids) form: the first n ids
    assert b.ids.tolist() == [4, 9]
    assert faiss.IDSelectorBatch(np.array([], np.int64)).ids.size == 0
    assert faiss.IDSelectorBatch([]).ids.size == 0  # an empty list (float64 to numpy) is an empty set


@pytest.mark.parametrize("bad", [[1.5, 2.0], np.array([1.0]), ["a"], [True, False]])
def test_batch_rejects_non_integer_ids(bad):
    with pytest.raises(TypeError):
        faiss.IDSelectorBatch(bad)


def test_range_and_not():
    r = faiss.IDSelectorRange(5, 9)
    assert (r.imin, r.imax) == (5, 9)
    empty = faiss.IDSelectorRange(9, 2)  # imin > imax: the empty set (the kernel tests imin <= id < imax)
    assert empty.imin > empty.imax
    with pytest.raises(TypeError):
        faiss.IDSelectorRange(1.5, 4)
    n1 = faiss.IDSelectorNot(r)
    assert n1._invert and n1._base is r
    n2 = faiss.IDSelectorNot(n1)  # Not of Not keeps what the inner selector keeps
    assert not n2._invert and n2._base is r
    with pytest.raises(TypeError):
        faiss.IDSelectorNot("not a selector")


def test_search_parameters():
    sel = faiss.IDSelectorBatch([1])
    p = faiss.SearchParameters(sel=sel)
    assert p.sel is sel
    assert faiss.SearchParameters().sel is None
    q = faiss.SearchParametersIVF(sel=sel, nprobe=12)
    assert isinstance(q, faiss.SearchParameters) and q.nprobe == 12 and q.sel is sel
    assert faiss.SearchParametersIVF().nprobe == 1  # faiss default
    with pytest.raises(TypeError):
        faiss.SearchParameters(sel=[1, 2])
