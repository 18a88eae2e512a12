"""The bf16 filter of flat searches of 1-2 queries over large stores (DESIGN.md "K1"): the scan streams a bf16 image of
the store and re-scores in fp32 every (row, query) pair whose approximate score can reach the threshold.  Its results
must be the fp32 scan's byte for byte.  The fp32 scan of the same build is a batch of 5 queries on the same index (the
first ones being the queries under test): K1 scores every (row, query) pair with the same arithmetic at any batch
size, and never uses the image above 2 queries.  The stores have narrow rows so that they pass the image's size
cutoff (16384 rows per SM) cheaply."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import oracle as O
from wise_b200 import _capi
from wise_b200 import faiss_compat as faiss

pytestmark = pytest.mark.gpu
FLT_MAX = np.finfo(np.float32).max


@pytest.fixture(scope="module")
def nbig():
    return 16384 * torch.cuda.get_device_properties(0).multi_processor_count + 1000


def _stats(index):
    s, r = C.c_int64(0), C.c_int64(0)
    _capi.check(_capi.lib().wb_flat_bf16_stats(index._h, C.byref(s), C.byref(r)))
    return s.value, r.value


def _flat(xb, ids):
    index = faiss.IndexIDMap(faiss.IndexFlatIP(xb.shape[1]))
    index.add_with_ids(xb, ids)
    return index


def _image_vs_fp32(xb, xq, k, params=None, index=None):
    """(D, positions) of the image path on a store holding xb, asserted byte-identical to the fp32 scan's."""
    n = xb.shape[0]
    ids = np.arange(n, dtype=np.int64) * 5 + 3
    index = index or _flat(xb, ids)
    kw = {"params": params} if params is not None else {}
    s0, r0 = _stats(index)
    D, I = index.search(xq, k, **kw)
    s1, r1 = _stats(index)
    assert s1 == s0 + 1, "the search did not take the bf16 image"
    nq = len(xq)
    Dr, Ir = index.search(np.concatenate([xq, xq[:1].repeat(5 - nq, 0)]), k, **kw)
    assert _stats(index) == (s1, r1), "a batch of 5 must take the fp32 scan"
    assert D.tobytes() == Dr[:nq].tobytes() and I.tobytes() == Ir[:nq].tobytes()
    return D, np.where(I >= 0, (I - 3) // 5, -1)


@pytest.mark.parametrize("d,nq,k", [(16, 1, 100), (16, 2, 100), (12, 2, 10), (36, 1, 1000), (8, 2, 50)])
def test_image_matches_fp32_scan_bytes(nbig, d, nq, k):
    xb = O.clustered_unit(nbig, d, 64, d)
    xq = O.clustered_unit(nq, d, 64, nq + k)
    D, P = _image_vs_fp32(xb, xq, k)
    Dr, Ir = O.flat_search(xb, xq, k)
    O.compare_topk(D, P, Dr, Ir)


def _mixed_scale(n, d, seed):
    rng = np.random.default_rng(seed)
    return (O.unit_gaussian(n, d, seed) * (10.0 ** rng.uniform(-6, 6, size=(n, 1)))).astype(np.float32)


def _subnormal(n, d, seed):
    x = O.unit_gaussian(n, d, seed) * np.float32(1e-39)  # every element an fp32 subnormal or zero
    return x.astype(np.float32)


def _near_flt_max(n, d, seed):
    x = O.unit_gaussian(n, d, seed)
    x[::97, 0] = FLT_MAX * np.float32(1 - 2.0 ** -10)  # within one bf16 ulp of FLT_MAX: its bf16 rounds to Inf
    x[1::97, 0] = -FLT_MAX
    return x


def _tiny(n, d, seed):
    x = O.unit_gaussian(n, d, seed) * np.float32(1e-25)  # normal floats whose squares underflow: norm2_max is 0
    return x.astype(np.float32)


def _bf16_equal_pairs(n, d, seed):
    """Rows 2i and 2i + 1 have equal bf16 images (low 16 bits 0x0001 / 0x0002 both round down) but different fp32
    values; every element of row 2i + 1 is the larger in magnitude."""
    u = O.clustered_unit(n // 2, d, 8, seed).view(np.uint32) & np.uint32(0xFFFF0000)
    x = np.empty((n, d), np.uint32)
    x[0::2], x[1::2] = u | np.uint32(1), u | np.uint32(2)
    return x.view(np.float32)


@pytest.mark.parametrize("case", ["clustered", "mixed_scale", "subnormal", "tiny", "near_flt_max", "bf16_equal_pairs"])
@pytest.mark.parametrize("nq", [1, 2])
def test_bound_cases(nbig, case, nq):
    n, d, k = nbig, 16, 50
    xb = {"clustered": lambda: O.clustered_unit(n, d, 16, 5), "mixed_scale": lambda: _mixed_scale(n, d, 6),
          "subnormal": lambda: _subnormal(n, d, 7), "tiny": lambda: _tiny(n, d, 14), "near_flt_max": lambda: _near_flt_max(n, d, 8),
          "bf16_equal_pairs": lambda: _bf16_equal_pairs(n, d, 9)}[case]()
    xq = O.clustered_unit(nq, d, 16, 10) if case != "mixed_scale" else _mixed_scale(nq, d, 11)
    if case == "near_flt_max":
        xq[:, 0] = 0.0  # the huge column does not enter the scores: they stay finite
    if case == "bf16_equal_pairs":
        xq[0] = xb[101]  # row 100 is its bf16 twin with the lower exact score
    D, P = _image_vs_fp32(xb, xq, k)
    if case in ("clustered", "near_flt_max", "bf16_equal_pairs"):
        Dr, Ir = O.flat_search(xb, xq, k)
        O.compare_topk(D, P, Dr, Ir)
    if case == "bf16_equal_pairs":
        assert P[0, 0] == 101 and D[0, 0] > D[0, 1]


def test_nan_rows_and_queries(nbig):
    n, d, k = nbig, 16, 50
    xb = O.clustered_unit(n, d, 16, 12)
    bad = np.array([0, 17, 4096, n - 1])
    xb[bad, 5] = np.nan
    xb[bad[1], :] = np.nan
    xq = O.clustered_unit(2, d, 16, 13)
    D, P = _image_vs_fp32(xb, xq, k)
    clean = np.setdiff1d(np.arange(n), bad)
    Dr, Ir = O.flat_search(xb[clean], xq, k, clean)
    O.compare_topk(D, P, Dr, Ir)
    xq[1, 3] = np.nan  # every score of that query is NaN: it returns the empty row
    D2, P2 = _image_vs_fp32(xb, xq, k)
    assert np.all(P2[1] == -1) and np.all(D2[1] == O.NEG_FLT_MAX)


def test_adds_after_the_image_is_built(nbig):
    """add -> search -> add (past the capacity, then within it) -> search: rows added after the image was built are
    found."""
    d, k = 16, 10
    xb = O.unit_gaussian(3 * nbig, d, 21)
    index = faiss.IndexFlatIP(d)
    index.add(xb[:nbig])
    D, I = index.search(xb[:2], k)
    assert I[:, 0].tolist() == [0, 1]
    for lo, hi, probe in [(nbig, nbig + 1000, [nbig + 1, nbig + 999]),      # past the capacity: the image is rebuilt
                          (nbig + 1000, nbig + 2000, [nbig + 1500, 7]),     # within the grown capacity: extended
                          (nbig + 2000, 3 * nbig, [3 * nbig - 1, 2 * nbig])]:
        index.add(xb[lo:hi])
        D, I = index.search(xb[probe], k)
        assert I[:, 0].tolist() == probe
        Dr, Ir = O.flat_search(xb[:hi], xb[probe], k)
        O.compare_topk(D, I, Dr, Ir)
    assert _stats(index)[0] == 4


def test_masked_filter_takes_the_image(nbig):
    n, d, k = nbig, 16, 100
    xb = O.clustered_unit(n, d, 32, 31)
    ids = np.arange(n, dtype=np.int64) * 5 + 3
    index = _flat(xb, ids)
    sel_ids = np.random.default_rng(5).choice(ids, n // 2, replace=False)
    xq = O.clustered_unit(2, d, 32, 32)
    D, P = _image_vs_fp32(xb, xq, k, params=faiss.SearchParameters(sel=faiss.IDSelectorBatch(sel_ids)), index=index)
    keep = np.isin(ids, sel_ids)
    Dr, Ir = O.flat_search(xb[keep], xq, k, np.nonzero(keep)[0])
    O.compare_topk(D, P, Dr, Ir)


def test_paths_without_the_image(nbig):
    """IVF stores, compacted filters, batches of 3+ queries and small stores do not use (or build) an image."""
    n, d, k = nbig, 16, 20
    xb = O.clustered_unit(n, d, 16, 41)
    index = _flat(xb, np.arange(n, dtype=np.int64))
    for nq in (3, 4, 5, 8):
        index.search(O.clustered_unit(nq, d, 16, nq), k)
    index.search(xb[:2], k, params=faiss.SearchParameters(sel=faiss.IDSelectorBatch(np.arange(100))))
    assert _stats(index) == (0, 0)
    index.search(xb[:1], k)
    s, r = _stats(index)
    assert s == 1 and 0 < r < n // 2  # re-scored pairs: a small part of the rows
    small = _flat(xb[:100000], np.arange(100000, dtype=np.int64))
    small.search(xb[:1], k)
    assert _stats(small) == (0, 0)
    q = faiss.IndexFlatIP(d)
    ivf = faiss.IndexIVFFlat(q, d, 16)
    ivf.train(xb[:100000])
    ivf.add(xb)
    ivf.nprobe = 4
    ivf.search(xb[:1], k)
    assert _stats(ivf) == (0, 0)
