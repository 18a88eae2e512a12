"""The int8 filter of flat searches of 1-2 queries over large stores (DESIGN.md "K1") on the inputs of
test_int8_model.py: the scan streams the int8 image of the store and re-scores in fp32 every (row, query) pair whose
approximate score can reach the threshold, so its results must be the fp32 scan's byte for byte.  The fp32 scan of the
same build is a batch of 5 queries on the same index (the first ones being the queries under test): K1 scores every
(row, query) pair with the same arithmetic at any batch size, and never uses the image above 2 queries."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import oracle as O
from wise_b200 import _capi
from wise_b200 import faiss_compat as faiss

pytestmark = pytest.mark.gpu
F32 = np.float32
FLT_MAX = np.finfo(F32).max


@pytest.fixture(scope="module")
def nbig():
    return 16384 * torch.cuda.get_device_properties(0).multi_processor_count + 1000


def _stats(index):
    s, r = C.c_int64(0), C.c_int64(0)
    _capi.check(_capi.lib().wb_flat_bf16_stats(index._h, C.byref(s), C.byref(r)))
    return s.value, r.value


def _image_vs_fp32(xb, xq, k):
    """(D, positions) of the image path on a flat store holding xb, asserted byte-identical to the fp32 scan's."""
    n = xb.shape[0]
    ids = np.arange(n, dtype=np.int64) * 5 + 3
    index = faiss.IndexIDMap(faiss.IndexFlatIP(xb.shape[1]))
    index.add_with_ids(xb, ids)
    s0, r0 = _stats(index)
    D, I = index.search(xq, k)
    s1, r1 = _stats(index)
    assert s1 == s0 + 1, "the search did not take the int8 image"
    nq = len(xq)
    Dr, Ir = index.search(np.concatenate([xq, xq[:1].repeat(5 - nq, 0)]), k)
    assert _stats(index) == (s1, r1), "a batch of 5 must take the fp32 scan"
    assert D.tobytes() == Dr[:nq].tobytes() and I.tobytes() == Ir[:nq].tobytes()
    return D, np.where(I >= 0, (I - 3) // 5, -1)


def _codes(x):
    """The scale and codes int8_image_kernel gives finite rows."""
    s = np.abs(x).max(axis=1, keepdims=True) / F32(127)
    return s, np.clip(np.rint(x / s), -127, 127)


def _store(case, n, d, seed):
    rng = np.random.default_rng(seed)
    if case == "clustered":
        return O.clustered_unit(n, d, 16, seed)
    if case == "dominant":  # every other element quantises to 0
        x = (O.unit_gaussian(n, d, seed) * F32(1e-3)).astype(F32)
        x[:, 0] = 1.0
        return x
    if case == "mixed_scale":
        return (O.unit_gaussian(n, d, seed) * (10.0 ** rng.uniform(-6, 6, size=(n, 1)))).astype(F32)
    if case == "subnormal":  # every element an fp32 subnormal or zero
        return (O.unit_gaussian(n, d, seed) * F32(1e-39)).astype(F32)
    if case == "tiny":  # normal floats whose squares underflow
        return (O.unit_gaussian(n, d, seed) * F32(1e-25)).astype(F32)
    if case == "near_flt_max":
        x = O.unit_gaussian(n, d, seed)
        x[::97, 0] = FLT_MAX * F32(1 - 2.0 ** -20)
        x[1::97, 0] = -FLT_MAX
        return x
    if case == "zero_rows":
        x = O.clustered_unit(n, d, 16, seed)
        x[::3] = 0.0
        return x
    if case == "coherent":  # all-positive rows and queries: rounding errors cannot cancel
        return np.abs(O.unit_gaussian(n, d, seed))
    raise ValueError(case)


@pytest.mark.parametrize("case", ["clustered", "dominant", "mixed_scale", "subnormal", "tiny", "near_flt_max",
                                  "zero_rows", "coherent"])
@pytest.mark.parametrize("nq", [1, 2])
def test_bound_cases(nbig, case, nq):
    n, d, k = nbig, 16, 50
    xb = _store(case, n, d, 5)
    xq = O.clustered_unit(nq, d, 16, 10)
    if case == "mixed_scale":
        xq = (xq * (10.0 ** np.array([-5.0, 5.0][:nq]))[:, None]).astype(F32)
    if case == "near_flt_max":
        xq[:, 0] = 0.0  # the huge column does not enter the scores: they stay finite
    if case == "coherent":
        xq = np.abs(xq)
    D, P = _image_vs_fp32(xb, xq, k)
    if case in ("clustered", "dominant", "near_flt_max", "zero_rows", "coherent"):
        Dr, Ir = O.flat_search(xb, xq, k)
        O.compare_topk(D, P, Dr, Ir)


@pytest.mark.parametrize("nq", [1, 2])
def test_wide_range_queries(nbig, nq):
    """Query elements far outside fp16's range, and queries whose scale spans 12 decades."""
    n, d, k = nbig, 16, 50
    xb = O.clustered_unit(n, d, 16, 15)
    rng = np.random.default_rng(16)
    xq = (O.unit_gaussian(nq, d, 17) * (10.0 ** rng.uniform(-6, 6, size=(nq, d)))).astype(F32)
    xq[0] *= F32(1e12)
    _image_vs_fp32(xb, xq, k)  # (the oracle's absolute score tolerance does not fit scores of 1e18)


def test_nan_and_inf_rows(nbig):
    n, d, k = nbig, 16, 50
    xb = O.clustered_unit(n, d, 16, 12)
    bad = np.array([0, 17, 4096, n - 1])
    xb[bad[0], 5] = np.nan
    xb[bad[1], :] = np.nan
    xb[bad[2], 3] = np.inf
    xb[bad[3], 7] = -np.inf
    xq = O.clustered_unit(2, d, 16, 13)
    D, P = _image_vs_fp32(xb, xq, k)
    assert not np.isin(P, bad[:2]).any()  # NaN scores are never results


def test_int8_equal_pairs(nbig):
    """Rows 2i and 2i + 1 differ (every element but the largest is 2^-12 larger in magnitude in row 2i + 1) and most
    pairs have equal scales and codes: one approximation, two exact scores, so the winner comes from re-scoring."""
    n, d, k = nbig, 16, 10
    a = O.clustered_unit(n // 2, d, 8, 19)
    b = (a * F32(1 + 2.0 ** -12)).astype(F32)
    top = np.argmax(np.abs(a), axis=1)
    b[np.arange(len(a)), top] = a[np.arange(len(a)), top]
    (sa, ca), (sb, cb) = _codes(a), _codes(b)
    same = np.nonzero((sa[:, 0] == sb[:, 0]) & np.all(ca == cb, axis=1))[0]
    assert len(same) > len(a) // 4
    xb = np.empty((2 * len(a), d), F32)
    xb[0::2], xb[1::2] = a, b
    j = int(same[100])
    xq = np.stack([b[j], b[int(same[200])]])
    D, P = _image_vs_fp32(xb, xq, k)
    assert P[0, 0] == 2 * j + 1 and P[0, 1] == 2 * j and D[0, 0] > D[0, 1]
    assert P[1, 0] == 2 * int(same[200]) + 1


def test_image_memory(nbig):
    """The image takes img_row_bytes(d) = 16 + d rounded up to 16 bytes per row of capacity (wb_flat_image_bytes):
    nothing before a search builds it, then (16 + 64) / 256 of the fp32 store at d = 64 and (16 + 112) / 400 at
    d = 100, whose codes are zero-padded."""
    lib = _capi.lib()
    for d, rb in ((64, 80), (100, 128)):
        n = nbig
        index = faiss.IndexFlatIP(d)
        index.add(O.clustered_unit(n, d, 16, 21))  # capacity == n
        index.search(O.clustered_unit(5, d, 16, 22), 10)  # the fp32 scan builds no image
        assert lib.wb_flat_image_bytes(index._h) == 0
        index.search(O.clustered_unit(1, d, 16, 23), 10)
        assert _stats(index)[0] == 1
        assert lib.wb_flat_image_bytes(index._h) == n * rb


@pytest.mark.parametrize("d", [20, 100])
@pytest.mark.parametrize("nq", [1, 2])
def test_padded_rows(nbig, d, nq):
    """Dimensions that are not a multiple of 16: the image row ends in zero codes, the fp16 query in zeros."""
    xb = O.clustered_unit(nbig, d, 64, d)
    xq = O.clustered_unit(nq, d, 64, d + nq)
    D, P = _image_vs_fp32(xb, xq, 100)
    Dr, Ir = O.flat_search(xb, xq, 100)
    O.compare_topk(D, P, Dr, Ir)
