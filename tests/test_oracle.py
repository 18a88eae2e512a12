"""CPU tests of the oracle (test infrastructure): its two implementations against each other,
against the committed golden fixtures, and the comparison harness itself."""
import os

import numpy as np
import pytest

from oracle import cpu as C
from oracle import oracle as O

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def test_golden_flat_small_both_oracles():
    g = np.load(os.path.join(GOLD, "flat_small.npz"))
    k = int(g["k"])
    D, I = O.flat_search(g["xb"], g["xq"], k, g["ids"])
    assert np.array_equal(I, g["I"]) and np.array_equal(D, g["D"])
    for mt in (False, True):
        D2, I2 = C.flat_search(g["xb"], g["xq"], k, g["ids"], mt=mt)
        O.compare_topk(D2, I2, g["D"], g["I"])
    # query 3 is row 5 itself, which has an exact duplicate at row 205: lowest position first
    assert g["I"][3, 0] == 5 * 7 + 3 and g["I"][3, 1] == 205 * 7 + 3
    assert g["D"][3, 0] == g["D"][3, 1]


@pytest.mark.parametrize("n,d,nq,k", [(1000, 64, 3, 5), (5, 16, 2, 10), (4096, 100, 9, 64), (2000, 768, 1, 100)])
def test_numpy_vs_c_flat(n, d, nq, k):
    xb = O.unit_gaussian(n, d, 1)
    xq = O.unit_gaussian(nq, d, 2)
    D, I = O.flat_search(xb, xq, k, chunk=777)
    for mt in (False, True):
        D2, I2 = C.flat_search(xb, xq, k, mt=mt)
        r = O.compare_topk(D2, I2, D, I)
        assert r["rows"] == nq
    if k > n:
        assert np.all(I[:, n:] == -1) and np.all(D[:, n:] == O.NEG_FLT_MAX)
        assert np.all(I[:, :n] >= 0)


def test_config1_shape_cpu():
    """BASELINE config[0]: 100k x 512, 16 queries, top-10 (the reference's own CPU-runnable case)."""
    xb = O.unit_gaussian(100000, 512, 1234)
    xq = O.unit_gaussian(16, 512, 4321)
    D, I = O.flat_search(xb, xq, 10)
    D2, I2 = C.flat_search(xb, xq, 10)
    r = O.compare_topk(D2, I2, D, I)
    assert r["exact_rows"] >= 15
    assert np.all(np.diff(D, axis=1) <= 0)


def test_empty_and_ragged():
    xq = O.unit_gaussian(2, 8, 3)
    D, I = O.flat_search(np.zeros((0, 8), np.float32), xq, 4)
    assert np.all(I == -1) and np.all(D == O.NEG_FLT_MAX)
    D, I = O.flat_search(O.unit_gaussian(3, 8, 4), xq, 4)
    assert np.all(I[:, 3] == -1) and np.all(I[:, :3] >= 0)


def test_ivf_oracles_agree_and_full_probe_equals_flat():
    n, d, nlist = 5000, 48, 32
    xb = O.clustered_unit(n, d, 40, 5)
    xq = O.clustered_unit(6, d, 40, 6)
    cent = O.kmeans_init(xb, nlist)
    a = O.ivf_assign(xb, cent)
    ids = np.arange(n, dtype=np.int64) + 1
    order = np.argsort(a, kind="stable")
    off = np.concatenate([[0], np.cumsum(np.bincount(a, minlength=nlist))])
    for nprobe in (1, 4, 32):
        D, I = O.ivf_search(xb, ids, a, cent, xq, 10, nprobe)
        D2, I2 = C.ivf_search(xb, ids, off, order, cent, xq, 10, nprobe)
        O.compare_topk(D2, I2, D, I)
    Df, If = O.flat_search(xb, xq, 10, ids)
    O.compare_topk(D, I, Df, If)  # nprobe == nlist: exhaustive


def test_faiss_random_is_mt19937():
    assert O.FaissRandom(5489).raw() == 3499211612  # first output of std::mt19937 default seed
    p = O.rand_perm(1000, 1235)
    assert sorted(p.tolist()) == list(range(1000))
    assert not np.array_equal(p, np.arange(1000))


def test_kmeans_objective_improves_and_centroids_unit():
    x = O.clustered_unit(3000, 24, 20, 9)
    c, objs = O.kmeans_train(x, 20, niter=6, spherical=True)
    assert np.allclose(np.linalg.norm(c, axis=1), 1.0, atol=1e-5)
    assert objs[-1] >= objs[0] and all(b >= a - 1e-3 for a, b in zip(objs, objs[1:]))
    # faiss's default for the IndexIVFFlat the reference builds (cp.spherical = False): centroids are plain means
    c2, _ = O.kmeans_train(x, 20, niter=6)
    assert np.all(np.linalg.norm(c2, axis=1) <= 1.0 + 1e-5) and np.any(np.linalg.norm(c2, axis=1) < 0.999)
    a2 = O.ivf_assign(x, c2)
    for l in range(20):
        if np.any(a2 == l):
            assert np.abs(O.kmeans_iteration(x, c2)[0][l] - x[a2 == l].astype(np.float64).mean(axis=0)).max() < 1e-5


def test_kmeans_split_fills_empty_cluster():
    x = O.clustered_unit(400, 16, 3, 10)
    c = O.kmeans_init(x, 8)
    c[7] = -c[0]  # a centroid nobody is closest to
    newc, assign, _, nsplit = O.kmeans_iteration(x, c, spherical=True)
    if not np.any(assign == 7):
        assert nsplit >= 1
    assert np.allclose(np.linalg.norm(newc, axis=1), 1.0, atol=1e-5)


def test_ivf_train_params_rule():
    assert O.ivf_train_params(10000) == (300, 10000)  # 3*sqrt(N) below 200k
    assert O.ivf_train_params(10_000_000) == (31620, 3_162_000)  # 10*round(sqrt(N)), 100 points per cell


def test_combined_query_is_unit():
    t, i, n = (O.unit_gaussian(1, 32, s) for s in (1, 2, 3))
    q = O.combined_query(t, i, n)
    assert q.dtype == np.float32 and abs(float(np.linalg.norm(q)) - 1) < 1e-6


def test_compare_topk_accepts_band_swaps_and_rejects_errors():
    D = np.array([[0.9, 0.5, 0.5 - 1e-7, 0.1]], np.float32)
    I = np.array([[1, 2, 3, 4]], np.int64)
    O.compare_topk(D, I, D, I)
    O.compare_topk(D, np.array([[1, 3, 2, 4]]), D, I)  # near-tie swap
    with pytest.raises(AssertionError):
        O.compare_topk(D, np.array([[2, 1, 3, 4]]), D, I)  # 0.9 vs 0.5 is not a tie
    with pytest.raises(AssertionError):
        O.compare_topk(D + np.float32(1e-4), I, D, I)  # score error > 1e-5
    with pytest.raises(AssertionError):
        O.compare_topk(D, np.array([[1, 99, 3, 4]]), D, I)  # wrong member, nowhere near the k-th boundary
    Dp = np.array([[0.9, O.NEG_FLT_MAX]], np.float32)
    O.compare_topk(Dp, np.array([[1, -1]]), Dp, np.array([[1, -1]]))
    with pytest.raises(AssertionError):
        O.compare_topk(Dp, np.array([[1, 5]]), Dp, np.array([[1, -1]]))


def test_one_term_tf32_filter_margin_bound():
    """The bound behind K2's filter epochs (DESIGN.md section 3): truncating both operands of a dot product to tf32
    (10 explicit mantissa bits, low 13 bits cleared) changes it by at most 2^-9 |x||q|; the kernel adds fp32
    accumulation slack on top.  Checked here in fp64 on random, clustered and adversarial (same-sign) vectors."""
    def tf32_trunc(a):
        return (a.astype(np.float32).view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)

    rng = np.random.default_rng(5)
    worst = 0.0
    for d in (3, 64, 768, 1024):
        x = rng.standard_normal((4000, d)).astype(np.float32) * rng.uniform(0.1, 8.0, size=(4000, 1)).astype(np.float32)
        q = rng.standard_normal((8, d)).astype(np.float32)
        x[:500] = np.abs(x[:500])  # same-sign products: the truncation errors all add up
        q[:2] = np.abs(q[:2])
        exact = x.astype(np.float64) @ q.astype(np.float64).T
        one_term = tf32_trunc(x).astype(np.float64) @ tf32_trunc(q).astype(np.float64).T
        bound = 2.0 ** -9 * np.linalg.norm(x.astype(np.float64), axis=1)[:, None] * np.linalg.norm(q.astype(np.float64), axis=1)[None, :]
        assert np.all(np.abs(exact - one_term) <= bound)
        assert np.all(one_term[:500, :2] <= exact[:500, :2])  # all-positive operands: truncation only shrinks the sum
        worst = max(worst, float((np.abs(exact - one_term) / bound).max()))
    assert 0.05 < worst <= 1.0  # the bound is within ~20x of what same-sign vectors actually reach: not vacuous


def test_chunked_fp64_references_match_the_oracle():
    """The torch fp64 references of tests/test_limits_gpu.py (run here on the CPU) agree exactly with O.flat_search /
    O.ivf_search, ties by insertion position included, across several query chunks and with k > ntotal."""
    from test_limits_gpu import coarse_fp64, ivf_topk_fp64, topk_fp64
    xb = O.unit_gaussian(700, 24, 1)
    xb[[10, 300, 650]] = xb[5]  # exact ties, decided by position
    xq = np.concatenate([O.unit_gaussian(40, 24, 2), xb[5:6]])
    ids = np.arange(700, dtype=np.int64) * 3 + 1
    for k in (1, 10, 64):
        D, I = topk_fp64(xb, xq, k, ids, device="cpu")
        Dr, Ir = O.flat_search(xb, xq, k, ids)
        assert np.array_equal(D, Dr) and np.array_equal(I, Ir), k
    assert I[-1, :4].tolist() == [ids[5], ids[10], ids[300], ids[650]]
    D, I = topk_fp64(xb[:30], xq, 64, device="cpu")
    Dr, Ir = O.flat_search(xb[:30], xq, 64)
    assert np.array_equal(D, Dr) and np.array_equal(I, Ir) and np.all(I[:, 30:] == -1)
    cent = O.unit_gaussian(16, 24, 3)
    assign = O.ivf_assign(xb, cent)
    for nprobe in (1, 3, 16):
        probes, gaps = coarse_fp64(cent, xq, nprobe, device="cpu")
        _, Pr = O.ivf_coarse(xq, cent, nprobe)
        assert np.array_equal(probes, Pr) and np.all(gaps >= 0)
        for k in (5, 200):
            D, I = ivf_topk_fp64(xb, ids, assign, probes, xq, k, device="cpu")
            Dr, Ir = O.ivf_search(xb, ids, assign, cent, xq, k, nprobe)
            assert np.array_equal(D, Dr) and np.array_equal(I, Ir), (nprobe, k)
