"""A numpy model of the bf16 filter of K1 (DESIGN.md "K1"): the store is streamed as its bf16 image, the query stays
fp32, and a (row, query) pair is skipped only when `approx + margin < threshold`.  The margin is the kernel's
(scan.cuh, consumer prologue); these tests check, against fp64, that it bounds |exact_fp32 - approx| on the inputs
where a bf16 bound is easiest to get wrong, so that a skipped row can never have reached the threshold."""
import numpy as np
import pytest

from oracle import oracle as O

F32 = np.float32
FLT_MAX = np.finfo(F32).max


def bf16(x):
    """Round-to-nearest-even fp32 -> bf16 (kept as fp32), NaN kept: bf16_image_kernel."""
    u = np.ascontiguousarray(x, F32).view(np.uint32).astype(np.uint64)
    r = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16 << 16).astype(np.uint32).view(F32)
    return np.where(np.isnan(x), F32(np.nan), r)


def fp32_dot(x, q):
    """fp32 inner products without BLAS (no flush of subnormals)."""
    with np.errstate(over="ignore", invalid="ignore"):
        return (x.astype(F32) * q.astype(F32)).sum(axis=1, dtype=F32)


def sumsq32(x):
    with np.errstate(over="ignore", invalid="ignore"):
        return (x.astype(F32) * x.astype(F32)).sum(axis=-1, dtype=F32)


def kernel_margin(q, norm2_max, ld):
    """The margin of scan.cuh, in fp32 arithmetic."""
    with np.errstate(over="ignore", invalid="ignore"):
        c = F32(3.90625e-3) + F32(ld) * F32(1.1920929e-7) * F32(1.1) + F32(1e-5)
        lost = F32(ld) * F32(2.0 ** -149)
        qn = np.sqrt(sumsq32(q) + lost)
        return F32(1.001) * (c * qn * np.sqrt(F32(norm2_max) + lost)
                             + F32(2.0 ** -134) * (np.sqrt(F32(ld)) * qn + F32(ld)))


def norm2_max_of(xb):
    n2 = sumsq32(xb)
    n2 = n2[~np.isnan(n2)]  # row_norm2_max_kernel: fmaxf ignores a NaN row
    return F32(max(0.0, n2.max())) if n2.size else F32(0)


def check_bound(xb, xq):
    """|exact_fp32 - approx| <= margin for every pair with a finite approximation; returns the largest ratio."""
    ld = xb.shape[1]
    n2 = norm2_max_of(xb)
    xh = bf16(xb)
    worst = 0.0
    for q in xq:
        m = kernel_margin(q, n2, ld)
        exact, approx = fp32_dot(xb, q), fp32_dot(xh, q)
        ok = np.isfinite(approx) & np.isfinite(exact)
        if not np.isfinite(m):
            continue  # every row is re-scored
        err = np.abs(exact[ok].astype(np.float64) - approx[ok].astype(np.float64))
        assert np.all(err <= np.float64(m)), (err.max(), m)
        # the skip rule itself: approx + margin < exact never happens
        with np.errstate(over="ignore"):
            assert not np.any(approx[ok] + m < exact[ok])
        if m > 0 and err.size:
            worst = max(worst, float(err.max() / m))
    return worst


def test_bf16_rounding_model():
    x = np.array([1.0, 1.00390625, 1.005859375, -3.0, 2.0 ** -140, 2.0 ** -130, FLT_MAX, np.inf, np.nan, 0.0], F32)
    r = bf16(x)
    assert r[0] == 1.0 and r[1] == 1.0 and r[2] == 1.0078125 and r[3] == -3.0  # (a tie goes to even)
    assert r[4] == 0.0 and r[5] == F32(2.0 ** -130)  # subnormals: absolute rounding to multiples of 2^-133
    assert np.isinf(r[6]) and np.isinf(r[7]) and np.isnan(r[8]) and r[9] == 0.0


def test_clustered_unit_rows():
    xb = O.clustered_unit(20000, 768, 16, 1)
    xq = O.clustered_unit(4, 768, 16, 2)
    w = check_bound(xb, xq)
    assert 0.01 < w < 1.0  # the bound holds and is not vacuous


def test_wildly_mixed_scale():
    rng = np.random.default_rng(3)
    xb = O.unit_gaussian(5000, 256, 3) * (10.0 ** rng.uniform(-8, 8, size=(5000, 1)))
    xb *= 10.0 ** rng.uniform(-3, 3, size=(1, 256))  # columns of different scale too
    xq = O.unit_gaussian(3, 256, 4) * (10.0 ** rng.uniform(-8, 8, size=(3, 1)))
    check_bound(xb.astype(F32), xq.astype(F32))


def test_subnormal_rows():
    xb = (O.unit_gaussian(5000, 128, 5) * F32(1e-39)).astype(F32)
    assert np.all(np.abs(xb) < np.finfo(F32).tiny)
    assert norm2_max_of(xb) == 0.0  # the relative term alone would be zero
    check_bound(xb, O.unit_gaussian(3, 128, 6))
    both = np.concatenate([xb, O.unit_gaussian(100, 128, 7) * F32(1e-30)])
    check_bound(both.astype(F32), O.unit_gaussian(3, 128, 8))


def test_tiny_normal_rows_whose_squares_underflow():
    xb = (O.unit_gaussian(5000, 128, 9) * F32(1e-25)).astype(F32)
    assert norm2_max_of(xb) == 0.0 and np.all(np.abs(xb[xb != 0]) >= np.finfo(F32).tiny)
    # the relative term alone would be zero, yet the approximations are off by far more than the subnormal term
    q = O.unit_gaussian(3, 128, 10)
    assert np.abs(fp32_dot(xb, q[0]) - fp32_dot(bf16(xb), q[0])).max() > 1e-30
    check_bound(xb, q)


def test_rows_within_one_bf16_ulp_of_flt_max():
    xb = O.unit_gaussian(2000, 64, 11)
    xb[::50, 0] = FLT_MAX * F32(1 - 2.0 ** -10)
    assert np.isinf(bf16(xb[:1, 0]))[0]
    n2 = norm2_max_of(xb)
    assert np.isinf(n2)
    q = O.unit_gaussian(2, 64, 12)
    q[:, 0] = 0.0
    m = kernel_margin(q[0], n2, 64)
    assert np.isinf(m)  # every row is re-scored: exact, if slow
    with np.errstate(invalid="ignore"):
        approx = fp32_dot(bf16(xb), q[0])
    assert np.isnan(approx[0])  # Inf * 0: a NaN approximation, re-scored by the rule
    check_bound(xb, q)


def test_bf16_equal_pairs_with_different_exact_scores():
    u = O.clustered_unit(2000, 128, 8, 13).view(np.uint32) & np.uint32(0xFFFF0000)
    a, b = (u | np.uint32(1)).view(F32), (u | np.uint32(2)).view(F32)
    assert np.array_equal(bf16(a), bf16(b))
    xb = np.concatenate([a, b])
    q = b[7:8].copy()
    ea, eb = fp32_dot(a, q[0]), fp32_dot(b, q[0])
    assert eb[7] > ea[7]  # one approximation, two exact scores: only re-scoring can order them
    check_bound(xb, q)


def test_nan_rows_do_not_enter_the_bound():
    xb = O.clustered_unit(3000, 64, 8, 14)
    xb[5, 3] = np.nan
    assert np.isfinite(norm2_max_of(xb))
    with np.errstate(invalid="ignore"):
        assert np.isnan(fp32_dot(bf16(xb), O.unit_gaussian(1, 64, 15)[0])[5])
    check_bound(xb, O.unit_gaussian(2, 64, 15))


@pytest.mark.parametrize("seed", range(3))
def test_coherent_errors_stay_inside_the_margin(seed):
    """All-positive rows and query: the bf16 rounding errors of one row cannot cancel."""
    xb = np.abs(O.unit_gaussian(4000, 512, 20 + seed))
    xq = np.abs(O.unit_gaussian(2, 512, 30 + seed))
    w = check_bound(xb, xq)
    assert 0.01 < w < 1.0
