"""A numpy model of the int8 filter of K1 (DESIGN.md "K1"): the store is streamed as its int8 image (a per-row scale s,
codes n, and the header's resid >= |x - s n| and xhat >= |s n|), the query is scaled by a power of two and rounded to
fp16, and a (row, query) pair is skipped only when `approx + margin < threshold`.  The image build is
int8_image_kernel's and the margin the kernel's (scan.cuh, consumer prologue), both in the kernel's fp32 arithmetic;
these tests check, against fp64, that the margin bounds |exact_fp32 - approx| on the inputs where it is easiest to get
wrong, so that a skipped row can never have reached the threshold."""
import numpy as np
import pytest

from oracle import oracle as O

F32 = np.float32
FLT_MAX = np.finfo(F32).max
TINY = np.finfo(F32).tiny


def _round_up_f32(v):
    """fp64 -> the smallest fp32 >= v (+Inf beyond FLT_MAX): __double2float_ru."""
    with np.errstate(over="ignore"):
        f = v.astype(F32)
    lo = f.astype(np.float64) < v
    f[lo] = np.nextafter(f[lo], F32(np.inf))
    return f


def build_image(xb):
    """int8_image_kernel: (s, codes n, resid, xhat) of every row."""
    xb = np.asarray(xb, F32)
    with np.errstate(invalid="ignore"):
        a = np.abs(xb)
        bad = ~np.all(a <= FLT_MAX, axis=1)
        mx = np.where(bad, F32(0), a.max(axis=1, initial=F32(0)))
    s = np.maximum(mx / F32(127), F32(2.0 ** -149)).astype(F32)
    s[mx == 0] = 0
    s[bad] = np.nan
    safe = np.where(s > 0, s, F32(1))[:, None]
    n = np.clip(np.rint(np.where(bad[:, None], F32(0), xb) / safe), -127, 127).astype(F32)
    n[~(s > 0)] = 0
    with np.errstate(invalid="ignore"):
        d = xb.astype(np.float64) - s.astype(np.float64)[:, None] * n.astype(np.float64)
    up = 1.0 + 2.0 ** -30
    resid = _round_up_f32(np.sqrt((d * d).sum(axis=1)) * up)
    xhat = _round_up_f32(s.astype(np.float64) * np.sqrt((n.astype(np.float64) ** 2).sum(axis=1)) * up)
    resid[bad] = np.inf
    xhat[bad] = 0
    return s, n, resid, xhat


def _pow2(e):
    return F32(2.0 ** int(e))


def query_terms(q, ld):
    """The consumer prologue: the fp16 query q^ and {A, B, C, 2^-e, T}, in fp32."""
    q = np.asarray(q, F32)
    with np.errstate(over="ignore", invalid="ignore"):
        s2 = (q * q).sum(dtype=F32)
        a = np.abs(q)
        mx = F32(np.nanmax(a)) if a.size and not np.all(np.isnan(a)) else F32(0)
        e = min(141 - int((np.array(mx, F32).view(np.uint32) >> 23) & 0xFF), 126)
        v = (q * _pow2(63) * _pow2(e - 63)) if e > 63 else q * _pow2(e)
        v = v.astype(F32)
        qh = v.astype(np.float16)
        d = v - qh.astype(F32)
        d2 = (d * d).sum(dtype=F32)
        h = F32(ld + 64)
        lost = F32(ld) * F32(2.0 ** -149)
        g = F32(2) * F32(1.01) * h * F32(2.0 ** -24) + F32(2.0 ** -21)
        qs = _pow2(-e)
        qn = np.sqrt(s2 + lost)
        dqn = (np.sqrt(d2 + lost) + np.sqrt(F32(ld)) * F32(2.0 ** -149)) * qs + F32(2.0 ** -149)
        T = qn + dqn
        A = F32(1.001) * (qn + g * T)
        B = F32(1.001) * (dqn + g * T)
        C = F32(1.001) * h * F32(2.0 ** -148)
    return qh, F32(A), F32(B), F32(C), F32(qs), F32(T)


def approx_and_margin(img, q, ld):
    s, n, resid, xhat = img
    qh, A, B, C, qs, T = query_terms(q, ld)
    with np.errstate(over="ignore", invalid="ignore", under="ignore"):
        acc = (n * qh.astype(F32)).sum(axis=1, dtype=F32)  # exact products (fp16 x int8), fp32 sums
        approx = ((acc * qs) * s) if qs > 1 else ((acc * s) * qs)
        margin = (A * resid + (B * xhat + C)).astype(F32)
        margin[~(T * (resid + xhat) <= F32(2.0 ** 126))] = np.inf
    return approx.astype(F32), margin


def fp32_dot(x, q):
    """fp32 inner products without BLAS (no flush of subnormals)."""
    with np.errstate(over="ignore", invalid="ignore", under="ignore"):
        return (x.astype(F32) * q.astype(F32)).sum(axis=1, dtype=F32)


def check_bound(xb, xq):
    """|exact_fp32 - approx| <= margin for every pair the filter may skip; returns the largest ratio."""
    xb = np.asarray(xb, F32)
    ld = xb.shape[1]
    img = build_image(xb)
    worst = 0.0
    for q in np.asarray(xq, F32):
        approx, m = approx_and_margin(img, q, ld)
        exact = fp32_dot(xb, q)
        with np.errstate(over="ignore", invalid="ignore"):
            skippable = np.isfinite(approx) & np.isfinite(m) & np.isfinite(approx + m)
        # an exact score of +-Inf must be queued; a NaN one is never inserted by the fp32 scan
        assert not np.any(skippable & np.isinf(exact))
        ok = skippable & np.isfinite(exact)
        err = np.abs(exact[ok].astype(np.float64) - approx[ok].astype(np.float64))
        assert np.all(err <= m[ok].astype(np.float64)), (err.max(), m[ok][np.argmax(err - m[ok])])
        # the skip rule itself: approx + margin < exact never happens
        assert not np.any(approx[ok] + m[ok] < exact[ok])
        if ok.any():
            r = err / np.maximum(m[ok].astype(np.float64), 1e-300)
            worst = max(worst, float(r.max()))
    return worst


def test_image_build_model():
    x = np.array([[1.0, -0.5, 0.25, 0.0], [0.0] * 4, [2.0 ** -147, -(2.0 ** -149), 0.0, 0.0],
                  [FLT_MAX, -FLT_MAX, 1.0, 0.0], [1.0, np.nan, 0.0, 0.0], [np.inf, 0.0, 0.0, 0.0]], F32)
    s, n, resid, xhat = build_image(x)
    assert s[0] == F32(1.0) / F32(127) and n[0, 0] == 127 and n[0, 1] == -64
    assert s[1] == 0 and np.all(n[1] == 0) and resid[1] == 0 and xhat[1] == 0
    # a subnormal row: s = the smallest subnormal, exact codes, no residual
    assert s[2] == F32(2.0 ** -149) and resid[2] == 0 and np.all(np.abs(n[2]) <= 127)
    assert np.isfinite(resid[3]) and np.isinf(xhat[3])  # |s n| ~ FLT_MAX sqrt(2): +Inf, not a wrapped value
    assert np.isnan(s[4]) and np.isinf(resid[4]) and np.isnan(s[5]) and np.isinf(resid[5])
    # the header bounds hold in exact arithmetic
    ok = np.isfinite(s)
    d = x[ok].astype(np.float64) - s[ok].astype(np.float64)[:, None] * n[ok]
    assert np.all(resid[ok].astype(np.float64) >= np.sqrt((d * d).sum(axis=1)))


def test_clustered_unit_rows():
    xb = O.clustered_unit(20000, 768, 16, 1)
    xq = O.clustered_unit(4, 768, 16, 2)
    w = check_bound(xb, xq)
    assert 0.01 < w < 1.0  # the bound holds and is not vacuous


def test_one_dominant_element():
    """Every other element quantises to 0: the residual is the whole rest of the row."""
    xb = (O.unit_gaussian(5000, 256, 3) * F32(1e-3)).astype(F32)
    xb[:, 0] = 1.0
    img = build_image(xb)
    assert np.all(img[1][:, 1:] == 0)
    check_bound(xb, O.unit_gaussian(3, 256, 4))


def test_wildly_mixed_scale():
    rng = np.random.default_rng(3)
    xb = O.unit_gaussian(5000, 256, 3) * (10.0 ** rng.uniform(-8, 8, size=(5000, 1)))
    xb *= 10.0 ** rng.uniform(-3, 3, size=(1, 256))  # columns of different scale too
    xq = O.unit_gaussian(3, 256, 4) * (10.0 ** rng.uniform(-8, 8, size=(3, 1)))
    check_bound(xb.astype(F32), xq.astype(F32))


def test_subnormal_rows():
    xb = (O.unit_gaussian(5000, 128, 5) * F32(1e-39)).astype(F32)
    assert np.all(np.abs(xb) < TINY)
    check_bound(xb, O.unit_gaussian(3, 128, 6))
    both = np.concatenate([xb, O.unit_gaussian(100, 128, 7) * F32(1e-30)])
    check_bound(both.astype(F32), O.unit_gaussian(3, 128, 8))


def test_tiny_normal_rows_whose_squares_underflow():
    xb = (O.unit_gaussian(5000, 128, 9) * F32(1e-25)).astype(F32)
    assert np.all(np.abs(xb[xb != 0]) >= TINY) and np.all((xb * xb).sum(axis=1, dtype=F32) == 0)
    check_bound(xb, O.unit_gaussian(3, 128, 10))
    check_bound(xb, (O.unit_gaussian(3, 128, 11) * F32(1e-20)).astype(F32))


def test_rows_near_flt_max():
    xb = O.unit_gaussian(2000, 64, 11)
    xb[::50, 0] = FLT_MAX * F32(1 - 2.0 ** -20)
    xb[1::50, :8] = -FLT_MAX
    q = O.unit_gaussian(2, 64, 12)
    q[:, :8] = 0.0
    img = build_image(xb)
    _, m = approx_and_margin(img, q[0], 64)
    assert np.all(np.isinf(m[::50])) and np.all(np.isinf(m[1::50]))  # always re-scored
    check_bound(xb, q)
    check_bound(xb, O.unit_gaussian(2, 64, 13))  # scores that overflow


def test_all_zero_rows():
    xb = O.clustered_unit(3000, 64, 8, 14)
    xb[::3] = 0.0
    approx, m = approx_and_margin(build_image(xb), O.unit_gaussian(1, 64, 15)[0], 64)
    assert np.all(approx[::3] == 0) and np.all(m[::3] > 0)
    check_bound(xb, O.unit_gaussian(2, 64, 15))


def test_nan_and_inf_rows_are_always_rescored():
    xb = O.clustered_unit(3000, 64, 8, 16)
    xb[5, 3] = np.nan
    xb[6, :] = np.nan
    xb[7, 0] = np.inf
    xb[8, 9] = -np.inf
    for q in O.unit_gaussian(2, 64, 17):
        approx, m = approx_and_margin(build_image(xb), q, 64)
        assert np.all(np.isnan(approx[5:9]))
    check_bound(xb, O.unit_gaussian(2, 64, 17))


def test_queries_with_a_wide_dynamic_range():
    xb = O.clustered_unit(4000, 128, 8, 18)
    rng = np.random.default_rng(19)
    xq = O.unit_gaussian(6, 128, 20) * (10.0 ** rng.uniform(-6, 6, size=(6, 128)))  # many elements off fp16's range
    xq[0] *= 1e30
    xq[1] *= 1e-35
    xq[2, :64] = 0.0
    xq[3] = 0.0
    xq[4, 0] = FLT_MAX / 4
    check_bound(xb, xq.astype(F32))
    qh, A, B, C, qs, T = query_terms(xq[5].astype(F32), 128)  # elements of 1e-6..1e6: scaled into fp16 range
    assert np.all(np.isfinite(qh.astype(F32))) and np.isfinite(A)


def test_nan_and_inf_queries():
    xb = O.clustered_unit(1000, 32, 8, 21)
    for bad in (np.nan, np.inf):
        q = O.unit_gaussian(1, 32, 22)[0]
        q[3] = bad
        approx, m = approx_and_margin(build_image(xb), q, 32)
        with np.errstate(invalid="ignore"):
            assert not np.any(np.isfinite(approx) & np.isfinite(m) & np.isfinite(approx + m))


def test_int8_equal_pairs_with_different_exact_scores():
    """Rows whose codes and scales are equal but whose exact scores differ: only re-scoring can order them."""
    a = O.clustered_unit(2000, 128, 8, 23)
    b = np.nextafter(a, np.copysign(F32(np.inf), a))  # one ulp larger in magnitude ...
    top = np.argmax(np.abs(a), axis=1)
    b[np.arange(len(a)), top] = a[np.arange(len(a)), top]  # ... except the largest element: the same scale
    ia, ib = build_image(a), build_image(b)
    same = (ia[0] == ib[0]) & np.all(ia[1] == ib[1], axis=1)
    assert same.sum() > 1000
    q = b[7:8].copy()
    assert fp32_dot(b, q[0])[7] > fp32_dot(a, q[0])[7]
    check_bound(np.concatenate([a, b]), q)


@pytest.mark.parametrize("seed", range(3))
def test_coherent_errors_stay_inside_the_margin(seed):
    """All-positive rows and query: the rounding errors of one row cannot cancel."""
    xb = np.abs(O.unit_gaussian(4000, 512, 20 + seed))
    xq = np.abs(O.unit_gaussian(2, 512, 30 + seed))
    w = check_bound(xb, xq)
    assert 0.01 < w < 1.0
