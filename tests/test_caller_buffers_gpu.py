"""The caller's side of the device-pointer entry points (include/wise_b200.h, Conventions): buffers at any offset that
keeps their element type's natural alignment, nothing written outside [0, n) of an output and every slot of it
written, calls ordered on a busy caller stream, and two handles searched from two threads at once.

Every other GPU test hands the library fresh `torch.empty` buffers (256-byte aligned, exactly as long as the result)
on the current stream and synchronises after each call, so none of this is visible there.  Here each buffer is the
interior of a larger allocation (`carved`): guard bands of G elements on both sides and the interior itself start as a
sentinel bit pattern, so a write past either end, a slot never written or an input the call modified all fail the
check.  The reference of every case is the same call on fresh aligned buffers on the current stream, and the results
must be byte-identical to it; each path is also compared once with the fp64 oracle, which anchors the reference."""
import ctypes as C
import os
import threading
from contextlib import contextmanager

import numpy as np
import pytest
import torch

from oracle import oracle as O
import range_oracle as R
from wise_b200 import _capi
from wise_b200 import faiss_compat as faiss

pytestmark = pytest.mark.gpu

G = 1024  # guard elements on each side of a carved buffer
F32, I32, I64 = torch.float32, torch.int32, torch.int64
# sentinel bit patterns, written and compared through an integer view of the same width
SENTINEL = {F32: (I32, 0x7FBADBAD), I32: (I32, 0x5A5A5A5A), I64: (I64, 0x5A5A5A5A5A5A5A5A)}
NEG_FLT_MAX = np.float32(-np.finfo(np.float32).max)
K2_MAX_Q = 65536  # queries per K2 call (run_flat_any), as in test_limits_gpu.py
SLEEP_CYCLES = int(2e8)  # ~0.1 s of GPU time: orders of magnitude above the host work of one warm call


def L():
    return _capi.lib()


# ---- buffers --------------------------------------------------------------------------------------------------------
def carved(n, dtype, offset, data=None):
    """An n-element view at element `offset` inside G + offset + n + G elements, all set to the sentinel; `data` (numpy)
    fills the interior of an input.  Returns (view, check): check() asserts both guards still hold the sentinel bit for
    bit and, for an output, that no interior slot does; for an input, that its bytes did not change."""
    ity, s = SENTINEL[dtype]
    base = torch.full((G + offset + n + G,), s, dtype=ity, device="cuda")
    lo, hi = G + offset, G + offset + n
    view = base.view(dtype)[lo:hi]
    esz = view.element_size()
    assert n == 0 or view.data_ptr() % 16 == (offset * esz) % 16  # the offset is the misalignment under test
    if data is not None:
        view.copy_(torch.from_numpy(np.ascontiguousarray(data).reshape(-1)).to(dtype).cuda())
    want = base[lo:hi].clone() if data is not None else None

    def check(what=""):
        for side, g in (("front", base[:lo]), ("back", base[hi:])):
            bad = torch.nonzero(g != s)
            assert bad.numel() == 0, f"{what}: {bad.numel()} {side} guard elements overwritten, first at {int(bad[0])}"
        inner = base[lo:hi]
        if want is None:
            bad = torch.nonzero(inner == s)
            assert bad.numel() == 0, f"{what}: {bad.numel()} of {n} output slots never written, first at {int(bad[0])}"
        else:
            assert torch.equal(inner, want), f"{what}: the call modified an input buffer"

    return view, check


def run(call, bufs, offs=None):
    """call(ptrs, stream) with the buffers of `bufs` (name -> (n, dtype, numpy data or None for an output)) on the
    current stream, then a synchronisation.  offs None: fresh aligned buffers (the reference); else every buffer is
    carved at offs.get(name, 0) elements and checked.  Returns the outputs as numpy arrays."""
    views, checks = {}, []
    for name, (n, dtype, data) in bufs.items():
        if offs is None:
            views[name] = (torch.empty(n, dtype=dtype, device="cuda") if data is None else
                           torch.from_numpy(np.ascontiguousarray(data).reshape(-1)).to(dtype).cuda())
        else:
            views[name], chk = carved(n, dtype, offs.get(name, 0), data)
            checks.append((name, chk))
    call({k: v.data_ptr() for k, v in views.items()}, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    for name, chk in checks:
        chk(f"{name} at offset {offs.get(name, 0)}")
    return {name: views[name].cpu().numpy() for name, (_, _, data) in bufs.items() if data is None}


def assert_same(got, want, what):
    """Byte equality of every array in `want`, with the first differing element named."""
    for name, w in want.items():
        g = got[name]
        assert g.shape == w.shape and g.dtype == w.dtype, (what, name, g.shape, w.shape)
        if g.tobytes() != w.tobytes():
            gb, wb = g.reshape(-1).view(np.uint8), w.reshape(-1).view(np.uint8)
            j = int(np.nonzero(gb != wb)[0][0]) // g.itemsize
            raise AssertionError(f"{what}: {name} differs from the aligned call at element {j}: "
                                 f"{g.reshape(-1)[j]!r} vs {w.reshape(-1)[j]!r}")


@contextmanager
def env(**kv):
    """Environment switches of the C API (read at every call) for the duration of a block."""
    old = {k: os.environ.get(k) for k in kv}
    os.environ.update({k: str(v) for k, v in kv.items()})
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def gemm_epochs(idx):
    a, b = C.c_int64(), C.c_int64()
    _capi.check(L().wb_gemm_stats(idx._h, C.byref(a), C.byref(b)))
    return a.value


def fused(idx):
    return int(L().wb_ivf_fused_searches(idx._h))


# ---- calls ----------------------------------------------------------------------------------------------------------
def search_bufs(xq, k):
    return {"q": (xq.size, F32, xq), "D": (len(xq) * k, F32, None), "I": (len(xq) * k, I64, None)}


def search_call(idx, nq, k, nprobe=1, flt=None):
    def call(p, st):
        if flt is None:
            _capi.check(L().wb_search_dev(idx._h, nq, p["q"], k, nprobe, p["D"], p["I"], st))
        else:
            _capi.check(L().wb_search_filtered_dev(idx._h, flt, nq, p["q"], k, nprobe, p["D"], p["I"], st))
    return call


def search(idx, xq, k, offs=None, nprobe=1, flt=None):
    out = run(search_call(idx, len(xq), k, nprobe, flt), search_bufs(xq, k), offs)
    return {"D": out["D"].reshape(len(xq), k), "I": out["I"].reshape(len(xq), k)}


def range_dev(idx, xq, thresh, offs=None, nprobe=1, flt=None):
    """wb_range_search_dev from `q`, then wb_range_result_copy_dev into `D` / `I`: {lims, D, I}."""
    nq = len(xq)
    box = {}

    def rsearch(p, st):
        lims = np.zeros(nq + 1, np.int64)
        res = C.c_void_p()
        _capi.check(L().wb_range_search_dev(idx._h, flt, nq, p["q"], float(thresh), nprobe, _capi.ptr(lims),
                                            C.byref(res), st))
        box.update(lims=lims, res=res)

    run(rsearch, {"q": (xq.size, F32, xq)}, None if offs is None else {"q": offs.get("q", 0)})
    try:
        n = int(box["lims"][-1])

        def rcopy(p, st):
            _capi.check(L().wb_range_result_copy_dev(box["res"], p["D"], p["I"], st))

        out = run(rcopy, {"D": (n, F32, None), "I": (n, I64, None)},
                  None if offs is None else {"D": offs.get("D", 0), "I": offs.get("I", 0)})
    finally:
        _capi.check(L().wb_range_result_free(box["res"]))
    out["lims"] = box["lims"]
    return out


# ---- stores ---------------------------------------------------------------------------------------------------------
class Store:
    def __init__(self, idx, xb, ids, xq, assign=None, cent=None, nprobe=1):
        self.idx, self.xb, self.ids, self.xq = idx, xb, ids, xq
        self.assign, self.cent, self.nprobe = assign, cent, nprobe

    def oracle(self, xq, k, nprobe=None):
        if self.cent is None:
            return O.flat_search(self.xb, xq, k, self.ids)
        return O.ivf_search(self.xb, self.ids, self.assign, self.cent, xq, k, nprobe or self.nprobe)

    def range_cand(self, xq):
        if self.cent is None:
            return None
        _, probes = O.ivf_coarse(xq, self.cent, self.nprobe)
        return [np.nonzero(np.isin(self.assign, p[p >= 0]))[0] for p in probes]


def _flat(n, d, seed, nq):
    xb = O.unit_gaussian(n, d, seed)
    ids = np.random.default_rng(seed).permutation(n).astype(np.int64) * 3 + 1
    idx = faiss.IndexIDMap(faiss.IndexFlatIP(d))
    idx.add_with_ids(xb, ids)
    xq = O.unit_gaussian(nq, d, seed + 1)
    xq[0] = xb[5]
    return Store(idx, xb, ids, xq)


NI, DI, NLIST, NPROBE = 40_000, 128, 64, 8


@pytest.fixture(scope="module")
def stores():
    """flat768: 60000 x 768 (ld == d: aligned queries go to the kernels as they are); flat70: 20000 x 70 (ld = 72:
    queries are always staged); ivf / ivf_ug: 40000 x 128, nlist 64, regrouped list by list / left in place."""
    out = {"flat768": _flat(60_000, 768, 11, 300), "flat70": _flat(20_000, 70, 21, K2_MAX_Q + 129)}
    xb = O.clustered_unit(NI, DI, 256, 31)
    ids = np.arange(NI, dtype=np.int64) * 5 + 2
    cent = O.unit_gaussian(NLIST, DI, 32)
    assign = O.ivf_assign(xb, cent)
    xq = O.clustered_unit(64, DI, 256, 33)
    for name, contiguous in (("ivf", 1), ("ivf_ug", 0)):
        idx = faiss.IndexIVFFlat(faiss.IndexFlatIP(DI), DI, NLIST, faiss.METRIC_INNER_PRODUCT)
        idx.set_centroids(cent)
        idx.add_with_ids(xb, ids)
        idx.nprobe = NPROBE
        with env(WB_IVF_CONTIGUOUS=contiguous):
            _capi.check(L().wb_ivf_finalize(idx._h))
        out[name] = Store(idx, xb, ids, xq, assign, cent, NPROBE)
    yield out
    out.clear()


# ---- 1. alignment matrix --------------------------------------------------------------------------------------------
FULL = [dict(q=0, D=0, I=0), dict(q=1, D=2, I=1), dict(q=2, D=3, I=0), dict(q=3, D=1, I=1)]
ONE = [dict(q=0, D=0, I=0), dict(q=1, D=3, I=1)]

# name -> (store, nq, k, env, witness, offsets).  The fused IVF search is asserted at k = 10, which its tail always
# fits (a larger k may fall back to two launches).
SEARCH_PATHS = {
    "k1-nq1": ("flat768", 1, 100, {}, "k1", FULL),
    "k1-nq4": ("flat768", 4, 100, {}, "k1", FULL),
    "k1-padded-nq4": ("flat70", 4, 100, {}, "k1", ONE),
    "k2ts-nq16": ("flat768", 16, 100, {"WB_GEMM_FORCE": 1}, "k2", ONE),
    "k2ss-nq300": ("flat768", 300, 100, {"WB_GEMM_FORCE": 1}, "k2", FULL),
    "ivf-fused-nq1": ("ivf", 1, 10, {}, "fused", ONE),
    "ivf-fused-nq4": ("ivf", 4, 10, {}, "fused", ONE),
    "ivf-twolaunch-nq4": ("ivf", 4, 100, {"WB_IVF_FUSE_COARSE": 0}, "unfused", ONE),
    "ivf-listmajor-nq64": ("ivf", 64, 100, {"WB_IVF_LISTMAJOR": 1}, "unfused", ONE),
    "ivf-querymajor-nq64": ("ivf", 64, 100, {"WB_IVF_LISTMAJOR": 0}, "unfused", ONE),
    "ivf-ungrouped-fused-nq4": ("ivf_ug", 4, 10, {}, "fused", ONE),
    "ivf-ungrouped-nq64": ("ivf_ug", 64, 100, {}, "unfused", ONE),
}
SEARCH_CASES = [(p, i) for p, spec in SEARCH_PATHS.items() for i in range(len(spec[-1]))]


def _witness(st, kind):
    return gemm_epochs(st.idx) if kind in ("k1", "k2") else fused(st.idx)


def _assert_witness(kind, before, after, what):
    if kind == "k1":
        assert after == before, f"{what}: took the tensor-core path"
    elif kind == "k2":
        assert after > before, f"{what}: did not take the tensor-core path"
    elif kind == "fused":
        assert after == before + 1, f"{what}: not one fused IVF search"
    else:
        assert after == before, f"{what}: took the fused IVF search"


@pytest.mark.parametrize("path,oi", SEARCH_CASES, ids=[f"{p}-off{i}" for p, i in SEARCH_CASES])
def test_search_alignment(stores, path, oi):
    name, nq, k, sw, kind, offsets = SEARCH_PATHS[path]
    st = stores[name]
    xq = st.xq[:nq]
    offs = offsets[oi]
    with env(**sw):
        want = search(st.idx, xq, k, nprobe=st.nprobe)
        w0 = _witness(st, kind)
        got = search(st.idx, xq, k, offs, nprobe=st.nprobe)
        _assert_witness(kind, w0, _witness(st, kind), path)
    assert_same(got, want, f"{path} {offs}")
    if oi == 0:
        O.compare_topk(want["D"], want["I"], *st.oracle(xq, k), band=4e-6)


FILTERS = {"mask": lambda ids: faiss.IDSelectorRange(0, int(np.median(ids))),
           "compact": lambda ids: faiss.IDSelectorBatch(ids[::20])}
FILTER_CASES = [("mask", 4, {}), ("compact", 4, {}), ("mask", 16, {"WB_GEMM_FORCE": 1})]


@pytest.mark.parametrize("fname,nq,sw", FILTER_CASES, ids=["mask-k1", "compact-k1", "mask-k2"])
@pytest.mark.parametrize("oi", [0, 1])
def test_filtered_search_alignment(stores, fname, nq, sw, oi):
    st = stores["flat768"]
    sel = FILTERS[fname](st.ids)
    flt = sel._filter(st.idx._hd)
    k, xq = 100, st.xq[:nq]
    with env(**sw):
        want = search(st.idx, xq, k, flt=flt)
        got = search(st.idx, xq, k, ONE[oi], flt=flt)
    assert_same(got, want, f"filtered {fname} nq={nq} {ONE[oi]}")
    if oi == 0:
        keep = np.isin(st.ids, sel.ids) if fname == "compact" else (st.ids >= sel.imin) & (st.ids < sel.imax)
        O.compare_topk(want["D"], want["I"], *O.flat_search(st.xb[keep], xq, k, st.ids[keep]), band=4e-6)


def _thresh(st, xq, hits):
    """A threshold with about `hits` rows above it for query 0."""
    s = np.sort(st.xb.astype(np.float64) @ xq[0].astype(np.float64))[::-1]
    return float(s[hits])


RANGE_CASES = [("flat768", 4, {}), ("flat768", 16, {"WB_GEMM_FORCE": 1}), ("ivf", 4, {})]


@pytest.mark.parametrize("name,nq,sw", RANGE_CASES, ids=["flat-k1", "flat-k2", "ivf"])
@pytest.mark.parametrize("oi", [0, 1])
def test_range_search_alignment(stores, name, nq, sw, oi):
    st = stores[name]
    xq = st.xq[:nq]
    t = _thresh(st, xq, 300)
    with env(**sw):
        want = range_dev(st.idx, xq, t, nprobe=st.nprobe)
        got = range_dev(st.idx, xq, t, ONE[oi], nprobe=st.nprobe)
    assert want["lims"][-1] > nq
    assert_same(got, want, f"range {name} nq={nq} {ONE[oi]}")
    if oi == 0:
        R.check(want["lims"].astype(np.uint64), want["D"], want["I"], st.xb, xq, t, st.ids, st.range_cand(xq))


def _sorted_parts(rng, P, nq, k, valid):
    """P sorted top-k lists [P][nq][k] over a few score levels (ties inside and across parts); part p holds valid[p]
    entries per query, then (-FLT_MAX, -1) padding."""
    D = np.full((P, nq, k), NEG_FLT_MAX, np.float32)
    I = np.full((P, nq, k), -1, np.int64)
    for p in range(P):
        for q in range(nq):
            v = valid[p]
            D[p, q, :v] = np.sort(rng.integers(0, 12, v).astype(np.float32) / 8)[::-1]
            I[p, q, :v] = rng.integers(0, 1 << 40, v) * 8 + p
    return D, I


@pytest.mark.parametrize("oi", [0, 1])
def test_merge_topk_alignment(oi):
    P, nq, k = 3, 5, 64
    rng = np.random.default_rng(5)
    Dp, Ip = _sorted_parts(rng, P, nq, k, [k, 40, k])
    bufs = {"Dp": (Dp.size, F32, Dp), "Ip": (Ip.size, I64, Ip), "D": (nq * k, F32, None), "I": (nq * k, I64, None)}

    def call(p, st):
        _capi.check(L().wb_merge_topk_dev(0, nq, k, P, p["Dp"], p["Ip"], p["D"], p["I"], st))

    want = run(call, bufs)
    got = run(call, bufs, {"Dp": 1, "Ip": 1, "D": 3, "I": 1} if oi else {})
    assert_same(got, want, "merge_topk")
    for q in range(nq):  # score descending, then part, then rank in part
        s, part, rank = Dp[:, q].ravel(), np.repeat(np.arange(P), k), np.tile(np.arange(k), P)
        o = np.lexsort((rank, part, -s.astype(np.float64)))[:k]
        assert np.array_equal(want["D"].reshape(nq, k)[q], s[o]) and np.array_equal(want["I"].reshape(nq, k)[q],
                                                                                      Ip[:, q].ravel()[o])


@pytest.mark.parametrize("oi", [0, 1])
def test_range_merge_alignment(oi):
    P, nq = 3, 6
    rng = np.random.default_rng(6)
    cnt = rng.integers(0, 20, (P, nq))
    cnt[1, 2] = cnt[0, 4] = 0
    lp = np.zeros((P, nq + 1), np.int64)
    lp[:, 1:] = np.cumsum(cnt, axis=1)
    stride = int(lp[:, -1].max()) + 5
    Dp = np.full((P, stride), np.nan, np.float32)
    Ip = np.full((P, stride), -7, np.int64)
    for p in range(P):
        for q in range(nq):
            a, b = lp[p, q], lp[p, q + 1]
            Dp[p, a:b] = np.sort(rng.integers(0, 6, b - a).astype(np.float32) / 4)[::-1]
            Ip[p, a:b] = rng.integers(0, 1 << 40, b - a) * 8 + p
    lims = lp.sum(0)
    total = int(lims[-1])
    bufs = {"lp": (lp.size, I64, lp), "Dp": (Dp.size, F32, Dp), "Ip": (Ip.size, I64, Ip),
            "lims": (lims.size, I64, lims), "D": (total, F32, None), "I": (total, I64, None)}

    def call(p, st):
        _capi.check(L().wb_range_merge_dev(0, nq, P, p["lp"], stride, p["Dp"], p["Ip"], p["lims"], p["D"], p["I"],
                                           st))

    want = run(call, bufs)
    got = run(call, bufs, {"lp": 1, "Dp": 1, "Ip": 1, "lims": 1, "D": 3, "I": 1} if oi else {})
    assert_same(got, want, "range_merge")
    for q in range(nq):  # score descending, then part, then order inside the part (a stable sort of the parts in order)
        s = np.concatenate([Dp[p, lp[p, q]:lp[p, q + 1]] for p in range(P)])
        i = np.concatenate([Ip[p, lp[p, q]:lp[p, q + 1]] for p in range(P)])
        o = np.argsort(-s.astype(np.float64), kind="stable")
        assert np.array_equal(want["D"][lims[q]:lims[q + 1]], s[o])
        assert np.array_equal(want["I"][lims[q]:lims[q + 1]], i[o])


@pytest.mark.parametrize("kind,d", [("flat", 128), ("flat", 70), ("ivf", DI)])
def test_add_with_ids_dev_alignment(stores, kind, d):
    """Rows and ids from unaligned device buffers: the stores (rows, ids and IVF lists) equal those of an aligned add."""
    n = 5000
    x = O.unit_gaussian(n, d, 40 + d)
    ids = np.arange(n, dtype=np.int64) * 11 + 4

    def make():
        if kind == "flat":
            return faiss.IndexIDMap(faiss.IndexFlatIP(d))
        idx = faiss.IndexIVFFlat(faiss.IndexFlatIP(d), d, NLIST, faiss.METRIC_INNER_PRODUCT)
        idx.set_centroids(stores["ivf"].cent)
        return idx

    out = []
    for offs in (None, {"x": 1, "ids": 1}):
        idx = make()
        run(lambda p, st: _capi.check(L().wb_add_with_ids_dev(idx._h, n, p["x"], p["ids"], st)),
            {"x": (x.size, F32, x), "ids": (n, I64, ids)}, offs)
        out.append(idx._export(0, n, want_assign=kind == "ivf"))
    for a, b in zip(*out):
        assert (a is None and b is None) or a.tobytes() == b.tobytes()
    assert np.array_equal(out[0][0], x) and np.array_equal(out[0][1], ids)
    if kind == "ivf":
        assert_best_list(x, stores["ivf"].cent, out[0][2], "add-time assignment")


def assert_best_list(x, cent, a, what):
    """Every row's list scores within 1e-5 of its best (3xTF32 may swap two centroids that tie to that bound)."""
    s = x.astype(np.float64) @ cent.astype(np.float64).T
    got = s[np.arange(len(x)), np.asarray(a, np.int64)]
    assert np.all(got >= s.max(1) - 1e-5), f"{what}: {int((got < s.max(1) - 1e-5).sum())} rows in a worse list"


def _kmeans_index(cent):
    idx = faiss.IndexIVFFlat(faiss.IndexFlatIP(cent.shape[1]), cent.shape[1], len(cent), faiss.METRIC_INNER_PRODUCT)
    idx.set_centroids(cent)
    return idx


def _kmeans_data(n=20_000, d=DI, nlist=NLIST):
    x = O.clustered_unit(n, d, 128, 50)
    cent = O.unit_gaussian(nlist, d, 51)
    cent[nlist - 4:] *= np.float32(1e-3)  # four lists that attract no point: the update splits them
    return x, cent


def _centroids(idx):
    return idx.centroids()


@pytest.mark.parametrize("oi", [0, 1])
def test_kmeans_alignment(oi):
    """assign (3xTF32 and plain TF32, n >= 1024: the assignment GEMM maps x with TMA) -> accumulate -> update, every
    buffer carved at offset 0 or 1.  Assignments, objective, sums, counts and the updated centroids are bit-equal to
    the aligned run; the sums are within fp32 rounding of an fp64 recomputation."""
    x, cent = _kmeans_data()
    n, d, nlist = x.shape[0], x.shape[1], len(cent)
    off = 1 if oi else 0
    res = []
    for offs in (None, dict(x=off, a=off, sums=off, counts=off)):
        idx = _kmeans_index(cent)
        out, objs = {}, {}
        for fn in ("wb_kmeans_assign_dev", "wb_kmeans_assign_fast_dev"):
            obj = C.c_double(0)
            a = run(lambda p, st: _capi.check(getattr(L(), fn)(idx._h, n, p["x"], p["a"], C.byref(obj), st)),
                    {"x": (x.size, F32, x), "a": (n, I32, None)}, offs)["a"]
            out[fn], objs[fn] = a, obj.value
        assign = out["wb_kmeans_assign_dev"]
        acc = run(lambda p, st: _capi.check(L().wb_kmeans_accumulate_dev(idx._h, n, p["x"], p["a"], p["sums"],
                                                                         p["counts"], st)),
                  {"x": (x.size, F32, x), "a": (n, I32, assign), "sums": (nlist * d, F32, None),
                   "counts": (nlist, I64, None)}, offs)
        out.update(acc)
        nsplit = C.c_int64(-1)
        run(lambda p, st: _capi.check(L().wb_kmeans_update_dev(idx._h, p["sums"], p["counts"], n, 1234,
                                                               C.byref(nsplit), st)),
            {"sums": (nlist * d, F32, acc["sums"]), "counts": (nlist, I64, acc["counts"])}, offs)
        out["nsplit"] = np.int64(nsplit.value)
        out["cent"] = _centroids(idx)
        res.append(({k: np.asarray(v) for k, v in out.items()}, objs))
    (want, wobj), (got, gobj) = res
    assert_same(got, want, f"k-means at offset {off}")
    # the objective's per-block partial sums are added with a double atomicAdd: equal up to their order
    for fn, v in wobj.items():
        assert abs(gobj[fn] - v) <= 1e-9 * abs(v), (fn, gobj[fn], v)
    assert want["nsplit"] >= 4
    a = want["wb_kmeans_assign_dev"].astype(np.int64)
    assert_best_list(x, cent, a, "k-means assignment")
    best = (x.astype(np.float64) * cent[a].astype(np.float64)).sum(1).sum()
    assert abs(wobj["wb_kmeans_assign_dev"] - best) <= 1e-5 * abs(best)
    ref = np.zeros((nlist, d), np.float64)
    np.add.at(ref, a, x.astype(np.float64))
    absum = np.zeros((nlist, d), np.float64)
    np.add.at(absum, a, np.abs(x.astype(np.float64)))
    cnt = np.bincount(a, minlength=nlist)
    assert np.array_equal(want["counts"], cnt)
    err = np.abs(want["sums"].reshape(nlist, d).astype(np.float64) - ref)
    assert np.all(err <= 2.0 ** -24 * cnt[:, None] * absum), float(err.max())


# ---- 2. edges of the write loops ------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["flat", "ivf-nprobe1", "compact-filter"])
def test_k_beyond_the_candidates_pads_every_slot(stores, case):
    """k above the number of candidates: 700 rows with k = 1000; one probed list (~625 rows) with k = 2048; a filter
    that keeps 300 rows (its compact copy) with k = 1000 on 16 queries.  The slots past the candidates must be written
    as (-FLT_MAX, -1).  (The tensor-core path never takes k > ntotal: it needs 8k rows or more.)"""
    nprobe, flt, sel = 1, None, None
    if case == "flat":
        st, nq, k = _flat(700, 70, 60, 16), 4, 1000
    elif case == "ivf-nprobe1":
        st, nq, k = stores["ivf"], 4, 2048
    else:
        st, nq, k = stores["flat768"], 16, 1000
        sel = faiss.IDSelectorBatch(st.ids[::200])
        flt = sel._filter(st.idx._hd)
    xq = st.xq[:nq]
    want = search(st.idx, xq, k, nprobe=nprobe, flt=flt)
    got = search(st.idx, xq, k, ONE[1], nprobe=nprobe, flt=flt)
    assert_same(got, want, f"k > candidates {case}")
    assert (want["I"] == -1).any()
    if sel is None:
        Dr, Ir = st.oracle(xq, k, nprobe)
    else:
        keep = np.isin(st.ids, sel.ids)
        Dr, Ir = O.flat_search(st.xb[keep], xq, k, st.ids[keep])
    O.compare_topk(want["D"], want["I"], Dr, Ir, band=4e-6)


@pytest.fixture(scope="module")
def k2_kmax_store():
    """270000 x 32: enough rows for the tensor-core path to take k = 2048 (its candidate list holds 2k rows)."""
    return _flat(270_000, 32, 70, 16)


@pytest.mark.parametrize("name,nq,sw", [("flat768", 4, {}), ("k2", 16, {"WB_GEMM_FORCE": 1}), ("ivf", 4, {})],
                         ids=["k1", "k2", "ivf"])
def test_k_max(stores, k2_kmax_store, name, nq, sw):
    st = k2_kmax_store if name == "k2" else stores[name]
    k, xq = 2048, st.xq[:nq]
    with env(**sw):
        want = search(st.idx, xq, k, nprobe=st.nprobe)
        e0 = gemm_epochs(st.idx)
        got = search(st.idx, xq, k, FULL[3], nprobe=st.nprobe)
        assert (gemm_epochs(st.idx) > e0) == (name == "k2")
    assert_same(got, want, f"k=2048 {name} nq={nq}")
    O.compare_topk(want["D"], want["I"], *st.oracle(xq, k), band=4e-6)


def test_nq_past_the_k2_query_chunk(stores):
    """65536 + 129 queries: the second K2 call writes its results at an offset of 65536 rows into the caller's D / I."""
    st = stores["flat70"]
    k, xq = 10, st.xq
    assert len(xq) == K2_MAX_Q + 129
    with env(WB_GEMM_FORCE=1):
        want = search(st.idx, xq, k)
        e0 = gemm_epochs(st.idx)
        got = search(st.idx, xq, k, ONE[1])
        assert gemm_epochs(st.idx) > e0
    assert_same(got, want, "nq past the K2 chunk")
    rows = np.array([0, 1, K2_MAX_Q - 1, K2_MAX_Q, K2_MAX_Q + 1, len(xq) - 1])
    O.compare_topk(want["D"][rows], want["I"][rows], *st.oracle(xq[rows], k), band=4e-6)


@pytest.mark.parametrize("name,nq,bad,sw", [("flat768", 4, 2, {}), ("flat768", 16, 5, {"WB_GEMM_FORCE": 1}),
                                            ("ivf", 4, 1, {})], ids=["k1", "k2", "ivf-fused"])
def test_nan_query_row_is_all_padding(stores, name, nq, bad, sw):
    st = stores[name]
    k = 100
    xq = st.xq[:nq].copy()
    xq[bad, 3] = np.nan
    with env(**sw):
        want = search(st.idx, xq, k, nprobe=st.nprobe)
        got = search(st.idx, xq, k, ONE[1], nprobe=st.nprobe)
    assert_same(got, want, f"NaN query {name} nq={nq}")
    assert np.all(want["I"][bad] == -1) and np.all(want["D"][bad] == NEG_FLT_MAX)
    ok = np.arange(nq) != bad
    O.compare_topk(want["D"][ok], want["I"][ok], *st.oracle(xq[ok], k), band=4e-6)


def test_range_zero_and_one_hit(stores):
    """A threshold above every score (no hit: the copy writes nothing, the guards hold) and a stored row as the query
    with a threshold between its own score (~1) and the next (~0.2): exactly one hit."""
    st = stores["flat768"]
    for xq, t, total in ((st.xq[:4], 10.0, 0), (st.xb[[7]], 0.5, 1)):
        want = range_dev(st.idx, xq, t)
        got = range_dev(st.idx, xq, t, {"q": 1, "D": 3, "I": 1})
        assert int(want["lims"][-1]) == total
        assert_same(got, want, f"range with {total} hits")
    assert want["I"][0] == st.ids[7]


def host_carved(n, dtype, offset, data=None):
    """carved() in host memory: (interior array, check)."""
    nd = np.dtype(dtype)
    ity = np.int32 if nd.itemsize == 4 else np.int64
    s = {np.float32: 0x7FBADBAD, np.int32: 0x5A5A5A5A, np.int64: 0x5A5A5A5A5A5A5A5A}[nd.type]
    base = np.full(G + offset + n + G, s, ity)
    lo, hi = G + offset, G + offset + n
    view = base.view(nd)[lo:hi]
    if data is not None:
        view[:] = np.asarray(data).reshape(-1)
    want = base[lo:hi].copy() if data is not None else None

    def check(what):
        assert np.all(base[:lo] == s) and np.all(base[hi:] == s), f"{what}: a guard was overwritten"
        if want is None:
            assert not np.any(base[lo:hi] == s), f"{what}: an output slot was never written"
        else:
            assert np.array_equal(base[lo:hi], want), f"{what}: the call modified an input buffer"

    return view, check


@pytest.mark.parametrize("name,nq", [("flat768", 4), ("flat768", 300), ("ivf", 4), ("ivf", 64)])
def test_host_entry_guards(stores, name, nq):
    """wb_search and wb_range_result_copy into the interior of larger host arrays."""
    st = stores[name]
    k, xq = 100, st.xq[:nq]
    D0, I0 = np.empty(nq * k, np.float32), np.empty(nq * k, np.int64)
    _capi.check(L().wb_search(st.idx._h, nq, _capi.ptr(xq), k, st.nprobe, _capi.ptr(D0), _capi.ptr(I0)))
    q, cq = host_carved(xq.size, np.float32, 1, xq)
    D, cD = host_carved(nq * k, np.float32, 3, None)
    I, cI = host_carved(nq * k, np.int64, 1, None)
    _capi.check(L().wb_search(st.idx._h, nq, q.ctypes.data, k, st.nprobe, D.ctypes.data, I.ctypes.data))
    for c, w in ((cq, "q"), (cD, "D"), (cI, "I")):
        c(f"wb_search {w}")
    assert D.tobytes() == D0.tobytes() and I.tobytes() == I0.tobytes()
    t = np.float32(_thresh(st, xq, 200))
    lims, Dr, Ir = st.idx.range_search(xq, t)
    res = C.c_void_p()
    lims2 = np.zeros(nq + 1, np.int64)
    _capi.check(L().wb_range_search(st.idx._h, None, nq, _capi.ptr(xq), float(t), st.nprobe,
                                    _capi.ptr(lims2), C.byref(res)))
    try:
        n = int(lims2[-1])
        D, cD = host_carved(n, np.float32, 1, None)
        I, cI = host_carved(n, np.int64, 1, None)
        _capi.check(L().wb_range_result_copy(res, D.ctypes.data, I.ctypes.data))
    finally:
        _capi.check(L().wb_range_result_free(res))
    cD("wb_range_result_copy D")
    cI("wb_range_result_copy I")
    assert np.array_equal(lims2, lims.astype(np.int64)) and D.tobytes() == Dr.tobytes() and I.tobytes() == Ir.tobytes()


# ---- 3. a busy caller stream ----------------------------------------------------------------------------------------
def on_busy_stream(call, inputs, outputs, pending=False):
    """On a side stream s: a long sleep, then copies of the new inputs into buffers that hold OTHER valid inputs, then
    call(ptrs, s), then clones of the outputs, all on s.  inputs: name -> (new, other) numpy arrays (same shape);
    outputs: name -> (n, dtype).  pending: assert that s is still busy right after call returns (the call did not
    synchronise it).  Returns the clones as numpy arrays after s.synchronize()."""
    s = torch.cuda.Stream()
    bufs = {k: torch.from_numpy(np.ascontiguousarray(o).reshape(-1)).cuda() for k, (_, o) in inputs.items()}
    news = {k: torch.from_numpy(np.ascontiguousarray(v).reshape(-1)).cuda() for k, (v, _) in inputs.items()}
    outs = {k: torch.zeros(n, dtype=dt, device="cuda") for k, (n, dt) in outputs.items()}
    torch.cuda.synchronize()
    ptrs = {k: v.data_ptr() for k, v in {**bufs, **outs}.items()}
    with torch.cuda.stream(s):
        torch.cuda._sleep(SLEEP_CYCLES)
        for k in bufs:
            bufs[k].copy_(news[k])
        call(ptrs, s.cuda_stream)
        busy = not s.query()
        clones = {k: v.clone() for k, v in outs.items()}
    s.synchronize()
    if pending:
        assert busy, "the call synchronised the caller's stream"
    return {k: v.cpu().numpy() for k, v in clones.items()}


BUSY_SEARCH = {"k1": ("flat768", 4, 100, {}, True), "ivf-fused": ("ivf", 4, 10, {}, True),
               "k2": ("flat768", 16, 100, {"WB_GEMM_FORCE": 1}, False),
               "listmajor": ("ivf", 64, 100, {"WB_IVF_LISTMAJOR": 1}, False)}


@pytest.mark.parametrize("path", list(BUSY_SEARCH))
def test_search_on_a_busy_stream(stores, path):
    name, nq, k, sw, pending = BUSY_SEARCH[path]
    st = stores[name]
    xq, other = st.xq[:nq], O.unit_gaussian(nq, st.xq.shape[1], 77)
    with env(**sw):
        want = search(st.idx, xq, k, nprobe=st.nprobe)  # also the warm-up of this shape
        f0 = fused(st.idx)
        got = on_busy_stream(search_call(st.idx, nq, k, st.nprobe), {"q": (xq, other)},
                             {"D": (nq * k, F32), "I": (nq * k, I64)}, pending)
        if path == "ivf-fused":
            assert fused(st.idx) == f0 + 1
    assert_same({k_: v.reshape(nq, k) for k_, v in got.items()}, want, f"busy stream {path}")


def test_merge_topk_on_a_busy_stream():
    P, nq, k = 4, 8, 100
    rng = np.random.default_rng(8)
    Dp, Ip = _sorted_parts(rng, P, nq, k, [k] * P)
    Do, Io = _sorted_parts(rng, P, nq, k, [k] * P)
    bufs = {"Dp": (Dp.size, F32, Dp), "Ip": (Ip.size, I64, Ip), "D": (nq * k, F32, None), "I": (nq * k, I64, None)}

    def call(p, st):
        _capi.check(L().wb_merge_topk_dev(0, nq, k, P, p["Dp"], p["Ip"], p["D"], p["I"], st))

    want = run(call, bufs)
    got = on_busy_stream(call, {"Dp": (Dp, Do), "Ip": (Ip, Io)}, {"D": (nq * k, F32), "I": (nq * k, I64)}, True)
    assert_same(got, want, "merge_topk on a busy stream")


def _flat_twin(x, ids, reserve=0):
    idx = faiss.IndexIDMap(faiss.IndexFlatIP(x.shape[1]))
    if reserve:
        idx.reserve(reserve)
    idx.add_with_ids(x, ids)
    return idx


@pytest.mark.parametrize("grow", [False, True], ids=["stale-filter", "growing-store"])
def test_add_then_search_on_a_busy_stream(grow):
    """wb_add_with_ids_dev on the busy stream, then at once a search on it.  stale-filter: a reserved store, a filter
    evaluated before the add; the search re-evaluates it after the add's ids have landed.  growing-store: 1000 rows
    (capacity 1024), the add of 3000 more grows the store.  The added rows include copies of the queries, so a search
    that misses them fails."""
    d, n0, n1, nq, k = 128, 20_000 if not grow else 1000, 3000, 4, 100
    x = O.unit_gaussian(n0 + n1, d, 90)
    xq = O.unit_gaussian(nq, d, 91)
    x[n0 + 17:n0 + 17 + nq] = xq
    ids = np.arange(n0 + n1, dtype=np.int64) * 3 + 1
    sel = faiss.IDSelectorRange(0, int(ids[n0 + n1 // 2]))  # keeps the first half of the new rows
    twin = _flat_twin(x, ids)
    want = search(twin, xq, k, flt=None if grow else sel._filter(twin._hd))
    idx = _flat_twin(x[:n0], ids[:n0], 0 if grow else n0 + n1)
    flt = None if grow else sel._filter(idx._hd)
    search(idx, xq, k, flt=flt)  # warm: the filter is evaluated over the first n0 rows
    other = O.unit_gaussian(n1, d, 92)

    def call(p, st):
        _capi.check(L().wb_add_with_ids_dev(idx._h, n1, p["x"], p["ids"], st))
        search_call(idx, nq, k, 1, flt)(p, st)

    got = on_busy_stream(call, {"x": (x[n0:], other), "ids": (ids[n0:], ids[n0:] + 1), "q": (xq, xq[::-1])},
                         {"D": (nq * k, F32), "I": (nq * k, I64)})
    assert idx.ntotal == n0 + n1
    assert_same({k_: v.reshape(nq, k) for k_, v in got.items()}, want, f"add then search, grow={grow}")
    assert np.all(want["I"][:, 0] == ids[n0 + 17:n0 + 17 + nq])
    keep = np.ones(len(ids), bool) if grow else ids < sel.imax
    O.compare_topk(want["D"], want["I"], *O.flat_search(x[keep], xq, k, ids[keep]), band=4e-6)


def test_range_search_on_a_busy_stream(stores):
    st = stores["flat768"]
    xq, other = st.xq[:4], O.unit_gaussian(4, 768, 93)
    t = _thresh(st, xq, 300)
    want = range_dev(st.idx, xq, t)
    n = int(want["lims"][-1])
    box = {}

    def call(p, st_):
        lims = np.zeros(5, np.int64)
        res = C.c_void_p()
        _capi.check(L().wb_range_search_dev(st.idx._h, None, 4, p["q"], float(t), 1, _capi.ptr(lims), C.byref(res),
                                            st_))
        box["lims"] = lims
        try:
            assert int(lims[-1]) == n, (int(lims[-1]), n)
            _capi.check(L().wb_range_result_copy_dev(res, p["D"], p["I"], st_))
        finally:
            _capi.check(L().wb_range_result_free(res))

    got = on_busy_stream(call, {"q": (xq, other)}, {"D": (n, F32), "I": (n, I64)})
    got["lims"] = box["lims"]
    assert_same(got, want, "range search on a busy stream")


def test_kmeans_chain_on_a_busy_stream():
    """assign (no objective: no synchronisation) -> accumulate -> update, all on the busy stream."""
    x, cent = _kmeans_data()
    n, d, nlist = x.shape[0], x.shape[1], len(cent)
    other = O.unit_gaussian(n, d, 94)

    def chain(idx):
        def call(p, st):
            _capi.check(L().wb_kmeans_assign_fast_dev(idx._h, n, p["x"], p["a"], None, st))
            _capi.check(L().wb_kmeans_accumulate_dev(idx._h, n, p["x"], p["a"], p["sums"], p["counts"], st))
            _capi.check(L().wb_kmeans_update_dev(idx._h, p["sums"], p["counts"], n, 1234, None, st))
        return call

    ref = _kmeans_index(cent)
    want = run(chain(ref), {"x": (x.size, F32, x), "a": (n, I32, None), "sums": (nlist * d, F32, None),
                            "counts": (nlist, I64, None)})
    want["cent"] = _centroids(ref)
    idx = _kmeans_index(cent)
    got = on_busy_stream(chain(idx), {"x": (x, other)},
                         {"a": (n, I32), "sums": (nlist * d, F32), "counts": (nlist, I64)})
    got["cent"] = _centroids(idx)
    assert_same(got, want, "k-means chain on a busy stream")
    assert not np.array_equal(want["cent"], cent)


# ---- 4. two handles from two threads --------------------------------------------------------------------------------
def test_two_handles_from_two_threads(stores):
    """Thread A searches flat768 (K1 at nq 1-16, K2 at nq 300) and range-searches it; thread B searches flat70 and the
    IVF index (fused at nq 1 / 4, list-major at nq 64), each through the host API on its own handles.  Every result is
    byte-identical to the same call made alone.  Fresh threads every round: the kernels' shared-memory opt-in is per
    host thread, so each round also makes first calls on new threads."""
    fa, fb, iv = stores["flat768"], stores["flat70"], stores["ivf"]
    t = _thresh(fa, fa.xq[:4], 300)
    jobs_a, jobs_b = [], []
    for r in range(5):
        for nq in (1, 4, 16, 300):
            jobs_a.append(("search", fa, nq, 100 if r % 2 else 10))
        if r < 3:
            jobs_a.append(("range", fa, 4, t))
    for r in range(4):
        for nq in (1, 4, 300):
            jobs_b.append(("search", fb, nq, 50))
        for nq, k in ((1, 10), (4, 10), (64, 100)):
            jobs_b.append(("search", iv, nq, k))

    def do(job):
        kind, st, nq, arg = job
        if kind == "search":
            D, I = st.idx.search(st.xq[:nq], arg)
            return D.tobytes() + I.tobytes()
        lims, D, I = st.idx.range_search(st.xq[:nq], arg)
        return lims.tobytes() + D.tobytes() + I.tobytes()

    want = {"a": [do(j) for j in jobs_a], "b": [do(j) for j in jobs_b]}
    e0, f0 = gemm_epochs(fa.idx), fused(iv.idx)
    for rnd in range(3):
        got, errors = {}, []

        def worker(name, jobs):
            try:
                got[name] = [do(j) for j in jobs]
            except Exception as e:  # reported below, in the test's thread
                errors.append((name, repr(e)))

        ths = [threading.Thread(target=worker, args=("a", jobs_a)), threading.Thread(target=worker, args=("b", jobs_b))]
        for th in ths:
            th.start()
        for th in ths:
            th.join(timeout=300)
        assert not any(th.is_alive() for th in ths), f"round {rnd}: a search thread did not finish"
        assert not errors, errors
        for name, jobs in (("a", jobs_a), ("b", jobs_b)):
            for j, (g, w) in enumerate(zip(got[name], want[name])):
                assert g == w, f"round {rnd} thread {name} job {j} ({jobs[j][0]} nq={jobs[j][2]}) differs"
    assert gemm_epochs(fa.idx) > e0 and fused(iv.idx) > f0
