#!/usr/bin/env python
"""Filtered search on one B200: cost of faiss SearchParameters(sel=IDSelector...) against the unfiltered search, and
the data behind the flat sparse/mask cutoff (kSparseCutoffDen in wise_b200/csrc/capi.cu, DESIGN.md "Filtered search").

    python scripts/bench_filtered.py [--rows 10000000] [--dim 768] [--out profiles/filtered/bench_filtered.jsonl]

Flat: bench.py's clustered 10M x 768 store (ids = positions), k = 100, batches 1 / 16 / 1024, random IDSelectorBatch
selectors keeping 1, 1/2, 1/8, 1/64, 1e-3 and 1e-5 of the rows plus one IDSelectorRange.  Per case: the filter build
(wb_filter_create_ids, host wall clock), the first search (which also gathers the compact copy on the sparse path),
the steady search (CUDA events around back-to-back wb_search_filtered_dev calls) and the unfiltered search of the same
queries in the same run.  Every timed result is verified with bench.parity_check restricted to the selected rows.
IVF: 2M x 512, nlist 1024, nprobe 8, batches 1 and 256, selected fractions 1 / 0.1 / 0.01, verified against an fp64
pass over the selected rows of the probed lists.
The store (>= 4 GB) is far larger than the 126 MB L2, so no flush is needed between steps.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import bench  # noqa: E402  (generators and parity_check)

FRACTIONS = [1.0, 1 / 2, 1 / 8, 1 / 64, 1e-3, 1e-5]


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return {"nvidia_smi": out.stdout.strip().splitlines()[0] if out.returncode == 0 else f"unavailable: {out.stderr.strip()}"}


def timed(call, steps, warmup):
    import torch
    for _ in range(warmup):
        call()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        call()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def make_filter(L, h, sel_ids=None, rng=None):
    """(wb_filter*, build ms): an id set, or the range rng = (imin, imax)."""
    from wise_b200 import _capi
    f = C.c_void_p()
    t0 = time.perf_counter()
    if rng is None:
        _capi.check(L.wb_filter_create_ids(h, sel_ids.size, _capi.ptr(sel_ids), 0, C.byref(f)))
    else:
        _capi.check(L.wb_filter_create_range(h, rng[0], rng[1], 0, C.byref(f)))
    return f, (time.perf_counter() - t0) * 1e3


def flat_part(a, device, emit):
    import torch
    from wise_b200 import _capi, faiss_compat as faiss
    L = _capi.lib()
    n, d, k = a.rows, a.dim, 100
    src = bench.RowSource(n, d, 2024, device)
    index = faiss.IndexIDMap(faiss.IndexFlatIP(d, device=0))
    bench.fill_index(index, src, 0, n)  # ids = insertion positions
    h = index._h
    st = torch.cuda.current_stream().cuda_stream
    rng = np.random.default_rng(7)
    cases = [(f"batch {fr:g}", np.sort(rng.choice(n, max(1, int(round(fr * n))), replace=False)).astype(np.int64), None)
             for fr in FRACTIONS]
    cases.append(("range 1/64", None, (n // 3, n // 3 + n // 64)))
    for nq in (1, 16, 1024):
        q = bench.make_queries(src.centres, nq, d, 3000 + nq, device)
        Dt = torch.empty((nq, k), device=device)
        It = torch.empty((nq, k), dtype=torch.int64, device=device)
        steps = {1: 50, 16: 20, 1024: 5}[nq]

        def search(f):
            return lambda: _capi.check(L.wb_search_filtered_dev(h, f, nq, q.data_ptr(), k, 1, Dt.data_ptr(), It.data_ptr(), st))

        base_ms = timed(search(None), steps, 3)
        for name, ids, r in cases:
            f, build_ms = make_filter(L, h, ids, r)
            try:
                count = int(L.wb_filter_count(f))
                e0, f0 = C.c_int64(0), C.c_int64(0)
                _capi.check(L.wb_gemm_stats(h, C.byref(e0), C.byref(f0)))
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                search(f)()
                torch.cuda.synchronize()
                first_ms = (time.perf_counter() - t0) * 1e3
                ms = timed(search(f), steps, 2)
                e1, f1 = C.c_int64(0), C.c_int64(0)
                _capi.check(L.wb_gemm_stats(h, C.byref(e1), C.byref(f1)))
                sel = torch.zeros(n, dtype=torch.bool, device=device)
                if ids is not None:
                    sel[torch.from_numpy(ids).to(device)] = True
                else:
                    sel[r[0]:r[1]] = True
                allowed = lambda s, e: (sel[s:e].unsqueeze(1).expand(e - s, nq),) * 2
                par = bench.parity_check(src, 0, n, q, Dt, It, k, 1, device, allowed=allowed)
            finally:
                _capi.check(L.wb_filter_free(f))
            emit({"part": "flat", "rows": n, "dim": d, "k": k, "batch": nq, "selector": name, "selected": count,
                  "fraction": count / n, "path": "compact" if count * 8 < n else "mask",
                  "filter_build_ms": round(build_ms, 3), "first_search_ms": round(first_ms, 3),
                  "compact_copy_ms_est": round(max(0.0, first_ms - ms), 3) if count * 8 < n else 0.0,
                  "search_ms": round(ms, 4), "unfiltered_ms": round(base_ms, 4),
                  "k2_fallbacks": f1.value - f0.value, "parity": par})
    del index
    torch.cuda.empty_cache()


def ivf_part(device, emit):
    import torch
    from wise_b200 import _capi, faiss_compat as faiss
    L = _capi.lib()
    n, d, nlist, k, nprobe, seed = 2_000_000, 512, 1024, 100, 8, 50
    gen = torch.Generator(device=device)
    gen.manual_seed(seed)
    centres = torch.nn.functional.normalize(torch.randn(bench.NCENTRES, d, device=device, generator=gen), dim=1)
    ivf = faiss.IndexIVFFlat(faiss.IndexFlatIP(d), d, nlist, faiss.METRIC_INNER_PRODUCT)
    ivf.set_centroids(bench.make_queries(centres, nlist, d, 11, device).cpu().numpy())
    bench.fill_index_clustered(ivf, 0, n, d, seed, device)
    _capi.check(L.wb_ivf_finalize(ivf._h))
    # storage-order rows, ids and lists for the check (ids = insertion positions)
    x, ids, assign = ivf._export(0, n, want_assign=True)
    X = torch.from_numpy(x).to(device)
    ids_t = torch.from_numpy(ids).to(device)
    lists_t = torch.from_numpy(assign.astype(np.int64)).to(device)
    cent = torch.from_numpy(ivf.centroids()).to(device).double()
    inv = torch.empty(n, dtype=torch.int64, device=device)
    inv[ids_t] = torch.arange(n, device=device)  # id (= insertion position) -> storage row
    del x
    st = torch.cuda.current_stream().cuda_stream
    rng = np.random.default_rng(9)
    for nq in (1, 256):
        q = bench.make_queries(centres, nq, d, 4000 + nq, device)
        Dt = torch.empty((nq, k), device=device)
        It = torch.empty((nq, k), dtype=torch.int64, device=device)
        steps = {1: 200, 256: 20}[nq]

        def search(f):
            return lambda: _capi.check(L.wb_search_filtered_dev(ivf._h, f, nq, q.data_ptr(), k, nprobe, Dt.data_ptr(),
                                                                It.data_ptr(), st))

        base_ms = timed(search(None), steps, 5)
        probes = (q.double() @ cent.T).topk(nprobe, dim=1).indices  # [nq, nprobe]
        for fr in (1.0, 0.1, 0.01):
            sel_ids = np.sort(rng.choice(n, int(round(fr * n)), replace=False)).astype(np.int64)
            f, build_ms = make_filter(L, ivf._h, sel_ids)
            try:
                ms = timed(search(f), steps, 5)
            finally:
                _capi.check(L.wb_filter_free(f))
            # verification: fp64 scores of the selected rows of the probed lists
            sel = torch.zeros(n, dtype=torch.bool, device=device)
            sel[torch.from_numpy(sel_ids).to(device)] = True
            selected = sel[ids_t]  # storage row -> selected?
            viol, max_err = 0, 0.0
            for j in range(nq):
                cand = selected & torch.isin(lists_t, probes[j])
                s64 = X[cand].double() @ q[j].double()
                kk = min(k, int(cand.sum()))
                viol += int((It[j, kk:] != -1).sum())  # padding only where fewer than k candidates exist
                if kk == 0:
                    continue
                rows = inv[It[j, :kk]]  # storage rows of the returned ids
                viol += int((~cand[rows]).sum())  # every returned row is a candidate
                ex = X[rows].double() @ q[j].double()
                max_err = max(max_err, float((ex - Dt[j, :kk].double()).abs().max()))
                kth = float(Dt[j, kk - 1])  # no candidate beats the k-th returned score by more than the tie band
                viol += max(0, int((s64 > kth + bench.TIE_BAND).sum()) - int((ex > kth + bench.TIE_BAND).sum()))
            emit({"part": "ivf", "rows": n, "dim": d, "nlist": nlist, "nprobe": nprobe, "k": k, "batch": nq,
                  "selector": f"batch {fr:g}", "fraction": fr, "filter_build_ms": round(build_ms, 3),
                  "search_ms": round(ms, 4), "unfiltered_ms": round(base_ms, 4),
                  "check": {"violations": viol, "max_abs_err": max_err, "ok": viol == 0 and max_err <= bench.SCORE_TOL}})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    ap.add_argument("--skip-ivf", action="store_true")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_filtered.py needs a B200: wise_b200 has no CPU fallback")
    device = torch.device("cuda", 0)
    torch.cuda.set_device(device)
    out = open(a.out, "a") if a.out else None

    def emit(rec):
        line = json.dumps(rec)
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()

    emit({"part": "gpu", **gpu_info()})
    flat_part(a, device, emit)
    if not a.skip_ivf:
        ivf_part(device, emit)


if __name__ == "__main__":
    main()
