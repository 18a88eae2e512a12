#!/usr/bin/env python
"""Range search on one B200 (faiss Index::range_search, DESIGN.md "Range search"): cost against the k = 100 search of
the same queries, in the same run.

    python scripts/bench_range.py [--rows 10000000] [--dim 768] [--out profiles/range/bench_range.jsonl]

Flat: bench.py's clustered 10M x 768 store (ids = positions), batches 1 / 16 / 1024, one threshold per batch chosen
from fp64 scores against the first 500k rows so that a query has about 10, 10^3 and 10^5 hits on average.  IVF:
2M x 512, nlist 1024, nprobe 8, batches 1 and 256, thresholds for about 10 and 10^3 hits.  Per case: host wall time of
wb_range_search plus the copy-out (wb_range_result_copy), the device time of its last scan pass (CUDA events around
the scan, wb_last_scan_ms), the same two numbers for wb_search with k = 100, and hits per query.  Every timed result
is verified in-run against an fp64 pass over the regenerated rows: each returned score within 1e-5 of fp64 and above
the threshold, every row with fp64 score above threshold + 4e-6 returned, none below threshold - 4e-6.
The stores (30 GB, 4 GB) are far larger than the 126 MB L2.
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

import bench  # noqa: E402

BAND = 4e-6


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return out.stdout.strip().splitlines()[0] if out.returncode == 0 else f"unavailable: {out.stderr.strip()}"


def run_range(L, h, q_host, thresh, nprobe):
    from wise_b200 import _capi
    nq = q_host.shape[0]
    lims = np.zeros(nq + 1, np.int64)
    res = C.c_void_p()
    t0 = time.perf_counter()
    _capi.check(L.wb_range_search(h, None, nq, _capi.ptr(q_host), float(thresh), nprobe, _capi.ptr(lims), C.byref(res)))
    t1 = time.perf_counter()
    D = np.empty(int(lims[-1]), np.float32)
    I = np.empty(int(lims[-1]), np.int64)
    _capi.check(L.wb_range_result_copy(res, _capi.ptr(D), _capi.ptr(I)))
    t2 = time.perf_counter()
    _capi.check(L.wb_range_result_free(res))
    return lims, D, I, (t1 - t0) * 1e3, (t2 - t0) * 1e3, float(L.wb_last_scan_ms(h))


def run_search(L, h, q_host, k, nprobe):
    from wise_b200 import _capi
    nq = q_host.shape[0]
    D = np.empty((nq, k), np.float32)
    I = np.empty((nq, k), np.int64)
    t0 = time.perf_counter()
    _capi.check(L.wb_search(h, nq, _capi.ptr(q_host), k, nprobe, _capi.ptr(D), _capi.ptr(I)))
    return (time.perf_counter() - t0) * 1e3, float(L.wb_last_scan_ms(h))


def best_of(fn, reps):
    out = [fn() for _ in range(reps)]
    return out[int(np.argmin([o[-2] if len(o) > 3 else o[0] for o in out]))], out


def verify(chunks, q, lims, D, I, thresh, cand=None):
    """chunks: iterable of (s, e, x[e-s, d] device); cand(s, e) -> bool [e-s, nq] candidate mask (None: all)."""
    import torch
    dev = q.device
    nq = q.shape[0]
    q64 = q.double()
    cnt = torch.from_numpy(np.diff(lims)).to(dev)
    qi = torch.repeat_interleave(torch.arange(nq, device=dev), cnt)
    It = torch.from_numpy(I).to(dev)
    Dt = torch.from_numpy(D).to(dev).double()
    strict = torch.zeros(nq, dtype=torch.int64, device=dev)
    got_strict = torch.zeros(nq, dtype=torch.int64, device=dev)
    max_err, below = 0.0, 0
    for s, e, x in chunks:
        S = x.double() @ q64.T  # [e-s, nq]
        if cand is not None:
            S = torch.where(cand(s, e), S, torch.full_like(S, -np.inf))
        strict += (S > thresh + BAND).sum(0)
        m = (It >= s) & (It < e)
        v = S[It[m] - s, qi[m]]
        max_err = max(max_err, float((v - Dt[m]).abs().max()) if m.any() else 0.0)
        below += int((v <= thresh - BAND).sum())
        got_strict += torch.bincount(qi[m][v > thresh + BAND], minlength=nq)
    ok = (max_err <= 1e-5 and below == 0 and bool((strict == got_strict).all()) and bool((Dt > np.float32(thresh)).all())
          and all(np.all(np.diff(D[lims[i]:lims[i + 1]]) <= 0) for i in range(nq)))
    return {"ok": ok, "max_abs_err": max_err, "returned_below_band": below,
            "missing_above_band": int((strict - got_strict).sum())}


def thresholds(sample, q, hits, n):
    S = (sample.double() @ q.double().T).flatten()
    return {h: float(torch_quantile(S, 1 - h / n)) for h in hits}


def torch_quantile(S, p):
    import torch
    k = max(1, int(round((1 - p) * S.numel())))
    return torch.topk(S, k).values[-1].item()


def flat_part(a, device, emit):
    import torch
    from wise_b200 import _capi, faiss_compat as faiss
    L = _capi.lib()
    n, d = a.rows, a.dim
    src = bench.RowSource(n, d, 2024, device)
    index = faiss.IndexIDMap(faiss.IndexFlatIP(d, device=0))
    bench.fill_index(index, src, 0, n)
    h = index._h
    _capi.check(L.wb_set_timing(h, 1))
    sample = next(iter(src.chunks(0, min(n, 500_000))))[2]
    for nq in (1, 16, 1024):
        q = bench.make_queries(src.centres, nq, d, 3000 + nq, device)
        qh = q.cpu().numpy()
        reps = {1: 5, 16: 3, 1024: 2}[nq]
        run_search(L, h, qh, 100, 1)
        s_best, _ = best_of(lambda: run_search(L, h, qh, 100, 1), reps)
        for hits, t in thresholds(sample, q, (10, 1000, 100_000), n).items():
            run_range(L, h, qh, t, 1)  # warm-up (pool growth)
            r, _ = best_of(lambda: run_range(L, h, qh, t, 1), reps)
            lims, D, I, call_ms, wall_ms, scan_ms = r
            par = verify(src.chunks(0, n), q, lims, D, I, t)
            emit({"part": "flat", "rows": n, "dim": d, "batch": nq, "target_hits": hits, "thresh": t,
                  "hits_per_query": float(lims[-1]) / nq, "max_hits": int(np.diff(lims).max()),
                  "range_wall_ms": round(wall_ms, 3), "range_call_ms": round(call_ms, 3),
                  "range_scan_device_ms": round(scan_ms, 3), "search100_wall_ms": round(s_best[0], 3),
                  "search100_scan_device_ms": round(s_best[1], 3), "parity": par})
            del lims, D, I, r
    del index
    torch.cuda.empty_cache()


def ivf_part(device, emit):
    import torch
    from wise_b200 import _capi, faiss_compat as faiss
    L = _capi.lib()
    n, d, nlist, nprobe, seed = 2_000_000, 512, 1024, 8, 77
    centres = bench.RowSource(1, d, seed, device).centres
    ivf = faiss.IndexIVFFlat(faiss.IndexFlatIP(d), d, nlist, faiss.METRIC_INNER_PRODUCT)
    ivf.set_centroids(bench.make_queries(centres, nlist, d, 11, device).cpu().numpy())
    bench.fill_index_clustered(ivf, 0, n, d, seed, device)
    _capi.check(L.wb_ivf_finalize(ivf._h))
    _capi.check(L.wb_set_timing(ivf._h, 1))
    x, ids, assign = ivf._export(0, n, want_assign=True)
    xt = torch.from_numpy(x).to(device)
    at = torch.from_numpy(assign.astype(np.int64)).to(device)
    cent = torch.from_numpy(ivf.centroids()).to(device).double()
    for nq in (1, 256):
        q = bench.make_queries(centres, nq, d, 500 + nq, device)
        qh = q.cpu().numpy()
        probes = torch.topk(q.double() @ cent.T, nprobe, dim=1).indices  # [nq, nprobe]
        member = torch.zeros(nq, nlist, dtype=torch.bool, device=device)
        member.scatter_(1, probes, True)
        cand = lambda s, e: member[:, at[s:e]].T
        reps = 5 if nq == 1 else 3
        run_search(L, ivf._h, qh, 100, nprobe)
        s_best, _ = best_of(lambda: run_search(L, ivf._h, qh, 100, nprobe), reps)
        S = torch.where(cand(0, n), xt.double() @ q.double().T, torch.full((n, nq), -np.inf, device=device, dtype=torch.float64))
        for hits in (10, 1000):
            t = float(torch.topk(S.flatten(), hits * nq).values[-1])
            run_range(L, ivf._h, qh, t, nprobe)
            r, _ = best_of(lambda: run_range(L, ivf._h, qh, t, nprobe), reps)
            lims, D, I, call_ms, wall_ms, scan_ms = r
            pos = np.argsort(ids)
            Ip = pos[np.searchsorted(ids[pos], I)]  # ids -> storage rows of the export
            par = verify([(0, n, xt)], q, lims, D, Ip, t, cand)
            emit({"part": "ivf", "rows": n, "dim": d, "nlist": nlist, "nprobe": nprobe, "batch": nq, "target_hits": hits,
                  "thresh": t, "hits_per_query": float(lims[-1]) / nq, "range_wall_ms": round(wall_ms, 3),
                  "range_call_ms": round(call_ms, 3), "range_scan_device_ms": round(scan_ms, 3),
                  "search100_wall_ms": round(s_best[0], 3), "search100_scan_device_ms": round(s_best[1], 3),
                  "parity": par})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    ap.add_argument("--skip-ivf", action="store_true")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_range.py needs a CUDA device")
    device = torch.device("cuda:0")
    fh = open(a.out, "a") if a.out else None

    def emit(rec):
        line = json.dumps(rec)
        print(line, flush=True)
        if fh:
            fh.write(line + "\n")
            fh.flush()

    emit({"gpu": gpu_info(), "torch": torch.__version__})
    flat_part(a, device, emit)
    if not a.skip_ivf:
        ivf_part(device, emit)


if __name__ == "__main__":
    main()
