"""Where the time of a one-query scan goes: per-CTA %globaltimer stamps (WB_PHASE_TS=1, wb_phase_stamps) of the fused
scan kernel for a flat store and an IVF index.  Prints, per case, the
median / max over CTAs of every phase boundary relative to the earliest CTA start, and the last CTA's merge time.
    python scripts/phase_times.py"""
import ctypes as C
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(__file__), ".."))
os.environ["WB_PHASE_TS"] = "1"
from wise_b200 import _capi, faiss_compat as faiss  # noqa: E402
from bench import fill_index_clustered, make_queries  # noqa: E402

L = _capi.lib()
dev = torch.device("cuda", 0)
NAMES = ["start", "centroids scored", "coarse barrier", "probes selected", "prologue done", "rows done", "final sort",
         "arrived", "merge selected", "results written", "heads staged", "heads T0", "heads compacted", "heads ranked"]


def stamps(idx, qd, k, nprobe, ctas=148):
    D = torch.empty(qd.shape[0], k, device=dev)
    I = torch.empty(qd.shape[0], k, dtype=torch.int64, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    out = []
    for _ in range(6):
        _capi.check(L.wb_search_dev(idx._h, qd.shape[0], qd.data_ptr(), k, nprobe, D.data_ptr(), I.data_ptr(), st))
        torch.cuda.synchronize()
        buf = np.zeros((ctas, 16), np.uint64)
        _capi.check(L.wb_phase_stamps(idx._h, buf.ctypes.data_as(C.c_void_p), ctas))
        out.append(buf.astype(np.int64))
    return out[-1]  # a warm one


def report(tag, ts, extra):
    t0 = ts[:, 0].min()
    rec = {"case": tag, **extra}
    last = int(np.argmax(ts[:, 7]))  # the CTA that arrived last ran the merge; other CTAs hold stale stamps there
    for i, name in enumerate(NAMES):
        col = ts[:, i] if i < 8 else ts[last:last + 1, i]
        live = col[col > 0]
        if live.size == 0:
            continue
        rel = (live - t0) / 1e3
        rec[name] = {"median_us": round(float(np.median(rel)), 2), "max_us": round(float(rel.max()), 2), "ctas": int(live.size)}
    print(json.dumps(rec), flush=True)


def main():
    for n, d in ((100_000, 512), (1_250_000, 768)):
        flat = faiss.IndexIDMap(faiss.IndexFlatIP(d))
        centres, _ = fill_index_clustered(flat, 0, n, d, 50, dev)
        q = make_queries(centres, 1, d, 7, dev)
        report("flat", stamps(flat, q, 100, 1), {"rows": n, "d": d})
        del flat
        torch.cuda.empty_cache()
    n, d, nlist = 2_000_000, 512, 1024
    flat = faiss.IndexIDMap(faiss.IndexFlatIP(d))
    centres, _ = fill_index_clustered(flat, 0, nlist, d, 50, dev)
    x, _, _ = flat._export(0, nlist)
    ivf = faiss.IndexIVFFlat(faiss.IndexFlatIP(d), d, nlist, faiss.METRIC_INNER_PRODUCT)
    ivf.set_centroids(x)
    fill_index_clustered(ivf, 0, n, d, 50, dev)
    q = make_queries(centres, 1, d, 8, dev)
    for nprobe in (8, 32):
        report("ivf", stamps(ivf, q, 100, nprobe), {"rows": n, "nlist": nlist, "nprobe": nprobe})


if __name__ == "__main__":
    main()
