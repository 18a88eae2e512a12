"""The int8 filter of K1 on bench.py's flagship store (10M x 768 clustered rows, top-100): per search of 1 and 2
queries, the image bytes streamed, the (row, query) pairs re-scored in fp32 (wb_flat_bf16_stats), the bytes actually
read (image + re-scored rows) over the scan kernel's time, and the image's memory.  One JSON line per batch size.

    python scripts/bench_bf16_scan.py [--rows N] [--dim D] [--k K] [--searches S] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_name_and_power():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else None
    except (OSError, subprocess.SubprocessError):
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--searches", type=int, default=50)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch

    import bench
    from wise_b200 import _capi
    from wise_b200 import faiss_compat as faiss
    from wise_b200.sharded import ShardedIndex

    if not torch.cuda.is_available():
        raise SystemExit("needs a B200")
    device = torch.device("cuda", 0)
    L = _capi.lib()
    src = bench.RowSource(a.rows, a.dim, 2024, device)
    index = faiss.IndexIDMap(faiss.IndexFlatIP(a.dim, device=0))
    bench.fill_index(index, src, 0, a.rows)
    L.wb_set_timing(index._h, 1)
    search = ShardedIndex(index).search_dev  # device queries in, device (D, I) out: the path bench.py times
    ld = (a.dim + 3) & ~3
    row_bytes = 16 + ((ld + 15) & ~15)  # img_row_bytes (scan.cuh): a 16-byte header and the codes

    def stats():
        s, r = C.c_int64(0), C.c_int64(0)
        _capi.check(L.wb_flat_bf16_stats(index._h, C.byref(s), C.byref(r)))
        return s.value, r.value

    lines = []
    for nq in (1, 2):
        qs = bench.make_queries(src.centres, nq * (a.searches + 5), a.dim, 2025, device).view(a.searches + 5, nq, a.dim)
        for i in range(5):
            search(qs[i], a.k)
        torch.cuda.synchronize()
        s0, r0 = stats()
        for i in range(a.searches):
            search(qs[5 + i], a.k)
        torch.cuda.synchronize()
        s1, r1 = stats()
        buf = (C.c_float * 128)()
        n = L.wb_scan_ms_history(index._h, buf, min(a.searches, 128))
        scan_ms = float(np.mean([buf[i] for i in range(n)]))
        img_bytes = a.rows * row_bytes
        pairs = (r1 - r0) / max(1, s1 - s0)
        read = img_bytes + pairs * ld * 4  # a pair re-scored reads its fp32 row (from L2 when queries share it)
        line = {"batch": nq, "searches_on_image": s1 - s0, "searches": a.searches, "scan_ms": scan_ms,
                "image_bytes_per_search": img_bytes, "rescored_pairs_per_search": pairs,
                "rescored_fraction": pairs / (a.rows * nq), "bytes_read_per_search": read,
                "read_tb_per_s": read / (scan_ms * 1e-3) / 1e12,
                "fp32_equivalent_tb_per_s": a.rows * ld * 4 / (scan_ms * 1e-3) / 1e12,
                "image_memory_bytes": img_bytes, "fp32_store_bytes": a.rows * ld * 4,
                "rows": a.rows, "dim": a.dim, "k": a.k, "gpu": gpu_name_and_power()}
        print(json.dumps(line), flush=True)
        lines.append(line)
    if a.out:
        with open(a.out, "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
