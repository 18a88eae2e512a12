"""Host-call time per search of an index over N GPUs of one process (faiss_compat devices=, wb_group), N = 1, 2, 4, 8
(as many as the box has), against the single-GPU index holding every row:

  - flat 10M x 768 at batches 1, 16 and 1024 (k = 100);
  - IVF 2M x 512, nlist 1024, nprobe 8, one query (k = 100);
  - the fan-out itself: one query over 1000 rows per GPU, where the search is nothing but the group's overhead;
  - the same flat and IVF searches through `ShardedIndex` (one process per GPU, started with torch.multiprocessing as
    the multi-GPU tests start it; rank 0's host-call time).

The stores are integer-valued, so every result must be byte-identical to the single-GPU index's; the script checks it
for every timed search and fails otherwise.  One JSON line per measurement, plus the GPU name and power limit, goes to
--out.  Run: python scripts/bench_group.py --out profiles/r04/bench_group.jsonl"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from wise_b200 import faiss_compat as faiss  # noqa: E402


def chunks(n, d, seed, chunk=1 << 20, dev=0, lo=0, hi=None):
    """Integer-valued rows m / 4, m in [-3, 3], generated on GPU `dev` chunk by chunk (the store never sits on the host
    whole); only rows [lo, hi) are returned.  The same seed gives the same rows on every GPU."""
    hi = n if hi is None else hi
    g = torch.Generator(device=f"cuda:{dev}")
    g.manual_seed(seed)
    for a in range(0, n, chunk):
        m = min(chunk, n - a)
        x = torch.randint(-3, 4, (m, d), generator=g, device=f"cuda:{dev}", dtype=torch.int8)
        s0, s1 = max(lo, a), min(hi, a + m)
        if s0 < s1:
            yield s0, (x[s0 - a:s1 - a].float() / 4).cpu().numpy()


def build_flat(n, d, devices, dev=0, lo=0, hi=None):
    idx = faiss.IndexIDMap(faiss.IndexFlatIP(d, devices=devices))  # ids = global positions, on every leg
    hi = n if hi is None else hi
    idx.reserve(hi - lo)
    for a, x in chunks(n, d, 1, dev=dev, lo=lo, hi=hi):
        idx.add_with_ids(x, np.arange(a, a + x.shape[0], dtype=np.int64))
    return idx


def build_ivf(n, d, nlist, devices, dev=0, lo=0, hi=None):
    idx = faiss.IndexIVFFlat(faiss.IndexFlatIP(d, devices=devices), d, nlist)
    cent = next(chunks(nlist, d, 2, dev=dev))[1]
    idx.set_centroids(cent)
    hi = n if hi is None else hi
    idx.reserve(hi - lo)
    for a, x in chunks(n, d, 3, dev=dev, lo=lo, hi=hi):
        idx.add_with_ids(x, np.arange(a, a + x.shape[0], dtype=np.int64))
    idx.nprobe = 8
    return idx


def _sharded_worker(rank, world, port, out, flat_rows, ivf_rows, reps, qfile):
    """One rank of the ShardedIndex leg: builds its contiguous slice, runs the same timed searches as every rank."""
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), WISE_B200_DEVICE=str(rank))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from wise_b200.sharded import ShardedIndex, shard_range
        qs = dict(np.load(qfile))
        res = {}
        lo, hi = shard_range(flat_rows, rank, world)
        sh = ShardedIndex(build_flat(flat_rows, 768, [rank], dev=rank, lo=lo, hi=hi))
        for b in (1, 16, 1024):
            med, best, (D, I) = time_calls(sh, qs[f"flat{b}"], 100, reps if b < 1024 else max(5, reps // 5))
            res.update({f"flat{b}_D": D, f"flat{b}_I": I, f"flat{b}_t": np.array([med, best])})
        del sh
        lo, hi = shard_range(ivf_rows, rank, world)
        sh = ShardedIndex(build_ivf(ivf_rows, 512, 1024, [rank], dev=rank, lo=lo, hi=hi))
        med, best, (D, I) = time_calls(sh, qs["ivf1"], 100, reps * 4)
        res.update({"ivf1_D": D, "ivf1_I": I, "ivf1_t": np.array([med, best])})
        if rank == 0:
            np.savez(out, **res)
    finally:
        dist.destroy_process_group()


def time_calls(idx, q, k, reps, warmup=5):
    for _ in range(warmup):
        out = idx.search(q, k)
    t = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = idx.search(q, k)
        t.append(time.perf_counter() - t0)
    return float(np.median(t)) * 1e6, float(np.min(t)) * 1e6, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--flat-rows", type=int, default=10_000_000)
    ap.add_argument("--ivf-rows", type=int, default=2_000_000)
    ap.add_argument("--reps", type=int, default=50)
    a = ap.parse_args()
    os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
    ngpu = torch.cuda.device_count()
    if ngpu < 1:
        raise SystemExit("no GPU")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    ns = [n for n in (1, 2, 4, 8) if n <= ngpu]
    k = 100
    rng = np.random.default_rng(9)
    out = open(a.out, "w")

    def emit(rec):
        rec["gpu"] = gpu[0] if gpu else "?"
        print(json.dumps(rec), flush=True)
        out.write(json.dumps(rec) + "\n")

    emit({"what": "box", "gpus": gpu})
    # fan-out cost: a store so small that the search itself is a few microseconds
    qtiny = (rng.integers(-3, 4, (1, 64)) / 4).astype(np.float32)
    for n in ns:
        idx = build_flat(1000 * n, 64, list(range(n)))
        med, best, res = time_calls(idx, qtiny, 10, a.reps * 4)
        emit({"what": "fanout_tiny_flat", "gpus": n, "rows": 1000 * n, "call_us_median": med, "call_us_min": best})
        del idx
    # flat 10M x 768
    qs = {b: (rng.integers(-3, 4, (b, 768)) / 4).astype(np.float32) for b in (1, 16, 1024)}
    qivf = (rng.integers(-3, 4, (1, 512)) / 4).astype(np.float32)
    single = build_flat(a.flat_rows, 768, [0])
    ref = {b: single.search(qs[b], k) for b in qs}
    for n in ns:
        idx = single if n == 1 else build_flat(a.flat_rows, 768, list(range(n)))
        for b, q in qs.items():
            med, best, res = time_calls(idx, q, k, a.reps if b < 1024 else max(5, a.reps // 5))
            ok = all(np.array_equal(u.view(np.uint8), v.view(np.uint8)) for u, v in zip(res, ref[b]))
            emit({"what": "flat", "rows": a.flat_rows, "d": 768, "gpus": n, "batch": b, "k": k, "call_us_median": med,
                  "call_us_min": best, "qps": b * 1e6 / med, "identical_to_single": ok})
            if not ok:
                raise SystemExit("result differs from the single-GPU index")
        if n > 1:
            del idx
    del single
    # IVF 2M x 512, nlist 1024, nprobe 8, one query
    q = qivf
    single = build_ivf(a.ivf_rows, 512, 1024, [0])
    r0 = single.search(q, k)
    for n in ns:
        idx = single if n == 1 else build_ivf(a.ivf_rows, 512, 1024, list(range(n)))
        med, best, res = time_calls(idx, q, k, a.reps * 4)
        ok = all(np.array_equal(u.view(np.uint8), v.view(np.uint8)) for u, v in zip(res, r0))
        emit({"what": "ivf", "rows": a.ivf_rows, "d": 512, "nlist": 1024, "nprobe": 8, "gpus": n, "batch": 1, "k": k,
              "call_us_median": med, "call_us_min": best, "qps": 1e6 / med, "identical_to_single": ok})
        if not ok:
            raise SystemExit("result differs from the single-GPU index")
        if n > 1:
            del idx
    del single
    # ShardedIndex: one process per GPU, the same rows, queries and checks
    import socket
    import tempfile

    import torch.multiprocessing as mp
    with tempfile.TemporaryDirectory() as tmp:
        qfile = os.path.join(tmp, "q.npz")
        np.savez(qfile, ivf1=qivf, **{f"flat{b}": q for b, q in qs.items()})
        for n in ns:
            with socket.socket() as sk:
                sk.bind(("127.0.0.1", 0))
                port = sk.getsockname()[1]
            res_file = os.path.join(tmp, f"sharded{n}.npz")
            mp.spawn(_sharded_worker, args=(n, port, res_file, a.flat_rows, a.ivf_rows, a.reps, qfile), nprocs=n,
                     join=True)
            got = np.load(res_file)
            for b in qs:
                ok = all(np.array_equal(u.view(np.uint8), v.view(np.uint8))
                         for u, v in zip((got[f"flat{b}_D"], got[f"flat{b}_I"]), ref[b]))
                med, best = got[f"flat{b}_t"]
                emit({"what": "flat_sharded_index", "rows": a.flat_rows, "d": 768, "gpus": n, "batch": b, "k": k,
                      "call_us_median": float(med), "call_us_min": float(best), "qps": b * 1e6 / float(med),
                      "identical_to_single": ok})
                if not ok:
                    raise SystemExit("ShardedIndex result differs from the single-GPU index")
            ok = all(np.array_equal(u.view(np.uint8), v.view(np.uint8)) for u, v in zip((got["ivf1_D"], got["ivf1_I"]), r0))
            med, best = got["ivf1_t"]
            emit({"what": "ivf_sharded_index", "rows": a.ivf_rows, "d": 512, "nlist": 1024, "nprobe": 8, "gpus": n,
                  "batch": 1, "k": k, "call_us_median": float(med), "call_us_min": float(best), "qps": 1e6 / float(med),
                  "identical_to_single": ok})
            if not ok:
                raise SystemExit("ShardedIndex result differs from the single-GPU index")
    out.close()


if __name__ == "__main__":
    main()
