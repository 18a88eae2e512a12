#!/usr/bin/env python
"""Sharded range search (ShardedIndex.range_search, DESIGN.md "Range search") on 1-8 B200s of one box: cost of each
step against the sharded k = 100 search of the same queries, in the same run.

    python -m torch.distributed.run --nproc-per-node G scripts/bench_sharded_range.py [--rows 10000000] [--dim 768]
        [--out profiles/range_sharded/bench_sharded_range.jsonl]

Workload: bench.py's clustered 10M x 768 store (ids = positions) split over the G ranks with shard_range, batches 1 / 16
/ 1024, one threshold per batch chosen from fp64 scores against the first 500k rows so that a query has about 10, 10^3
and 10^5 hits on average (as scripts/bench_range.py).  Per case (rank 0 writes, times are the maximum over the ranks):
host wall time of range_search (numpy in and out) and of range_search_dev (device queries, device D / I), the
range_search_dev time split by CUDA events into the local call (wb_range_search_dev + copy-out), the counts exchange,
the payload exchange and the merge (wb_range_merge_dev), and the wall time of the sharded search_dev / search with
k = 100.  Every timed result is verified in-run: range_search_dev must equal range_search byte for byte, and that result
is checked against fp64 over the regenerated rows (each rank checks the hits in its own rows; the verdicts are
combined), with the tolerances of bench_range.py.  The store (30 GB) is far larger than the 126 MB L2.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import numpy as np  # noqa: E402

import bench  # noqa: E402
from bench_range import gpu_info, thresholds, verify  # noqa: E402


class PhaseEvents:
    """CUDA events at the step boundaries of range_search_dev: the local call, the counts all-gather (the first
    collective), the payload (the flag all-reduce and the two all-gathers) and the merge."""

    def __init__(self, sharded_module, sh):
        import torch
        self.torch, self.marks = torch, []
        local, merge, dist = sh._local_range_search, sh._range_merge, sharded_module.dist
        gather, reduce = dist.all_gather_into_tensor, dist.all_reduce

        def mark(name):
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            self.marks.append((name, ev))

        def timed(name, fn):
            def call(*args, **kw):
                out = fn(*args, **kw)
                mark(name)
                return out
            return call

        sh._local_range_search = timed("local", local)
        sh._range_merge = timed("merge", merge)

        class Dist:  # the torch.distributed calls of sharded.py, each followed by an event
            def __getattr__(self, name):
                return getattr(dist, name)

            def all_gather_into_tensor(s, *a, **kw):
                out = gather(*a, **kw)
                mark("counts" if not any(n == "counts" for n, _ in self.marks) else "payload")
                return out

            def all_reduce(s, *a, **kw):
                out = reduce(*a, **kw)
                mark("payload")
                return out

        sharded_module.dist = Dist()
        self.mark = mark

    def start(self):
        self.marks = []
        self.mark("start")

    def split_ms(self):
        """ms of each step of the last call (steps that did not run are 0)."""
        self.torch.cuda.synchronize()
        out = {"local": 0.0, "counts": 0.0, "payload": 0.0, "merge": 0.0}
        for (_, a), (name, b) in zip(self.marks, self.marks[1:]):
            out[name] += a.elapsed_time(b)
        return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file (rank 0)")
    a = ap.parse_args()
    import torch
    import torch.distributed as dist
    from wise_b200 import faiss_compat as faiss
    from wise_b200 import sharded as S

    if not torch.cuda.is_available():
        sys.exit("bench_sharded_range.py needs a CUDA device")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)
    fh = open(a.out, "a") if (a.out and rank == 0) else None

    def emit(rec):
        if rank == 0:
            line = json.dumps(rec)
            print(line, flush=True)
            if fh:
                fh.write(line + "\n")
                fh.flush()

    def worst(x):  # max over the ranks
        t = torch.tensor([x], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    emit({"gpu": gpu_info(), "torch": torch.__version__, "world": world,
          "exchange": os.environ.get("WISE_B200_EXCHANGE", "peer")})
    n, d = a.rows, a.dim
    lo, hi = S.shard_range(n, rank, world)
    src = bench.RowSource(n, d, 2024, device)
    index = faiss.IndexIDMap(faiss.IndexFlatIP(d, device=local_rank))
    bench.fill_index(index, src, lo, hi)
    sh = S.ShardedIndex(index)
    phases = PhaseEvents(S, sh)
    sample = next(iter(src.chunks(0, min(n, 500_000))))[2]
    for nq in (1, 16, 1024):
        q = bench.make_queries(src.centres, nq, d, 3000 + nq, device)
        qh = q.cpu().numpy()
        reps = {1: 5, 16: 3, 1024: 2}[nq]
        # sharded k = 100 search of the same queries
        sh.search_dev(q, 100)
        sh.search(qh, 100)
        s_dev, s_host = [], []
        for _ in range(reps):
            barrier()
            t0 = time.perf_counter()
            sh.search_dev(q, 100)
            torch.cuda.synchronize()
            s_dev.append(worst((time.perf_counter() - t0) * 1e3))
            barrier()
            t0 = time.perf_counter()
            sh.search(qh, 100)
            s_host.append(worst((time.perf_counter() - t0) * 1e3))
        ths = thresholds(sample, q, (10, 1000, 100_000), n)
        if world > 1:  # the same thresholds on every rank
            tt = torch.tensor([ths[h] for h in (10, 1000, 100_000)], dtype=torch.float64, device=device)
            dist.broadcast(tt, 0)
            ths = dict(zip((10, 1000, 100_000), tt.tolist()))
        for hits, t in ths.items():
            sh.range_search(qh, t)  # warm-up (pool growth)
            sh.range_search_dev(q, t)
            host_ms, dev_ms, splits, same = [], [], [], True
            for _ in range(reps):
                barrier()
                t0 = time.perf_counter()
                lims, D, I = sh.range_search(qh, t)
                host_ms.append(worst((time.perf_counter() - t0) * 1e3))
                barrier()
                phases.start()
                t0 = time.perf_counter()
                ld, Dd, Id = sh.range_search_dev(q, t)
                torch.cuda.synchronize()
                dev_ms.append(worst((time.perf_counter() - t0) * 1e3))
                splits.append({k: worst(v) for k, v in phases.split_ms().items()})
                same = (same and np.array_equal(ld.numpy().astype(np.uint64), lims)
                        and np.array_equal(Dd.cpu().numpy(), D) and np.array_equal(Id.cpu().numpy(), I))
                del ld, Dd, Id
            par = verify(src.chunks(lo, hi), q, lims.astype(np.int64), D, I, t)
            ok = torch.tensor([int(par["ok"] and same)], dtype=torch.int64, device=device)
            if world > 1:
                dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            best = int(np.argmin(dev_ms))
            emit({"rows": n, "dim": d, "world": world, "batch": nq, "target_hits": hits, "thresh": t,
                  "hits_per_query": float(lims[-1]) / nq, "max_hits": int(np.diff(lims.astype(np.int64)).max()),
                  "range_search_wall_ms": round(min(host_ms), 3), "range_search_dev_wall_ms": round(dev_ms[best], 3),
                  "range_search_dev_split_ms": {k: round(v, 3) for k, v in splits[best].items()},
                  "search100_dev_wall_ms": round(min(s_dev), 3), "search100_wall_ms": round(min(s_host), 3),
                  "dev_equals_host": bool(same), "parity_rank0": par, "parity_all_ranks_ok": bool(ok.item())})
            del lims, D, I
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
