#!/usr/bin/env python
"""bench.py - the headline benchmark of BASELINE.json on B200:
IndexFlatIP exact top-100 over 10M x 768 fp32 (ViT-L/14 dim), synthetic unit vectors.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl ours|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one search of a batch of B queries (default B=1: the bandwidth-bound case the
reference serves, /root/reference/api/routes.py:1407) over the whole database:
  value    QPS with queries already in HBM (wb_search_dev), CUDA events on the launching stream
  e2e      QPS through the public API `index.search(numpy, k)` with pinned HOST buffers: H2D of
           the queries and D2H of (D, I) inside the timed region (result sets up to 64 KB are written by the
           emitting kernel straight into pinned host memory over PCIe, larger ones are copied; same bytes either way)
  roofline achieved = N*d*4 bytes / scan-kernel duration (events inside the library, same stream)
           vs the measured copy bandwidth in MEASURED_PEAKS.json
  parity_check  the (D, I) of the LAST timed step verified after the timed region on every rank against an fp64
           pass over the regenerated rows (torch, chunked): returned scores within 1e-5, no row outside the
           result beats the k-th score beyond the 4e-6 near-tie band, all ranks returned identical bytes, and a
           planted exact duplicate (last row == row 0, on different ranks when N > 1) ties in insertion order
  secondary (N = 1) the same measurement at batch 16 (K2, HBM roofline) and batch 1024 (K2 256-query blocks,
           tensor roofline against the TF32 peak measured live with the library's own MMA shape), each with its own
           parity_check; batch 1024 also carries the BLAS-path CPU baseline; `ivf_one_query`: IndexIVFFlat 2M x 512,
           nlist 1024, ONE query per call (the product's case): device path and host call at nprobe 8 / 32 with the
           coarse quantizer inside the list-scan launch and as its own launch, byte-identity, exhaustive parity check
  cpu_baseline  the faiss-equivalent C restatement (oracle/cpu_flat.c) on this box's host cores,
           on a bounded row sample, scaled linearly (faiss itself is not installable: BASELINE.md 3)
N > 1: the 10M rows are split into N contiguous shards (strong scaling), one process per GPU; the exchange of
the k candidates per query is the library's own NVLink peer-memory kernel (exchange.cuh), NCCL carries only the
benchmark's barriers and reductions.
`--impl reference` times the CPU restatement with all host threads (rank 0 only), on the full 10M x 768 matrix
when host memory allows.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "QPS, IndexFlatIP top-100 (10Mx768 fp32)"
HBM_FALLBACK_GBS = 6650.0  # B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent
GEN_CHUNK = 250_000        # rows per generator chunk (global grid: the same rows whatever the sharding)
NCENTRES = 4096
SCORE_TOL = 1e-5           # BASELINE.json north_star
TIE_BAND = 4e-6            # near-tie band of the parity contract (DESIGN.md section 5)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=1)
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--cpu-sample-rows", type=int, default=1_000_000)
    ap.add_argument("--sweep", default="", help="comma list of extra batch sizes to report, e.g. 2,4,8")
    ap.add_argument("--secondary", default="auto", help="comma list of extra batch sizes measured WITH roofline and "
                    "parity_check (default: 16,1024 on one GPU at batch 1; 'none' to skip)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--mixed", action="store_true",
                    help="config 5: half of the batch are 'combined' queries normalise(2.0*t + 1.0*i - 0.2*n) "
                         "(/root/reference/api/routes.py:759-850)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the (D, I) the last one returned as DIR/D.npy and DIR/I.npy")
    return ap.parse_args()


DUMP_MAX_BYTES = 60 << 20  # keeps the two files, headers included, under 64 MB


def dump_outputs(out_dir, D, I):
    """--dump-outputs: the scores D (float32) and ids I (int64 stored as float64, exact below 2**53) of the last timed
    step, so that two builds can be compared output for output on the same seeded inputs.  When the pair exceeds
    DUMP_MAX_BYTES, a fixed seeded sample of the query rows is written instead (the same rows for the same arguments)."""
    D = np.asarray(D, dtype=np.float32)
    I = np.asarray(I).astype(np.float64)
    row_bytes = D.shape[1] * (D.itemsize + I.itemsize)
    if D.shape[0] * row_bytes > DUMP_MAX_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(D.shape[0], DUMP_MAX_BYTES // row_bytes, replace=False))
        D, I = D[rows], I[rows]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "D.npy"), D)
    np.save(os.path.join(out_dir, "I.npy"), I)


def workload_name(a, batch=None):
    b = a.batch if batch is None else batch
    return f"IndexFlatIP top-{a.k} over {a.rows}x{a.dim} fp32, query batch {b}" + (" (mixed text/combined)" if a.mixed else "")


def config_of(a, batch=None):
    """Identical on both arms (ours / reference) for the same command line."""
    return {"workload": workload_name(a, batch), "rows": a.rows, "dim": a.dim, "k": a.k,
            "batch": a.batch if batch is None else batch,
            "generator": f"clustered unit vectors, {NCENTRES} centres, noise 0.6 (SURVEY.md 8d)",
            "l2": "database (>= 3.8 GB per GPU) is far larger than the 126 MB L2; no flush needed"}


# ------------------------------------------------------------------------------------------------
# synthetic "CLIP-like" data (SURVEY.md 8d): rows = normalise(c_j + 0.6 g), generated on the device
# ------------------------------------------------------------------------------------------------
class RowSource:
    """Global rows [0, rows) on a fixed chunk grid, chunk c seeded by (seed, c): any rank can regenerate any
    row.  The LAST row is an exact copy of row 0 (the planted duplicate of the parity check)."""

    def __init__(self, rows, d, seed, device, ncentres=NCENTRES):
        import torch
        self.rows, self.d, self.seed, self.device = rows, d, seed, device
        gen = torch.Generator(device=device)
        gen.manual_seed(seed)
        self.centres = torch.nn.functional.normalize(torch.randn(ncentres, d, device=device, generator=gen), dim=1)
        self._row0 = None

    def _chunk(self, c):
        import torch
        s, e = c * GEN_CHUNK, min(self.rows, (c + 1) * GEN_CHUNK)
        g2 = torch.Generator(device=self.device)
        g2.manual_seed(self.seed * 1_000_003 + c)
        j = torch.randint(0, self.centres.shape[0], (e - s,), device=self.device, generator=g2)
        x = self.centres[j] + 0.6 * torch.randn(e - s, self.d, device=self.device, generator=g2) / (self.d ** 0.5)
        return torch.nn.functional.normalize(x, dim=1)

    def row0(self):
        if self._row0 is None:
            self._row0 = self._chunk(0)[0].clone()
        return self._row0

    def chunks(self, lo, hi):
        """Yield (s, e, x[e-s, d]) covering [lo, hi) in grid order."""
        for c in range(lo // GEN_CHUNK, (hi + GEN_CHUNK - 1) // GEN_CHUNK):
            cs, ce = c * GEN_CHUNK, min(self.rows, (c + 1) * GEN_CHUNK)
            x = self._chunk(c)
            if ce == self.rows and self.rows > 1:
                x[-1] = self.row0()  # planted duplicate
            s, e = max(cs, lo), min(ce, hi)
            yield s, e, x[s - cs:e - cs].contiguous()


def fill_index(index, src, lo, hi):
    import torch
    from wise_b200 import _capi
    L = _capi.lib()
    st = torch.cuda.current_stream().cuda_stream
    index.reserve(hi - lo)
    for s, e, x in src.chunks(lo, hi):
        ids = torch.arange(s, e, dtype=torch.int64, device=src.device)
        _capi.check(L.wb_add_with_ids_dev(index._h, e - s, x.data_ptr(), ids.data_ptr(), st))
        torch.cuda.synchronize()


def fill_index_clustered(index, lo, hi, d, seed, device, chunk=500_000, ncentres=NCENTRES):
    """Older helper kept for scripts/: rows [lo, hi) of a clustered store (chunks addressed by their start row)."""
    import torch
    from wise_b200 import _capi
    L = _capi.lib()
    gen = torch.Generator(device=device)
    gen.manual_seed(seed)
    centres = torch.nn.functional.normalize(torch.randn(ncentres, d, device=device, generator=gen), dim=1)
    st = torch.cuda.current_stream().cuda_stream
    index.reserve(hi - lo)
    sample = None
    for s in range(lo, hi, chunk):
        e = min(hi, s + chunk)
        g2 = torch.Generator(device=device)
        g2.manual_seed(seed * 1_000_003 + s)
        j = torch.randint(0, ncentres, (e - s,), device=device, generator=g2)
        x = centres[j] + 0.6 * torch.randn(e - s, d, device=device, generator=g2) / (d ** 0.5)
        x = torch.nn.functional.normalize(x, dim=1).contiguous()
        ids = torch.arange(s, e, dtype=torch.int64, device=device)
        _capi.check(L.wb_add_with_ids_dev(index._h, e - s, x.data_ptr(), ids.data_ptr(), st))
        torch.cuda.synchronize()
        if sample is None:
            sample = x
    return centres, sample


MIXED = False


def make_queries(centres, nq, d, seed, device):
    import torch
    gen = torch.Generator(device=device)
    gen.manual_seed(seed)

    def draw(m):
        j = torch.randint(0, centres.shape[0], (m,), device=device, generator=gen)
        v = centres[j] + 0.6 * torch.randn(m, d, device=device, generator=gen) / (d ** 0.5)
        return torch.nn.functional.normalize(v, dim=1)

    q = draw(nq)
    if MIXED and nq > 1:  # second half: text x2.0 + image x1.0 - negative x0.2, renormalised
        h = nq // 2
        q[h:] = torch.nn.functional.normalize(2.0 * q[h:] + 1.0 * draw(nq - h) - 0.2 * draw(nq - h), dim=1)
    return q.contiguous()


# ------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """SM clock + throttle reasons of one GPU every 20 ms while the timed region runs (NVML through
    nvidia_ml_py: `nvidia-smi -lms` block-buffers its pipe output and delivered only 1-7 lines per run)."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.sm, self.reasons, self.power = [], set(), []
        self.sm_max = None
        self._halt = threading.Event()

    def run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.gpu]) if vis and vis.split(",")[self.gpu].isdigit() else self.gpu
            h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            while not self._halt.is_set():
                self.sm.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                try:
                    r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    for bit, name in self.REASONS.items():
                        if r & bit:
                            self.reasons.add(name)
                    self.power.append(pynvml.nvmlDeviceGetPowerUsage(h) / 1000.0)
                except Exception:
                    pass
                time.sleep(0.02)
        except Exception:
            pass

    def finish(self):
        self._halt.set()
        self.join(timeout=2)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.sm_max,
                "reasons": sorted(self.reasons), "samples": len(self.sm),
                "power_w_max": max(self.power) if self.power else None, "source": "nvml"}


def cpu_info():
    model = "unknown"
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    return {"model": model, "cpu_count": os.cpu_count(), "affinity": len(os.sched_getaffinity(0))}


def mem_available_bytes():
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable:"):
                return int(line.split()[1]) * 1024
    except OSError:
        pass
    return 0


def host_threads():
    """All the host threads this process may use (torch.distributed.run exports OMP_NUM_THREADS=1: ignored)."""
    return max(1, len(os.sched_getaffinity(0)))


def cpu_restatement(sample_rows, q, k, n_full, mt, reps=3):
    """Time oracle/cpu_flat.c (faiss-equivalent restatement) on `sample_rows`, scale to n_full rows."""
    from oracle import cpu as OC
    OC.set_threads(host_threads())
    OC.flat_search(sample_rows[:1000], q, k, mt=mt)  # warm-up (thread pool, page-in)
    ts = []
    for _ in range(reps):
        t = time.perf_counter()
        OC.flat_search(sample_rows, q, k, mt=mt)
        ts.append(time.perf_counter() - t)
    t_med = float(np.median(ts))
    scale = n_full / sample_rows.shape[0]
    return q.shape[0] / (t_med * scale), t_med, (OC.max_threads() if mt else min(q.shape[0], OC.max_threads())), OC.simd_name()


def cpu_blas(sample_rows, q, k, n_full, reps=3):
    """faiss's n >= 20 path restated: OpenBLAS sgemm tiles + partial selection (oracle/cpu.py blas_flat_search)."""
    from oracle import cpu as OC
    th = host_threads()
    OC.blas_flat_search(sample_rows[:20000], q, k, threads=th)
    ts = []
    for _ in range(reps):
        t = time.perf_counter()
        OC.blas_flat_search(sample_rows, q, k, threads=th)
        ts.append(time.perf_counter() - t)
    t_med = float(np.median(ts))
    scale = n_full / sample_rows.shape[0]
    return q.shape[0] / (t_med * scale), t_med, th


def cpu_ivf(xs, assign, centroids, q, k, nprobe, n_full, reps=3):
    """cpu_baseline leg of config 3 (scripts/bench_configs.py): the restated IndexIVFFlat.search
    (oracle/cpu_flat.c orc_ivf_search: parallel over queries like faiss parallel_mode 0) on a row sample with the
    index's own centroids and list assignment; QPS scaled to n_full rows."""
    from oracle import cpu as OC
    OC.set_threads(host_threads())
    nlist = centroids.shape[0]
    order = np.argsort(assign, kind="stable").astype(np.int64)
    offs = np.concatenate([[0], np.cumsum(np.bincount(assign, minlength=nlist))]).astype(np.int64)
    OC.ivf_search(xs, None, offs, order, centroids, q, k, nprobe)
    ts = []
    for _ in range(reps):
        t = time.perf_counter()
        OC.ivf_search(xs, None, offs, order, centroids, q, k, nprobe)
        ts.append(time.perf_counter() - t)
    t_med = float(np.median(ts))
    return q.shape[0] / (t_med * n_full / xs.shape[0]), t_med, min(q.shape[0], host_threads())


def cpu_kmeans_iteration(xs, centroids, n_full):
    """cpu_baseline leg of config 4: one restated Clustering iteration (oracle.kmeans_iteration: numpy / OpenBLAS fp64
    assignment + update) on a point sample against ALL centroids; seconds scaled to n_full points."""
    from oracle import oracle as O
    from threadpoolctl import threadpool_limits
    with threadpool_limits(limits=host_threads()):
        t = time.perf_counter()
        O.kmeans_iteration(xs, centroids)
        dt = time.perf_counter() - t
    return dt * n_full / xs.shape[0], dt, host_threads()


# ------------------------------------------------------------------------------------------------
def gen_clustered_host(n, d, seed, threads):
    """oracle.clustered_unit's distribution, generated chunk-parallel (numpy releases the GIL in the RNG)."""
    from concurrent.futures import ThreadPoolExecutor
    rng = np.random.default_rng(seed)
    centres = rng.standard_normal((NCENTRES, d), dtype=np.float32)
    centres /= np.linalg.norm(centres, axis=1, keepdims=True)
    x = np.empty((n, d), np.float32)
    step = 100_000

    def work(s):
        e = min(n, s + step)
        r = np.random.default_rng(seed * 1_000_003 + s)
        j = r.integers(0, NCENTRES, size=e - s)
        g = r.standard_normal((e - s, d), dtype=np.float32)
        g *= np.float32(0.6 / np.sqrt(d))
        g += centres[j]
        g /= np.linalg.norm(g, axis=1, keepdims=True)
        x[s:e] = g

    with ThreadPoolExecutor(max_workers=threads) as ex:
        list(ex.map(work, range(0, n, step)))
    return centres, x


def run_reference(a):
    """--impl reference: the reference's CPU path (faiss-equivalent restatement; faiss is absent), all host
    threads.  Rank 0 only.  Full 10M x 768 when host memory allows, else a bounded sample scaled linearly."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from oracle import cpu as OC
    th = host_threads()
    OC.set_threads(th)
    need = a.rows * a.dim * 4
    avail = mem_available_bytes()
    n_s = a.rows if avail > need + (12 << 30) else min(a.cpu_sample_rows, a.rows)
    if os.environ.get("WB_REF_ROWS"):
        n_s = min(a.rows, int(os.environ["WB_REF_ROWS"]))
    t0 = time.perf_counter()
    centres, xb = gen_clustered_host(n_s, a.dim, 2024, th)
    rq = np.random.default_rng(2025)
    q = centres[rq.integers(0, NCENTRES, size=a.batch)] + np.float32(0.6 / np.sqrt(a.dim)) * rq.standard_normal((a.batch, a.dim), dtype=np.float32)
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    q = np.ascontiguousarray(q, np.float32)
    t_gen = time.perf_counter() - t0
    use_blas = a.batch >= 20  # faiss: knn_inner_product switches to the BLAS path at 20 queries [faiss-upstream]

    def step():
        if use_blas:
            return OC.blas_flat_search(xb, q, a.k, threads=th)
        return OC.flat_search(xb, q, a.k, mt=True)

    OC.flat_search(xb[:1000], q[:1], a.k, mt=True)
    for _ in range(a.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        D, I = step()
    dt = time.perf_counter() - t0
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, D, I)
    scale = a.rows / n_s
    ms_step = dt / a.steps * 1e3 * scale
    qps = a.batch / (ms_step / 1e3)
    fn = "oracle/cpu.py blas_flat_search (OpenBLAS sgemm tiles + argpartition)" if use_blas else \
        f"oracle/cpu_flat.c orc_flat_search_mt ({OC.simd_name()}, database split over the threads)"
    sample = (("the full matrix" if n_s == a.rows else f"{n_s} of {a.rows} rows per step (time scaled x{scale:g})") +
              f"; {fn}; {th} threads; generated in {t_gen:.1f} s; faiss itself is not installable here")
    line = {"impl": "reference", "metric": METRIC, "value": qps, "unit": "queries/s", "n_gpus": a.gpus, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": config_of(a), "host": cpu_info(),
            "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": th, "kind": "port", "sample": sample},
            "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
def ivf_one_query_secondary(device, k):
    """secondary.ivf_one_query (N = 1): the product's IVF case - ONE query per call (/root/reference/api/routes.py:1407 with
    nprobe from config, :899-902) - on IndexIVFFlat 2M x 512, nlist 1024.  Device path (CUDA events around 200
    back-to-back searches) with the coarse quantizer inside the list-scan launch and as its own launch, the host API
    (numpy in, numpy out), byte-identity of the two, and an exhaustive check (nprobe = nlist) of the returned (D, I)
    against an fp64 pass over regenerated rows.  Any failure is reported in the entry instead of raising: this
    measurement must never cost the headline line."""
    import torch
    from wise_b200 import _capi, faiss_compat as faiss
    L = _capi.lib()
    n, d, nlist, seed, chunk = 2_000_000, 512, 1024, 50, 500_000
    out = {"config": {"workload": f"IndexIVFFlat nlist={nlist} top-{k} over {n}x{d} fp32, query batch 1",
                      "centroids": "the first nlist rows of the store (no training: searches are what is timed)"}}
    saved = os.environ.get("WB_IVF_FUSE_COARSE")
    try:
        gen = torch.Generator(device=device)
        gen.manual_seed(seed)
        centres = torch.nn.functional.normalize(torch.randn(NCENTRES, d, device=device, generator=gen), dim=1)

        def rows_of(s):  # the chunk fill_index_clustered adds at row s
            e = min(n, s + chunk)
            g2 = torch.Generator(device=device)
            g2.manual_seed(seed * 1_000_003 + s)
            j = torch.randint(0, NCENTRES, (e - s,), device=device, generator=g2)
            x = centres[j] + 0.6 * torch.randn(e - s, d, device=device, generator=g2) / (d ** 0.5)
            return torch.nn.functional.normalize(x, dim=1).contiguous()

        ivf = faiss.IndexIVFFlat(faiss.IndexFlatIP(d), d, nlist, faiss.METRIC_INNER_PRODUCT)
        ivf.set_centroids(rows_of(0)[:nlist].cpu().numpy())
        fill_index_clustered(ivf, 0, n, d, seed, device, chunk=chunk)
        q = make_queries(centres, 1, d, 8, device)
        qh = q.cpu().numpy()
        st = torch.cuda.current_stream().cuda_stream
        D = torch.empty(1, k, device=device)
        I = torch.empty(1, k, dtype=torch.int64, device=device)

        def device_ms(nprobe, reps=200):
            call = lambda: _capi.check(L.wb_search_dev(ivf._h, 1, q.data_ptr(), k, nprobe, D.data_ptr(), I.data_ptr(), st))
            for _ in range(20):
                call()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(reps):
                call()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / reps, D.cpu().numpy().copy(), I.cpu().numpy().copy()

        per = {}
        for nprobe in (8, 32):
            ivf.nprobe = nprobe
            os.environ["WB_IVF_FUSE_COARSE"] = "0"
            two_ms, D2, I2 = device_ms(nprobe)
            os.environ["WB_IVF_FUSE_COARSE"] = "1"
            f0, l0 = L.wb_ivf_fused_searches(ivf._h), L.wb_launch_count(ivf._h)
            one_ms, D1, I1 = device_ms(nprobe)
            nsearch = 220
            fused, launches = L.wb_ivf_fused_searches(ivf._h) - f0, L.wb_launch_count(ivf._h) - l0
            wall = []
            for _ in range(220):
                t0 = time.perf_counter()
                Dh, Ih = ivf.search(qh, k)
                wall.append(time.perf_counter() - t0)
            per[f"nprobe{nprobe}"] = {
                "device_ms_per_search": one_ms, "device_ms_two_launches": two_ms,
                "e2e_ms_per_call_median": float(np.median(wall[20:]) * 1e3), "launches_per_search": launches / nsearch,
                "fused_searches": int(fused), "same_bytes_as_two_launches": bool(
                    np.array_equal(I1, I2) and np.array_equal(D1.view(np.uint32), D2.view(np.uint32))
                    and np.array_equal(Ih, I1) and np.array_equal(Dh.view(np.uint32), D1.view(np.uint32)))}
        out.update(per)
        # exhaustive setting: every list probed -> the result must be the exact top-k of all rows
        ivf.nprobe = nlist
        Dx, Ix = ivf.search(qh, k)
        best_s = torch.full((0,), 0.0, dtype=torch.float64, device=device)
        best_i = torch.zeros((0,), dtype=torch.int64, device=device)
        q64 = q[0].double()
        for s0 in range(0, n, chunk):
            sc = rows_of(s0).double() @ q64
            best_s = torch.cat([best_s, sc])
            best_i = torch.cat([best_i, torch.arange(s0, s0 + sc.numel(), device=device)])
            top = torch.topk(best_s, min(4 * k, best_s.numel()))
            best_s, best_i = top.values, best_i[top.indices]
        ref_s, ref_i = best_s.cpu().numpy(), best_i.cpu().numpy()
        score_of = dict(zip(ref_i.tolist(), ref_s.tolist()))
        kth = ref_s[k - 1]
        err = max(abs(float(Dx[0, j]) - score_of.get(int(Ix[0, j]), float("nan"))) for j in range(k))
        bad = sum(1 for j in range(k) if int(Ix[0, j]) not in score_of or score_of[int(Ix[0, j])] < kth - 4e-6)
        out["parity_check"] = {"setting": f"nprobe = nlist = {nlist} (exhaustive)", "rows_checked": n, "max_abs_err": err,
                               "violations": int(bad), "sorted": bool(np.all(np.diff(Dx[0]) <= 0)), "score_tol": 1e-5,
                               "tie_band": 4e-6,
                               "ok": bool(err <= 1e-5 and bad == 0 and np.all(np.diff(Dx[0]) <= 0)
                                          and all(v["same_bytes_as_two_launches"] for v in per.values()))}
    except Exception as e:  # noqa: BLE001 - reported, never raised
        out["error"] = repr(e)[:400]
    finally:
        if saved is None:
            os.environ.pop("WB_IVF_FUSE_COARSE", None)
        else:
            os.environ["WB_IVF_FUSE_COARSE"] = saved
    return out


def parity_check(src, lo, hi, q, D, I, k, world, device, allowed=None):
    """Verify (D, I) = global top-k of queries q (all [*, .] device tensors, identical on every rank) against an fp64
    pass over THIS rank's regenerated rows; partial counts are summed over the ranks.  Returns a dict (rank-identical).
    allowed(s, e) -> (strict, loose) bool masks [e-s, nq] restricts the candidate set (IVF: rows of the probed lists;
    `strict` rows MUST be considered, returned rows must at least be `loose`)."""
    import torch
    import torch.distributed as dist
    nq = q.shape[0]
    q64 = q.double()
    D64 = D.double()
    kth = D64[:, k - 1]                              # k-th returned score per query
    above = torch.zeros(nq, dtype=torch.int64, device=device)        # rows whose exact score beats kth + band
    ret_above = torch.zeros(nq, dtype=torch.int64, device=device)    # ... of which are in the returned list
    found = torch.zeros(nq, dtype=torch.int64, device=device)        # returned ids located in my shard
    max_err = torch.zeros(1, dtype=torch.float64, device=device)
    rows_checked = 0
    outsiders = 0  # returned rows that are not candidates at all (IVF: not in a probed list)
    qcols = torch.arange(nq, device=device).unsqueeze(1).expand(nq, k)
    for s, e, x in src.chunks(lo, hi):
        s64 = x.double() @ q64.T                     # [m, nq] exact scores (fp64 accumulate of the fp32 inputs)
        beats = s64 > (kth + TIE_BAND).unsqueeze(0)
        loose = None
        if allowed is not None:
            strict, loose = allowed(s, e)
            beats &= strict
        above += beats.sum(dim=0)
        m = (I >= s) & (I < e)
        if bool(m.any()):
            ri, qi = (I[m] - s), qcols[m]
            ex = s64[ri, qi]
            if loose is not None:
                outsiders += int((~loose[ri, qi]).sum())
            max_err = torch.maximum(max_err, (ex - D64[m]).abs().max().reshape(1))
            ret_above.index_add_(0, qi, (ex > kth[qi] + TIE_BAND).long())
            found.index_add_(0, qi, torch.ones_like(qi))
        rows_checked += e - s
        del s64
    t_rows = torch.tensor([rows_checked, outsiders], dtype=torch.int64, device=device)
    ident = True
    if world > 1:
        for t in (above, ret_above, found, t_rows):
            dist.all_reduce(t)
        dist.all_reduce(max_err, op=dist.ReduceOp.MAX)
        for t in (I, D.view(torch.int32)):
            mx, mn = t.clone(), t.clone()
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            dist.all_reduce(mn, op=dist.ReduceOp.MIN)
            ident = ident and bool((mx == mn).all())
    sorted_ok = bool((D[:, 1:] <= D[:, :-1]).all())
    valid = (I >= 0).sum(dim=1)  # fewer than k only when the candidate set is smaller than k (-1 padding)
    uniq_ok = all(int(torch.unique(I[j][I[j] >= 0]).numel()) == int(valid[j]) for j in range(min(nq, 64)))
    violations = int((above - ret_above).clamp(min=0).sum()) + int((found != valid).sum()) + int(t_rows[1].item())
    return {"rows_checked": int(t_rows[0].item()), "queries": nq, "max_abs_err": float(max_err.item()),
            "violations": violations, "sorted": sorted_ok, "unique_ids": uniq_ok, "ranks_identical": ident,
            "score_tol": SCORE_TOL, "tie_band": TIE_BAND,
            "ok": bool(violations == 0 and float(max_err.item()) <= SCORE_TOL and sorted_ok and uniq_ok and ident)}


def run_ours(a):
    import torch
    import torch.distributed as dist
    from wise_b200 import _capi
    from wise_b200 import faiss_compat as faiss
    from wise_b200.sharded import ShardedIndex, shard_range

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != a.gpus:
        raise SystemExit(f"--gpus {a.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run --nproc-per-node {a.gpus}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: wise_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)
    L = _capi.lib()

    lo, hi = shard_range(a.rows, rank, world)
    src = RowSource(a.rows, a.dim, 2024, device)
    centres = src.centres
    index = faiss.IndexIDMap(faiss.IndexFlatIP(a.dim, device=local_rank))
    fill_index(index, src, lo, hi)
    assert index.ntotal == hi - lo
    sharded = ShardedIndex(index)
    L.wb_set_timing(index._h, 1)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_steps(nq, steps, warmup):
        """Device-resident queries; returns (ms per step [max over ranks], scan-kernel ms per step, launches,
        queries of the last step, its D, its I)."""
        qs = make_queries(centres, nq * (steps + warmup), a.dim, 2025, device).view(steps + warmup, nq, a.dim)
        for i in range(warmup):
            sharded.search_dev(qs[i], a.k)
        barrier()
        l0 = L.wb_launch_count(index._h) + (L.wb_exch_launch_count(sharded.exchange.h) if sharded.exchange else 0)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for i in range(steps):
            D, I = sharded.search_dev(qs[warmup + i], a.k)
        ev1.record()
        barrier()
        ms = ev0.elapsed_time(ev1) / steps
        launches = (L.wb_launch_count(index._h) + (L.wb_exch_launch_count(sharded.exchange.h) if sharded.exchange else 0)) - l0
        # per-launch scan durations OF THE TIMED REGION: event pairs recorded by the library around the
        # scan kernel(s) on the launching stream (ring of 128), read back after the region has ended
        buf = (ctypes.c_float * 128)()
        n = L.wb_scan_ms_history(index._h, buf, min(steps, 128))
        scan_ms = [buf[i] for i in range(n)]
        t = torch.tensor([ms], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), float(np.mean(scan_ms)), int(launches), qs[steps + warmup - 1], D, I

    def timed_e2e(nq, steps, warmup):
        """Public API, pinned host buffers in, numpy out; wall clock around synchronous calls."""
        q_all = make_queries(centres, nq * (steps + warmup), a.dim, 2026, device).view(steps + warmup, nq, a.dim).cpu()
        pinned = torch.empty((nq, a.dim), dtype=torch.float32).pin_memory()
        api = index if world == 1 else sharded  # the call a user makes: index.search(numpy, k)
        for i in range(warmup):
            pinned.copy_(q_all[i])
            api.search(pinned.numpy(), a.k)
        barrier()
        t0 = time.perf_counter()
        for i in range(steps):
            pinned.copy_(q_all[warmup + i])
            D, I = api.search(pinned.numpy(), a.k)
        barrier()
        dt = (time.perf_counter() - t0) / steps
        t = torch.tensor([dt], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) * 1e3, q_all[steps + warmup - 1], D, I

    def preroll(nq):
        """Untimed, all ranks: keep the GPU under the same load for ~0.6 s so that the clock samples bracket the
        timed region (the number of searches must be the same on every rank: the exchange is a collective)."""
        qpre = make_queries(centres, nq, a.dim, 2024, device)
        barrier()
        t_pre = time.perf_counter()
        for _ in range(3):
            sharded.search_dev(qpre, a.k)
        torch.cuda.synchronize()
        t3 = torch.tensor([(time.perf_counter() - t_pre) / 3], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t3, op=dist.ReduceOp.MAX)
        for _ in range(int(min(2000, max(1, 0.6 / max(float(t3.item()), 1e-5))))):
            sharded.search_dev(qpre, a.k)
        torch.cuda.synchronize()

    peaks_file = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_file):
        peaks = json.load(open(peaks_file))
        peak, peak_src = float(peaks["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy)"
    else:
        peaks, peak, peak_src = {}, HBM_FALLBACK_GBS, "fallback (B200_PROFILING.md)"
    local_bytes = (hi - lo) * a.dim * 4
    tf32_peak = {}

    def measure_tf32_peak():
        """TF32 tensor peak of THIS GPU with the library's own MMA shape: burst (one 5 ms launch) and sustained
        (~2 s back to back, second half timed: the power cap has settled)."""
        if not tf32_peak:
            torch.cuda.synchronize()
            time.sleep(1.0)  # the burst figure is taken first, on a GPU that has idled: not in the wake of a capped run
            tb, ts = ctypes.c_double(), ctypes.c_double()
            _capi.check(L.wb_tf32_peak(local_rank, 20000, 400, ctypes.byref(tb), ctypes.byref(ts)))
            tf32_peak.update({"burst": tb.value, "sustained": ts.value})
        return tf32_peak

    def roofline_of(batch, scan_ms):
        traffic = None
        tf = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tf):
            for t in json.load(open(tf)).get("captures", []):
                if t.get("rows") == hi - lo and t.get("dim") == a.dim and t.get("batch") == batch:
                    traffic = t.get("dram_bytes_per_launch")
        if batch < 5:   # K1: CUDA-core scan, HBM-bound; one pass of the row store per <= 8 queries
            passes = (batch + 7) // 8
            achieved = local_bytes * passes / (scan_ms * 1e-3) / 1e9
            return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": traffic, "kernel": "scan_topk_kernel", "bytes_per_launch": local_bytes,
                    "launch_ms": scan_ms / passes, "peak_source": peak_src}
        if batch <= 128:  # K2, one query block: ONE pass over the rows per search -> HBM is the roofline
            achieved = local_bytes / (scan_ms * 1e-3) / 1e9
            return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": traffic, "kernel": "gemm_topk_kernel (all epochs of a search, compactions included)",
                    "bytes_per_launch": local_bytes, "launch_ms": scan_ms, "peak_source": peak_src,
                    "note": "tcgen05 TF32 filter epochs + exact fp32 re-scoring of the candidates"}
        # K2 in 256-query blocks: tensor pipe; all epochs of a search timed together
        flop = 2.0 * batch * (hi - lo) * a.dim
        achieved = flop / (scan_ms * 1e-3) / 1e12
        pk = measure_tf32_peak()
        return {"bound": "tensor", "achieved": achieved, "peak": pk["sustained"], "unit": "TFLOP/s",
                "frac": achieved / pk["sustained"], "traffic": traffic,
                "kernel": "filter2_topk_kernel (all epochs of a search: 3xTF32 first epoch, one-term 256-query filter "
                          "epochs, exact fp32 re-scoring, compactions)",
                "flop_per_search": flop, "search_ms": scan_ms, "peak_burst": pk["burst"],
                "frac_of_burst": achieved / pk["burst"],
                "frac_of_bf16_sustained_half": (achieved / (float(peaks["bf16_tflops_sustained"]) / 2.0)
                                                if "bf16_tflops_sustained" in peaks else None),
                "peak_source": "wb_tf32_peak measured in this run on this GPU: back-to-back tcgen05.mma.cta_group::2."
                               "kind::tf32 M=256 N=256 K=8, no loads; sustained = 2nd half of 400 x 5 ms launches "
                               "(power cap settled), burst = best single launch",
                "note": "algorithmic flops 2*B*N*d; the filter epochs issue each flop once (one-term TF32)"}

    def dup_tie_check():
        """The planted duplicate: query = row 0 exactly; rows 0 and rows-1 hold the same vector (on different ranks when
        N > 1), so they tie bit for bit and must come back in insertion order."""
        qd = src.row0().view(1, a.dim).contiguous()
        D, I = sharded.search_dev(qd, a.k)
        torch.cuda.synchronize()
        Dh, Ih = D[0].cpu().numpy(), I[0].cpu().numpy()
        return {"ids": [int(Ih[0]), int(Ih[1])], "scores_equal_bits": bool(Dh[0].tobytes() == Dh[1].tobytes()),
                "ok": bool(Ih[0] == 0 and Ih[1] == a.rows - 1 and Dh[0].tobytes() == Dh[1].tobytes())}

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    preroll(a.batch)
    ms_step, scan_ms, launches, q_last, D_last, I_last = timed_steps(a.batch, a.steps, a.warmup)
    clocks = sampler.finish() if sampler else None
    if a.dump_outputs and rank == 0:  # every rank holds the same merged (D, I)
        dump_outputs(a.dump_outputs, D_last.cpu().numpy(), I_last.cpu().numpy())
    e2e_ms, q_e2e, D_e2e, I_e2e = timed_e2e(a.batch, a.steps, a.warmup)

    parity = None
    if not a.no_parity:
        parity = parity_check(src, lo, hi, q_last, D_last, I_last, a.k, world, device)
        # the last end-to-end step too (host API): its result must satisfy the same contract
        pe = parity_check(src, lo, hi, q_e2e.to(device), torch.from_numpy(D_e2e).to(device),
                          torch.from_numpy(I_e2e).to(device), a.k, world, device)
        parity["e2e_step"] = {k_: pe[k_] for k_ in ("max_abs_err", "violations", "ranks_identical", "ok")}
        parity["duplicate_tie"] = dup_tie_check()
        parity["ok"] = bool(parity["ok"] and pe["ok"] and parity["duplicate_tie"]["ok"])

    sweep = {}
    for b in [int(t) for t in a.sweep.split(",") if t.strip()]:
        m, s_ms, _, _, _, _ = timed_steps(b, max(3, a.steps // 3), 3)
        sweep[str(b)] = {"qps": b / (m / 1e3), "ms_per_step": m, "scan_ms": s_ms,
                         "scan_gbs": (hi - lo) * a.dim * 4 / (s_ms * 1e-3) / 1e9}

    sec_list = []
    if a.secondary == "auto":
        sec_list = [16, 1024] if (world == 1 and a.batch == 1) else []
    elif a.secondary != "none":
        sec_list = [int(t) for t in a.secondary.split(",") if t.strip()]
    secondary = {}
    for b in sec_list:
        steps_b = max(5, min(a.steps, 20 if b <= 128 else 10))
        smp = ClockSampler(local_rank) if rank == 0 else None
        if smp:
            smp.start()
        preroll(b)
        m, s_ms, ln, qb_last, Db, Ib = timed_steps(b, steps_b, 3)
        clk = smp.finish() if smp else None
        e_ms, _, _, _ = timed_e2e(b, steps_b, 3)
        entry = {"config": config_of(a, b), "value": b / (m / 1e3), "unit": "queries/s", "steps": steps_b, "warmup": 3,
                 "ms_per_step": m, "roofline": roofline_of(b, s_ms),
                 "e2e": {"value": b / (e_ms / 1e3), "unit": "queries/s", "ms_per_step": e_ms,
                         "h2d_bytes_per_step": b * a.dim * 4, "d2h_bytes_per_step": b * a.k * 12},
                 "gpu_launches": ln, "clocks": clk}
        if not a.no_parity:
            entry["parity_check"] = parity_check(src, lo, hi, qb_last, Db, Ib, a.k, world, device)
        secondary[f"batch{b}"] = entry
    if a.secondary == "auto" and world == 1 and a.batch == 1:
        secondary["ivf_one_query"] = ivf_one_query_secondary(device, a.k)

    if rank == 0:
        line = {
            "metric": METRIC, "value": a.batch / (ms_step / 1e3), "unit": "queries/s", "n_gpus": world, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": config_of(a),
            "shard": {"rows_per_gpu": hi - lo, "parallelism": f"row-shard x{world}",
                      "exchange": "NVLink peer-memory mailbox kernel (no NCCL on the search path)" if world > 1 else "none"},
            "roofline": roofline_of(a.batch, scan_ms),
            "e2e": {"value": a.batch / (e2e_ms / 1e3), "unit": "queries/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": a.batch * a.dim * 4, "d2h_bytes_per_step": a.batch * a.k * 12,
                    "d2h_how": "kernel stores into pinned host memory" if a.batch * a.k * 12 <= 65536
                               and os.environ.get("WB_DIRECT_RESULTS", "1") != "0" else "cudaMemcpyAsync"},
            "gpu_launches": launches, "clocks": clocks, "parity_check": parity,
        }
        if sweep:
            line["batch_sweep"] = sweep
        if secondary:
            line["secondary"] = secondary
        if world == 1 and not a.no_cpu_baseline:
            n_s = min(a.cpu_sample_rows, hi - lo)
            xs = np.empty((n_s, a.dim), np.float32)
            _capi.check(L.wb_export_rows(index._h, 0, n_s, _capi.ptr(xs), None, None))
            qh = make_queries(centres, a.batch, a.dim, 2027, device).cpu().numpy()
            qps1, t1, cores1, simd = cpu_restatement(xs, qh, a.k, a.rows, mt=False)
            qpsm, tm, coresm, _ = cpu_restatement(xs, qh, a.k, a.rows, mt=True)
            line["cpu_baseline"] = {
                "value": qps1, "unit": "queries/s", "cores": cores1, "kind": "port",
                "sample": f"first {n_s} of {a.rows} rows, {a.batch} queries, 3 reps, median {t1:.3f} s scaled x{a.rows / n_s:g}; "
                          f"oracle/cpu_flat.c orc_flat_search_seq ({simd}) = faiss's own threading (parallel over queries only)",
                "all_cores": {"value": qpsm, "cores": coresm, "median_s": tm, "fn": "orc_flat_search_mt"},
                "host": cpu_info()}
            if "batch1024" in secondary:  # faiss's BLAS path (n >= 20) on the host cores, bounded sample
                n_b = min(200_000, n_s)
                q1k = make_queries(centres, 1024, a.dim, 2028, device).cpu().numpy()
                qpsb, tb, th = cpu_blas(xs[:n_b], q1k, a.k, a.rows)
                secondary["batch1024"]["cpu_baseline"] = {
                    "value": qpsb, "unit": "queries/s", "cores": th, "kind": "port",
                    "sample": f"first {n_b} of {a.rows} rows, 1024 queries, 3 reps, median {tb:.3f} s scaled x{a.rows / n_b:g}; "
                              "oracle/cpu.py blas_flat_search = faiss exhaustive_inner_product_blas restated "
                              "(OpenBLAS sgemm tiles + partial selection)"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    global MIXED
    a = parse()
    MIXED = a.mixed
    # Keep stdout clean for the ONE JSON line: libraries (NCCL prints its version banner) get stderr.
    real_stdout = os.fdopen(os.dup(1), "w")
    sys.stdout.flush()
    os.dup2(2, 1)
    sys.stdout = real_stdout
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
    real_stdout.flush()


if __name__ == "__main__":
    main()
