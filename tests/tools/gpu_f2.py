"""Dev script (round 2): the 256-query SS filter kernel (gemm_ss.cuh) - TF32 peak microbenchmark and parity of large
batches against the oracle.
    python tests/tools/gpu_f2.py [all|peak|check]"""
import ctypes as C, os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import numpy as np
from oracle import oracle as O
from wise_b200 import faiss_compat as faiss, _capi
L = _capi.lib()


def stats(idx):
    a, b = C.c_int64(), C.c_int64(); L.wb_gemm_stats(idx._h, C.byref(a), C.byref(b)); return a.value, b.value


def peak():
    for iters, reps in ((2000, 4), (20000, 600)):
        tb, ts = C.c_double(), C.c_double()
        _capi.check(L.wb_tf32_peak(0, iters, reps, C.byref(tb), C.byref(ts)))
        print(f"tf32 peak: iters={iters} reps={reps}: burst {tb.value:.1f} TFLOP/s, sustained {ts.value:.1f} TFLOP/s", flush=True)


def check(n, d, nq, k, clustered=False):
    xb = O.clustered_unit(n, d, 64, 1) if clustered else O.unit_gaussian(n, d, 100)
    xq = O.clustered_unit(nq, d, 64, 2) if clustered else O.unit_gaussian(nq, d, 200)
    idx = faiss.IndexFlatIP(d); idx.add(xb)
    t = time.time(); D, I = idx.search(xq, k); dt = time.time() - t
    Dr, Ir = O.flat_search(xb, xq, k)
    err = np.abs(D - Dr)[Ir >= 0].max()
    try:
        r = O.compare_topk(D, I, Dr, Ir, band=4e-6)
    except AssertionError as e:
        r = "FAIL " + str(e)[:300]
    print(f"n={n} d={d} nq={nq} k={k}: {r} maxerr={err:.2e} {dt*1e3:.2f} ms gemm(epochs,fallbacks)={stats(idx)}", flush=True)


if __name__ == "__main__":
    what = sys.argv[1] if len(sys.argv) > 1 else "all"
    if what in ("all", "peak"):
        peak()
    if what in ("all", "check"):
        os.environ["WB_GEMM_FORCE"] = "1"
        for cfg in [(100000, 512, 200, 100), (131072, 768, 300, 100, True), (300000, 64, 1000, 10), (60000, 70, 129, 100, True),
                    (200000, 768, 1024, 100, True), (150001, 772, 257, 10)]:
            check(*cfg)
