// capi.cu - the C-ABI of libwiseb200.so (include/wise_b200.h): index handles, HBM row store,
// kernel launch configuration.  Host-side plumbing only; every flop happens in scan.cuh /
// merge.cuh / kmeans.cuh.  No CPU fallback: without a CUDA device every compute call fails.
#include <cuda_runtime.h>
#include <float.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <condition_variable>
#include <functional>
#include <memory>
#include <mutex>
#include <random>
#include <string>
#include <thread>
#include <type_traits>
#include <vector>

#include "../../include/wise_b200.h"
#include "csr.cuh"
#include "exchange.cuh"
#include "gemm.cuh"
#include "gemm_ss.cuh"
#include "ivf_lm.cuh"
#include "kmeans.cuh"
#include "merge.cuh"
#include "range.cuh"
#include "scan.cuh"
#include "tarstore.h"

using namespace wb;

// ---- errors ------------------------------------------------------------------------------
static thread_local std::string g_err;
static int fail(const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return 1;
}
#define CK(...) /* variadic: the call may hold template-argument commas */                                  \
    do {                                                                                                    \
        cudaError_t e_ = (__VA_ARGS__);                                                                     \
        if (e_ != cudaSuccess)                                                                              \
            return fail("%s failed: %s (%s:%d)", #__VA_ARGS__, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)
#define TRY(call)              \
    do {                       \
        int r_ = (call);       \
        if (r_ != 0) return r_; \
    } while (0)

// Opt `Kernel` in to `bytes` of dynamic shared memory, once per device and host thread.
template <auto Kernel>
static cudaError_t smem_optin(int bytes) {
    static thread_local bool done[64] = {};
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess || (dev < 64 && done[dev])) return e;
    e = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess && dev < 64) done[dev] = true;
    return e;
}

extern "C" const char* wb_last_error(void) { return g_err.c_str(); }
extern "C" const char* wb_version(void) { return "wise_b200 0.1 (sm_100a)"; }
extern "C" int wb_device_count(int* count) {
    CK(cudaGetDeviceCount(count));
    return 0;
}

// ---- owned device / pinned memory ----------------------------------------------------------
struct DevFree {
    void operator()(void* p) const { cudaFree(p); }
};
struct HostFree {
    void operator()(void* p) const { cudaFreeHost(p); }
};
template <class T>
using DevPtr = std::unique_ptr<T, DevFree>;
template <class T>
using PinPtr = std::unique_ptr<T, HostFree>;
struct EventDestroy {
    void operator()(cudaEvent_t e) const { cudaEventDestroy(e); }
};
using EventPtr = std::unique_ptr<CUevent_st, EventDestroy>;

// cudaMalloc into an owner; `out` keeps what it held when the allocation fails
template <class T>
static cudaError_t dev_alloc(DevPtr<T>* out, size_t bytes) {
    T* p = nullptr;
    const cudaError_t e = cudaMalloc(&p, bytes);
    if (e == cudaSuccess) out->reset(p);
    return e;
}

// Grow-only scratch (at least 64 KB, contents not kept when it grows) in device memory, or, when `Pinned`, in pinned
// host memory: a copy between pageable memory and the device is staged by the driver and blocks the call; small
// transfers go through a pinned buffer instead and stay asynchronous.
template <bool Pinned>
struct GrowBuf {
    std::unique_ptr<void, std::conditional_t<Pinned, HostFree, DevFree>> mem;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return 0;
        mem.reset();
        cap = 0;
        const size_t want = std::max(bytes, (size_t)1 << 16);
        void* p = nullptr;
        if constexpr (Pinned)
            CK(cudaHostAlloc(&p, want, cudaHostAllocMapped | cudaHostAllocPortable));  // kernels may write into it (UVA)
        else
            CK(cudaMalloc(&p, want));
        mem.reset(p);
        cap = want;
        return 0;
    }
    void* get() const { return mem.get(); }
    template <class T>
    T* as() const { return reinterpret_cast<T*>(mem.get()); }
};
using DevBuf = GrowBuf<false>;
using PinBuf = GrowBuf<true>;

struct wb_index {
    int device = 0;
    int d = 0, ld = 0;
    bool ivf = false;
    int64_t nlist = 0;
    bool trained = true;
    bool spherical = false;  // k-means: L2-renormalise the centroids after every update (faiss cp.spherical)
    cudaStream_t stream = nullptr;
    // row store (insertion order)
    DevPtr<float> rows;
    DevPtr<int64_t> ids;
    DevPtr<int32_t> assign;  // IVF: list of each row
    int64_t n = 0, cap = 0;
    DevPtr<float> norm2_max;  // device scalar: max |row|^2 over everything ever added (K2 filter margin)
    // int8 image of a flat store (the filter rows of 1-2 query scans, DESIGN.md "K1"): row r is the header and int8 codes
    // of rows[r] (int8_image_kernel), stride img_row_bytes(ld); img_cap rows allocated.  Built lazily by the first search
    // that uses it:
    // rows [img_n, n) are converted before such a search.  Rows reach the store only through add_common (appended at
    // n), which keeps img_n <= n right; anything that rewrites or removes stored rows must reset img_n to 0.
    DevPtr<uint8_t> img;
    int64_t img_n = 0, img_cap = 0;
    cudaEvent_t img_ev = nullptr;    // recorded after the last conversion, on img_st: searches on other streams wait
    cudaStream_t img_st = nullptr;
    DevPtr<unsigned long long> img_rescored;  // device counter: (row, query) pairs the int8 filter re-scored
    int64_t img_searches = 0;                 // searches served by the image
    // IVF quantizer + inverted lists.  `ids` always stay in INSERTION order.  After a (re)grouping the rows are
    // stored list by list (insertion order kept inside a list): row_pos[row] is then the insertion position of a
    // storage row - the tie rule and the id lookup - and slot_row is null.  When the transient second copy of the rows
    // does not fit, the rows stay where they are and slot_row[CSR slot] is the storage row of each list slot.
    DevPtr<float> centroids;   // [nlist, ld]
    DevPtr<uint32_t> slot_row; // [n] or null (slot == storage row)
    DevPtr<uint32_t> row_pos;  // [map_cap] or null (storage row == insertion position)
    int64_t map_cap = 0;
    DevPtr<int64_t> list_off;  // [nlist + 1]
    bool csr_dirty = true;
    // scratch
    DevBuf parts, qbuf, dbuf, ibuf, pD, pI, xbuf, idbuf, misc, kperm, koff, gimg, gimg2, gkeys, gstate, gmargin, eD, eI, tailcnt, ccnt, ctot, lmA, lmB, lmC, lmD, lmE, lmF, lmG;
    PinBuf pin_q, pin_o;  // pinned staging of small query / result transfers of the host API
    static constexpr int kAddSlots = 8;   // wb_add_with_ids_pinned: one event per in-flight pinned buffer
    cudaEvent_t add_ev[kAddSlots] = {};
    bool add_pending[kAddSlots] = {};
    int64_t gemm_launches = 0, gemm_fallbacks = 0;
    DevBuf rpool, rqid, rgrp, rstate, roff, rrun;  // range search: hit pool, query tags, sort buffer, counters, lims, runs
    DevBuf phase;               // WB_PHASE_TS=1: per-CTA phase stamps of the last fused-tail scan launch (diagnostics)
    DevBuf ckeys;               // fused coarse quantizer: ordered centroid scores of the queries of one launch
    bool coop_ok = false;       // the device takes cooperative launches (fused coarse quantizer, coarse.cuh)
    int64_t coarse_fused = 0;   // IVF searches served by ONE launch (coarse quantizer inside the list scan)
    // device properties
    int sm_count = 148;
    int smem_max = 0;
    // accounting
    int64_t launches = 0;
    bool timing = false;
    static constexpr int kEvRing = 128;  // event pairs of the most recent timed scan launches
    cudaEvent_t ev0[kEvRing] = {}, ev1[kEvRing] = {};
    int64_t ev_count = 0;

    // The caller has made `device` current.  The members free the memory once the stream is gone.
    ~wb_index() {
        if (!stream) return;
        cudaStreamSynchronize(stream);
        for (cudaEvent_t e : add_ev)
            if (e) cudaEventDestroy(e);
        if (img_ev) cudaEventDestroy(img_ev);
        for (int i = 0; i < kEvRing; ++i) {
            if (ev0[i]) cudaEventDestroy(ev0[i]);
            if (ev1[i]) cudaEventDestroy(ev1[i]);
        }
        cudaStreamDestroy(stream);
    }
};

static int set_dev(const wb_index* h) {
    CK(cudaSetDevice(h->device));
    return 0;
}

// ---- construction --------------------------------------------------------------------------
static int create_common(int d, int device, bool ivf, int64_t nlist, wb_index** out) {
    if (!out) return fail("out is NULL");
    *out = nullptr;
    if (d <= 0 || d > 65536) return fail("invalid dimension %d", d);
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail("no CUDA device available (%s): wise_b200 has no CPU fallback", cudaGetErrorString(e));
    if (device < 0 || device >= ndev) return fail("device %d out of range (%d devices)", device, ndev);
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return fail("device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
    std::unique_ptr<wb_index> h(new wb_index());
    h->device = device;
    h->d = d;
    h->ld = (d + 3) & ~3;
    h->ivf = ivf;
    h->nlist = nlist;
    h->trained = !ivf;
    h->sm_count = prop.multiProcessorCount;
    h->smem_max = (int)prop.sharedMemPerBlockOptin;
    h->coop_ok = prop.cooperativeLaunch != 0;
    CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    for (int i = 0; i < wb_index::kEvRing; ++i) {
        CK(cudaEventCreate(&h->ev0[i]));
        CK(cudaEventCreate(&h->ev1[i]));
    }
    CK(dev_alloc(&h->norm2_max, sizeof(float)));
    CK(cudaMemsetAsync(h->norm2_max.get(), 0, sizeof(float), h->stream));
    if (ivf) {
        CK(dev_alloc(&h->centroids, (size_t)nlist * h->ld * sizeof(float)));
        CK(cudaMemsetAsync(h->centroids.get(), 0, (size_t)nlist * h->ld * sizeof(float), h->stream));
        CK(dev_alloc(&h->list_off, (size_t)(nlist + 1) * sizeof(int64_t)));
        CK(cudaMemsetAsync(h->list_off.get(), 0, (size_t)(nlist + 1) * sizeof(int64_t), h->stream));
    }
    CK(cudaStreamSynchronize(h->stream));  // the zero-fills above must not race a first add on another stream
    *out = h.release();
    return 0;
}

extern "C" int wb_flat_create(int d, int device, wb_index** out) { return create_common(d, device, false, 0, out); }
extern "C" int wb_ivf_create(int d, int64_t nlist, int device, wb_index** out) {
    if (nlist <= 0 || nlist > (int64_t)1 << 30) return fail("invalid nlist %lld", (long long)nlist);
    return create_common(d, device, true, nlist, out);
}

extern "C" int wb_free(wb_index* h) {
    if (!h) return 0;
    cudaSetDevice(h->device);
    delete h;
    return 0;
}

extern "C" int64_t wb_dim(const wb_index* h) { return h ? h->d : -1; }
extern "C" int64_t wb_ntotal(const wb_index* h) { return h ? h->n : -1; }
extern "C" int wb_is_trained(const wb_index* h) { return h && h->trained; }
extern "C" int64_t wb_nlist(const wb_index* h) { return h ? h->nlist : -1; }
extern "C" int wb_is_ivf(const wb_index* h) { return h && h->ivf; }
extern "C" int64_t wb_launch_count(const wb_index* h) { return h ? h->launches : -1; }
extern "C" int64_t wb_ivf_fused_searches(const wb_index* h) { return h ? h->coarse_fused : -1; }
constexpr size_t kPhaseCtas = 1024;  // phase stamps: CTAs of query group 0 (the kernel ignores blockIdx.x >= 1024)
extern "C" int wb_phase_stamps(wb_index* h, uint64_t* out_host, int ctas) {
    if (!h || !out_host) return fail("NULL argument");
    if (!h->phase.get()) return fail("no phase stamps: set WB_PHASE_TS=1 before the search");
    if (ctas < 1 || (size_t)ctas > kPhaseCtas) return fail("ctas out of range");
    TRY(set_dev(h));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(out_host, h->phase.get(), (size_t)ctas * 16 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    return 0;
}
extern "C" int wb_gemm_stats(const wb_index* h, int64_t* epochs, int64_t* fallbacks) {
    if (!h) return fail("NULL index");
    if (epochs) *epochs = h->gemm_launches;
    if (fallbacks) *fallbacks = h->gemm_fallbacks;
    return 0;
}
extern "C" int wb_flat_bf16_stats(wb_index* h, int64_t* searches, int64_t* rescored) {
    if (!h) return fail("NULL index");
    unsigned long long r = 0;
    if (h->img_rescored) {
        TRY(set_dev(h));
        CK(cudaDeviceSynchronize());  // launches on any stream add to the counter
        CK(cudaMemcpy(&r, h->img_rescored.get(), sizeof r, cudaMemcpyDeviceToHost));
    }
    if (searches) *searches = h->img_searches;
    if (rescored) *rescored = (int64_t)r;
    return 0;
}
extern "C" int64_t wb_flat_image_bytes(const wb_index* h) {
    return h ? h->img_cap * img_row_bytes(h->ld) : 0;
}
extern "C" int wb_set_timing(wb_index* h, int on) {
    if (!h) return fail("NULL index");
    h->timing = on != 0;
    h->ev_count = 0;
    return 0;
}
// The event pair around one timed scan, in the ring slot that wb_last_scan_ms / wb_scan_ms_history read.
static int timing_begin(wb_index* h, bool on, cudaStream_t st) {
    if (on) CK(cudaEventRecord(h->ev0[h->ev_count % wb_index::kEvRing], st));
    return 0;
}
static int timing_end(wb_index* h, bool on, cudaStream_t st) {
    if (!on) return 0;
    CK(cudaEventRecord(h->ev1[h->ev_count % wb_index::kEvRing], st));
    h->ev_count++;
    return 0;
}
static float scan_ms_at(wb_index* h, int64_t i) {
    const int s = (int)(i % wb_index::kEvRing);
    if (cudaEventSynchronize(h->ev1[s]) != cudaSuccess) return -1.f;
    float ms = -1.f;
    if (cudaEventElapsedTime(&ms, h->ev0[s], h->ev1[s]) != cudaSuccess) return -1.f;
    return ms;
}
extern "C" float wb_last_scan_ms(wb_index* h) {
    if (!h || h->ev_count == 0) return -1.f;
    if (cudaSetDevice(h->device) != cudaSuccess) return -1.f;
    return scan_ms_at(h, h->ev_count - 1);
}
extern "C" int wb_scan_ms_history(wb_index* h, float* out_ms, int cap) {
    if (!h || !out_ms || cap <= 0) return 0;
    if (cudaSetDevice(h->device) != cudaSuccess) return 0;
    const int64_t n = std::min<int64_t>(std::min<int64_t>(h->ev_count, wb_index::kEvRing), cap);
    for (int64_t i = 0; i < n; ++i) out_ms[i] = scan_ms_at(h, h->ev_count - n + i);
    return (int)n;
}
extern "C" int wb_storage(wb_index* h, void** rows_dev, int64_t* ld) {
    if (!h) return fail("NULL index");
    if (rows_dev) *rows_dev = h->rows.get();
    if (ld) *ld = h->ld;
    return 0;
}

// ---- capacity ------------------------------------------------------------------------------
static int ensure_capacity(wb_index* h, int64_t need) {
    if (need <= h->cap) return 0;
    if (need >= (int64_t)0xFFFFFFFEll) return fail("an index shard is limited to 2^32-2 rows per GPU");
    int64_t newcap = std::max<int64_t>(need, std::max<int64_t>(1024, h->cap + h->cap / 2));
    // everything is allocated and copied before the handle changes: a failure leaves it as it was
    DevPtr<float> nrows;
    DevPtr<int64_t> nids;
    DevPtr<int32_t> nas;
    DevPtr<uint32_t> npos;
    const bool grow_pos = h->row_pos && newcap > h->map_cap;
    CK(dev_alloc(&nrows, (size_t)newcap * h->ld * sizeof(float)));
    CK(dev_alloc(&nids, (size_t)newcap * sizeof(int64_t)));
    if (h->ivf) CK(dev_alloc(&nas, (size_t)newcap * sizeof(int32_t)));
    if (grow_pos) CK(dev_alloc(&npos, (size_t)newcap * sizeof(uint32_t)));
    if (h->n > 0) {
        if (grow_pos)
            CK(cudaMemcpyAsync(npos.get(), h->row_pos.get(), (size_t)h->n * sizeof(uint32_t), cudaMemcpyDeviceToDevice, h->stream));
        CK(cudaMemcpyAsync(nrows.get(), h->rows.get(), (size_t)h->n * h->ld * sizeof(float), cudaMemcpyDeviceToDevice, h->stream));
        CK(cudaMemcpyAsync(nids.get(), h->ids.get(), (size_t)h->n * sizeof(int64_t), cudaMemcpyDeviceToDevice, h->stream));
        if (h->ivf)
            CK(cudaMemcpyAsync(nas.get(), h->assign.get(), (size_t)h->n * sizeof(int32_t), cudaMemcpyDeviceToDevice, h->stream));
    }
    CK(cudaStreamSynchronize(h->stream));
    if (grow_pos) {
        h->row_pos = std::move(npos);
        h->map_cap = newcap;
    }
    h->rows = std::move(nrows);
    h->ids = std::move(nids);
    h->assign = std::move(nas);
    h->cap = newcap;
    return 0;
}

extern "C" int wb_reserve(wb_index* h, int64_t n) {
    if (!h) return fail("NULL index");
    TRY(set_dev(h));
    return ensure_capacity(h, n);
}

extern "C" int wb_capacity(wb_index* h, int64_t* cap_rows, int64_t* free_bytes) {
    if (!h || !cap_rows || !free_bytes) return fail("NULL argument");
    TRY(set_dev(h));
    size_t free_b = 0, total_b = 0;
    CK(cudaMemGetInfo(&free_b, &total_b));
    *cap_rows = h->cap;
    *free_bytes = (int64_t)free_b;
    return 0;
}

// ---- scan launch ---------------------------------------------------------------------------
struct ScanCfg {
    int NQ, RW, P, ck, nchunks, stages, single_copy;
    size_t smem;
};

static int env_int(const char* name, int dflt) {
    const char* v = getenv(name);
    return v && *v ? atoi(v) : dflt;
}

// Pick queries-per-CTA, rows-per-warp and ring depth so that everything fits the 227 KB of
// shared memory: [ring | queries | top-k lists + queues | barriers].  `img`: the ring holds rows of the int8 image
// (ck = the image's row length img_row_bytes(ld), in floats); whole-row stages only.
// Measured on B200 (profiles/r01_scan_sweep.md): one bulk copy engine request costs the producer
// ~27 cycles, so stages hold WHOLE rows - a flat row group is then one contiguous copy (7.2 TB/s);
// chunked stages (one 1 KB copy per row and chunk) top out at 4.0 TB/s and are only the fallback
// for rows too wide for two whole-row stages.
static int plan_scan(const wb_index* h, int64_t nq, int k, bool gather, int nprobe, ScanCfg* c, bool img = false) {
    constexpr int kMaxStages = 8;
    const int ld = h->ld;
    int NQ = gather ? 1 : (nq >= 8 ? 8 : nq > 2 ? 4 : nq > 1 ? 2 : 1);
    const int P = pow2_ceil(k + kMinQueue);
    const int np = gather ? nprobe : 0;
    const int rowf = img ? img_row_bytes(ld) / 4 : ld;  // ring floats per row
    for (; NQ >= 1; NQ >>= 1) {
        for (int RW = kMaxRowsPerWarp; RW >= 1; RW >>= 1) {  // whole-row stages
            const int gr = kConsumerWarps * RW;
            const size_t fixed = scan_smem_layout(NQ, ld, P, rowf, 0, np, gr, img).total;
            const size_t stage_bytes = (size_t)gr * rowf * 4;
            if (fixed + 2 * stage_bytes + 64 > (size_t)h->smem_max) continue;
            if (stage_bytes >= (1u << 20)) continue;  // mbarrier tx-count limit
            const int stages = (int)std::min<size_t>(kMaxStages, ((size_t)h->smem_max - fixed - 64) / (stage_bytes + 24));
            *c = ScanCfg{NQ, RW, P, rowf, 1, stages, gather ? 0 : 1, 0};
            c->smem = scan_smem_layout(NQ, ld, P, rowf, stages, np, gr, img).total;
            return 0;
        }
        if (img) continue;
        const int RW = kMaxRowsPerWarp;  // chunked fallback: very wide rows
        const int gr = kConsumerWarps * RW;
        for (int ck = std::min(1024, ld) & ~3; ck >= 32; ck = (ck / 2) & ~3) {
            const size_t fixed = scan_smem_layout(NQ, ld, P, ck, 0, np, gr).total;
            const size_t stage_bytes = (size_t)gr * ck * 4;
            if (fixed + 2 * stage_bytes + 64 > (size_t)h->smem_max) continue;
            const int stages = (int)std::min<size_t>(kMaxStages, ((size_t)h->smem_max - fixed - 64) / (stage_bytes + 24));
            *c = ScanCfg{NQ, RW, P, ck, (ld + ck - 1) / ck, stages, 0, 0};
            c->smem = scan_smem_layout(NQ, ld, P, ck, stages, np, gr).total;
            return 0;
        }
    }
    return fail("scan does not fit shared memory (d=%d, k=%d)", h->d, k);
}

constexpr int kRangeStage = 256;  // staged hits per query and CTA in the range scan (P of its shared lists)

// The plan plan_scan makes for a search of `nq` queries (k = 0: a range search), so that tests can choose shapes by the
// path they take: out = {NQ, RW, ck, nchunks, stages}.
extern "C" int wb_scan_plan(wb_index* h, int64_t nq, int64_t k, int gather, int64_t nprobe, int out[5]) {
    if (!h || !out) return fail("NULL argument");
    if (nq < 1 || k < 0 || k > WB_MAX_K || nprobe < 0 || nprobe > WB_MAX_K) return fail("bad scan plan arguments");
    ScanCfg c;
    TRY(plan_scan(h, nq, k == 0 ? kRangeStage - kMinQueue : (int)k, gather != 0, (int)nprobe, &c));
    const int v[5] = {c.NQ, c.RW, c.ck, c.nchunks, c.stages};
    for (int i = 0; i < 5; ++i) out[i] = v[i];
    return 0;
}

constexpr int kScanSmemOptin = 232448;  // the scan kernels opt in to the most a block may have (227 KB)

// Opt `Kernel` in to the scans' shared memory, launch it on `st` and check the launch.
template <auto Kernel, class... Args>
static int launch(dim3 grid, int block, size_t smem, cudaStream_t st, const Args&... args) {
    CK(smem_optin<Kernel>(kScanSmemOptin));
    Kernel<<<grid, block, smem, st>>>(args...);
    CK(cudaGetLastError());
    return 0;
}

template <int V>
using Int = std::integral_constant<int, V>;

// fn(Int<RW>) for the rows per warp of a scan plan: plan_scan picks 4, 2 or 1; anything else runs as 1.
template <class Fn>
static auto with_rw(int RW, Fn&& fn) {
    switch (RW) {
        case 4: return fn(Int<4>{});
        case 2: return fn(Int<2>{});
        default: return fn(Int<1>{});
    }
}

// fn(Int<NQ>, Int<RW>, std::bool_constant<GATHER>) for the scan kernel instance of a plan: NQ = 1, 2, 4 or 8 queries per
// CTA over contiguous rows, or one query per CTA over the rows of its probed lists (GATHER).
template <class Fn>
static int with_scan_instance(int NQ, int RW, bool gather, Fn&& fn) {
    auto rw = [&](auto nq, auto g) -> int {
        if (RW != 4 && RW != 2 && RW != 1) return fail("bad RW %d", RW);
        return with_rw(RW, [&](auto rw) { return fn(nq, rw, g); });
    };
    if (gather) return rw(Int<1>{}, std::true_type{});
    switch (NQ) {
        case 1: return rw(Int<1>{}, std::false_type{});
        case 2: return rw(Int<2>{}, std::false_type{});
        case 4: return rw(Int<4>{}, std::false_type{});
        case 8: return rw(Int<8>{}, std::false_type{});
    }
    return fail("bad NQ %d", NQ);
}

static void apply_scan_cfg(const ScanCfg& c, ScanParams& p) {
    p.P = c.P;
    p.ck = c.ck;
    p.nchunks = c.nchunks;
    p.stages = c.stages;
    p.single_copy = c.single_copy;
    p.rw = c.RW;
    p.rank_sort = c.P <= kConsumerThreads;  // measured: slower than bitonic at P = 512
}

// Cooperative launch of the gather kernel (fused coarse quantizer: the CTAs of a query group meet at a barrier, so all
// of them must be resident - the cooperative launch guarantees it or fails).
static cudaError_t launch_scan_coop(const ScanCfg& c, ScanParams& p, dim3 grid, cudaStream_t st) {
    apply_scan_cfg(c, p);
    return with_rw(c.RW, [&](auto RW) {
        const cudaError_t e = smem_optin<scan_topk_kernel<1, RW, true>>(kScanSmemOptin);
        if (e != cudaSuccess) return e;
        void* args[] = {&p};
        return cudaLaunchCooperativeKernel(reinterpret_cast<const void*>(scan_topk_kernel<1, RW, true>), grid,
                                           dim3(kScanThreads), args, c.smem, st);
    });
}

// p.img set: the int8 filter instance (flat, NQ <= 2)
static int launch_scan(const ScanCfg& c, bool gather, ScanParams& p, dim3 grid, cudaStream_t st) {
    apply_scan_cfg(c, p);
    return with_scan_instance(c.NQ, c.RW, gather, [&](auto NQ, auto RW, auto G) {
        if constexpr (!G && NQ <= 2) {
            if (p.img) return launch<scan_topk_kernel<NQ, RW, false, true>>(grid, kScanThreads, c.smem, st, p);
        }
        if (p.img) return fail("no int8 filter scan for NQ %d", (int)NQ);
        return launch<scan_topk_kernel<NQ, RW, G>>(grid, kScanThreads, c.smem, st, p);
    });
}

// Sort-buffer size of the merge: everything at once when it is small, else k + a 2048-entry queue.
static int merge_buffer_entries(int k, int64_t nparts, int nthreads = kMergeThreads) {
    const int64_t M = nparts * (int64_t)k;
    const int full = pow2_ceil(k + 2 * nthreads);
    if (M <= full) return std::max(2, pow2_ceil((int)std::max<int64_t>(M, k)));
    return full;
}

static int launch_merge_keys(wb_index* h, int64_t nq, int k, int64_t nparts, const uint64_t* keys, const int64_t* ids,
                             float* D, int64_t* I, cudaStream_t st) {
    MergeParams m{};
    m.nq = nq;
    m.k = k;
    m.nparts = nparts;
    m.S = merge_buffer_entries(k, nparts);
    m.keys = keys;
    m.ids = ids;
    m.D = D;
    m.I = I;
    CK(smem_optin<merge_topk_kernel<true>>(8192 * 8));
    merge_topk_kernel<true><<<(unsigned)nq, kMergeThreads, (size_t)m.S * 8, st>>>(m);
    CK(cudaGetLastError());
    h->launches++;
    return 0;
}

// Arrival counters of the fused tail merge: zero between launches (the last CTA of a group resets its own).
constexpr int64_t kMaxGridY = 32768;
static int ensure_tail_counters(wb_index* h, cudaStream_t st) {
    if (h->tailcnt.get()) return 0;
    // [arrivals | row-group dispensers | coarse-barrier arrivals]
    TRY(h->tailcnt.ensure((size_t)3 * kMaxGridY * sizeof(unsigned int)));
    CK(cudaMemsetAsync(h->tailcnt.get(), 0, (size_t)3 * kMaxGridY * sizeof(unsigned int), st));
    return 0;
}

// Can the scan kernel's last CTA run the merge (and the multi-GPU exchange) itself?  The sort buffer and the staged
// local winners must fit the (then idle) ring.
static bool tail_fusable(const ScanCfg& c, int k, int64_t nparts, int world, int* S_merge, int* heads_bytes) {
    *S_merge = 0;
    *heads_bytes = 0;
    const size_t ring_bytes = (size_t)c.stages * kConsumerWarps * c.RW * c.ck * 4;
    const int S = std::max(merge_buffer_entries(k, nparts, kConsumerThreads),
                           world > 1 ? merge_buffer_entries(k, world, kConsumerThreads) : 2);
    if ((size_t)S * 8 + (size_t)k * 12 + 64 > ring_bytes) return false;
    *S_merge = S;
    // merge through the heads of the sorted lists first (block_merge_heads, merge.cuh); the sort-based merge stays
    // behind it as the fallback, so both regions must fit
    if (nparts <= 256) {
        const HeadsPlan a = heads_plan(k, (int)nparts);
        if (a.ok && std::max(a.bytes, (size_t)S * 8) + (size_t)k * 12 + 64 <= ring_bytes) *heads_bytes = (int)a.bytes;
    }
    return true;
}

static void set_tail(ScanParams& p, wb_index* h, const ScanCfg& c, int S_merge, int heads_bytes, const int64_t* ids, float* D,
                     int64_t* I, int k, const ExchParams* ex) {
    p.fuse_tail = 1;
    p.S_merge = S_merge;
    p.heads_bytes = heads_bytes;
    p.phase_ts = nullptr;
    if (env_int("WB_PHASE_TS", 0) && h->phase.ensure(kPhaseCtas * 16 * sizeof(unsigned long long)) == 0)
        p.phase_ts = h->phase.as<unsigned long long>();
    p.tail_count = h->tailcnt.as<unsigned int>();
    p.group_count = c.nchunks == 1 ? h->tailcnt.as<unsigned int>() + kMaxGridY : nullptr;
    p.ids = ids;
    p.D = D;
    p.I = I;
    p.exchange = 0;
    if (ex) {
        p.exchange = 1;
        p.exch = *ex;
        p.exch.S = merge_buffer_entries(k, ex->world, kConsumerThreads);
    }
}

// The rows a filtered search may return (dense filter path, DESIGN.md "Filtered search"): bit p of allow[p / 32] is
// set for a selected insertion position p, and sel[t] counts the selected positions in [0, t * kGemmBM) (host).
struct RowMask {
    const uint32_t* allow;
    const int64_t* sel;
};

// CTAs per query group of a scan over `nrows` contiguous rows: enough to fill the SMs (twice over when there are
// several query groups), at most one per row group.
static int64_t flat_ctas(const wb_index* h, const ScanCfg& c, int64_t nrows, int64_t nq) {
    const int gr = kConsumerWarps * c.RW;
    const int64_t ngroups = (nrows + gr - 1) / gr;
    const int64_t qgroups = (nq + c.NQ - 1) / c.NQ;
    const int64_t S = std::min<int64_t>(std::max<int64_t>(ngroups, 1),
                                        std::max<int64_t>(1, ((int64_t)h->sm_count * (qgroups > 1 ? 2 : 1) + qgroups - 1) / qgroups));
    return std::min<int64_t>(S, (int64_t)h->sm_count);
}

// CTAs per query of a list scan: the SMs shared out among the queries.
static int64_t ivf_ctas(const wb_index* h, int64_t nq) {
    return nq >= h->sm_count ? 1 : std::max<int64_t>(1, (int64_t)h->sm_count / nq);
}

// The top-k scan launches of `nq` queries (K1, or K5 when `gather`: the probe table is in h->pI), one per <= kMaxGridY
// query groups of c.NQ, with p.nparts CTAs per group; then the K3 merge of the per-CTA lists unless p.fuse_tail has
// the kernel's last CTA merge them.  *exchanged tells the caller whether (D, I) already hold the GLOBAL result
// (written to ex->D / ex->I).
static int run_scan_groups(wb_index* h, const ScanCfg& c, bool gather, ScanParams& p, int64_t nq, const float* q_ld,
                           const int64_t* ids, float* D, int64_t* I, cudaStream_t st, bool timed, const ExchParams* ex,
                           bool* exchanged) {
    const int64_t qgroups = (nq + c.NQ - 1) / c.NQ;
    TRY(timing_begin(h, timed && h->timing, st));
    for (int64_t g0 = 0; g0 < qgroups; g0 += kMaxGridY) {
        const int64_t gy = std::min(kMaxGridY, qgroups - g0);
        const int64_t qoff = g0 * c.NQ;
        p.queries = q_ld + (size_t)qoff * h->ld;
        p.nq = (int)std::min<int64_t>(nq - qoff, gy * c.NQ);
        if (gather) p.probes = h->pI.as<int64_t>() + (size_t)qoff * p.nprobe;
        p.parts = h->parts.as<uint64_t>() + (size_t)qoff * p.nparts * p.k;
        if (p.fuse_tail) {  // the tail indexes (D, I) and the mailboxes by the query number inside this launch
            p.D = (ex ? ex->D : D) + (size_t)qoff * p.k;
            p.I = (ex ? ex->I : I) + (size_t)qoff * p.k;
            if (ex && qoff != 0) return fail("exchange-fused scans take at most %lld query groups", (long long)kMaxGridY);
        }
        TRY(launch_scan(c, gather, p, dim3((unsigned)p.nparts, (unsigned)gy), st));
        h->launches++;
    }
    TRY(timing_end(h, timed && h->timing, st));
    if (p.fuse_tail) {
        if (ex && exchanged) *exchanged = true;
        return 0;
    }
    return launch_merge_keys(h, nq, p.k, p.nparts, h->parts.as<uint64_t>(), ids, D, I, st);
}

constexpr size_t kMemReserve = (size_t)1 << 30;  // free device memory an optional copy of the rows must leave

// The int8 filter pays a fixed cost per CTA - its first few hundred rows are re-scored while the threshold is still
// loose, 32 latency-bound rows at a time - and saves three quarters of the bytes of every row.  Measured on a B200
// (1000 W, 1965 MHz max SM clock; profiles/r05), one query over N x 768, image against the fp32 scan: 0.5M rows (3378
// per SM) 0.285 against 0.242 ms, 1M (6757 per SM) 0.418 against 0.449 ms, 1.5M 0.538 against 0.653 ms.  The cutoff
// sits just below the smallest store measured to gain.  Batches of 3-4 queries were slower on the bf16 image that
// preceded this one (four queries double the shared-memory reads per byte), so the image serves 1-2 queries.
constexpr int64_t kImageMinRowsPerSm = 6144;
constexpr int64_t kImageMaxQueries = 2;

// Bring the int8 image of a flat store up to date for a search on `st` (rows [img_n, n) converted on `st`).  *ok =
// false when the image does not fit: it is allocated at the store's capacity only if that leaves kMemReserve free
// (else the index keeps no image); a failed allocation leaves the handle as it was.
static int ensure_image(wb_index* h, cudaStream_t st, bool* ok) {
    *ok = false;
    if (h->n == 0) return 0;
    const int rb = img_row_bytes(h->ld);
    if (h->n > h->img_cap) {
        const size_t bytes = (size_t)h->cap * rb;
        size_t free_b = 0, total_b = 0;
        CK(cudaMemGetInfo(&free_b, &total_b));
        if (free_b < bytes + kMemReserve) {
            h->img.reset();
            h->img_cap = h->img_n = 0;
            return 0;
        }
        DevPtr<uint8_t> img;
        if (dev_alloc(&img, bytes) != cudaSuccess) {
            cudaGetLastError();  // (clear the allocation error: the next launch check would report it)
            return 0;
        }
        h->img = std::move(img);
        h->img_cap = h->cap;
        h->img_n = 0;
    }
    if (!h->img_rescored) {
        DevPtr<unsigned long long> cnt;
        CK(dev_alloc(&cnt, sizeof(unsigned long long)));
        CK(cudaMemsetAsync(cnt.get(), 0, sizeof(unsigned long long), st));
        h->img_rescored = std::move(cnt);
    }
    if (!h->img_ev) CK(cudaEventCreateWithFlags(&h->img_ev, cudaEventDisableTiming));
    if (h->img_n < h->n) {
        const int64_t m = h->n - h->img_n;  // one warp per row
        int8_image_kernel<<<(unsigned)((m + 7) / 8), 256, 0, st>>>(h->rows.get() + (size_t)h->img_n * h->ld, h->ld, rb, m,
                                                                  h->img.get() + (size_t)h->img_n * rb);
        CK(cudaGetLastError());
        CK(cudaEventRecord(h->img_ev, st));
        h->launches++;
        h->img_n = h->n;
        h->img_st = st;
    } else if (st != h->img_st) {
        CK(cudaStreamWaitEvent(st, h->img_ev, 0));  // the last conversion ran on another stream
    }
    *ok = true;
    return 0;
}

// Exhaustive top-k of `nq` device queries (row stride ld) against `nrows` rows: K1 with the K3 merge (and, when `ex`
// is given, the multi-GPU exchange) fused into its tail; K1 + K3 as two launches when the tail cannot be fused.
// A search of 1-2 queries over a flat store's own rows, when the store is large, streams its int8 image and re-scores
// the candidates in fp32 (DESIGN.md "K1"); the fp32 scan serves everything else, and searches whose image does not fit.
static int run_flat_scan(wb_index* h, const float* rows, int64_t nrows, const float* q_dev, int64_t nq, int k,
                         const int64_t* ids, float* D, int64_t* I, cudaStream_t st, bool timed,
                         const ExchParams* ex = nullptr, bool* exchanged = nullptr, const RowMask* mask = nullptr) {
    if (exchanged) *exchanged = false;
    ScanCfg c;
    bool img = !h->ivf && rows == h->rows.get() && nq <= kImageMaxQueries && nrows >= kImageMinRowsPerSm * h->sm_count &&
               plan_scan(h, nq, k, false, 0, &c, true) == 0;
    if (img) TRY(ensure_image(h, st, &img));
    if (!img) TRY(plan_scan(h, nq, k, false, 0, &c));
    const int64_t S = flat_ctas(h, c, nrows, nq);
    TRY(h->parts.ensure((size_t)nq * S * k * sizeof(uint64_t)));
    ScanParams p{};
    p.rows = rows;
    p.nrows = nrows;
    p.ld = h->ld;
    p.k = k;
    p.nparts = (int)S;
    p.allow = mask ? mask->allow : nullptr;
    if (img) {
        p.img = h->img.get();
        p.rescored = h->img_rescored.get();
        h->img_searches++;
    }
    int S_merge = 0, heads_bytes = 0;
    if (tail_fusable(c, k, S, ex ? ex->world : 1, &S_merge, &heads_bytes)) {
        TRY(ensure_tail_counters(h, st));
        set_tail(p, h, c, S_merge, heads_bytes, ids, ex ? ex->D : D, ex ? ex->I : I, k, ex);
    }
    return run_scan_groups(h, c, false, p, nq, q_dev, ids, D, I, st, timed, ex, exchanged);
}

// ---- K2: tensor-core batched scan ---------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// 2-D TMA map of a row matrix [nrows, ld] (fp32) in kGemmBM x kGemmBK boxes: the A operand of every K2 kernel.
static int encode_rows_tmap(const float* rows, int ld, int64_t nrows, CUtensorMap* out) {
    static PFN_encodeTiled encode = nullptr;
    if (!encode) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        CK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres));
        if (qres != cudaDriverEntryPointSuccess || !p) return fail("cuTensorMapEncodeTiled is not available in this driver");
        encode = (PFN_encodeTiled)p;
    }
    cuuint64_t gdim[2] = {(cuuint64_t)ld, (cuuint64_t)nrows};
    cuuint64_t gstr[1] = {(cuuint64_t)ld * 4};
    cuuint32_t box[2] = {(cuuint32_t)kGemmBK, (cuuint32_t)kGemmBM};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = encode(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)rows, gdim, gstr, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail("cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
    return 0;
}

// Cost model behind the K1 / K2 choice, measured on B200 (profiles/r01/small_store_latency.txt, batch sweeps of
// profiles/r01 and r02): an 8-query K1 pass streams the rows at ~4.2 TB/s-equivalent (FMA-bound at 8 queries per CTA);
// K2 streams them once at ~6 TB/s but pays ~0.3 ms per search for its epoch launches, compactions and the one
// stream synchronisation that reads the overflow flag.
constexpr double kK1BatchBytesPerS = 4.2e12;
constexpr double kK2StreamBytesPerS = 6.0e12;
constexpr double kK2FixedSeconds = 0.3e-3;
constexpr int64_t kK2MinBatch = 5;  // measured: K2 5.8 ms vs K1 8.1 ms at 5..8 queries (10M x 768)

// Range search (DESIGN.md "Range search"): the hits of one chunk of queries are held on the device at 20 bytes each
// (pool key + query tag, one sort buffer); a chunk holds at most this many, and so does an enlarged K2 candidate list.
constexpr int64_t kRangeBudgetHits = (int64_t)1 << 28;
constexpr int kRangeEpochs = 64;  // K2 range epochs of one batch, re-runs included (12x growth: ~6 + ~6 re-runs)

// Can the tensor-core path take this problem?  (candidate capacity `cap` rows form epoch 0)
static bool gemm_eligible(const wb_index* h, int64_t nrows, int64_t nq, int k, int* cap_out) {
    if (nq < kK2MinBatch) return false;
    if (nrows >= ((int64_t)1 << 31) - 256) return false;  // TMA coordinates are int32
    int64_t cap = std::min<int64_t>(4096, std::max<int64_t>(256, ((nrows / 64) + 127) / 128 * 128));
    if (cap < 2 * (int64_t)k || nrows < 4 * cap) return false;
    // K2 pays ~0.3 ms of fixed cost per search (epoch launches, compactions, one stream sync) and then streams the
    // rows at ~6 TB/s; K1 needs ceil(nq/8) passes at ~4.2 TB/s-equivalent but has no fixed cost.  Small stores with
    // few queries are faster on K1 (e.g. 100k x 512 with 16 queries: 0.1 ms vs 0.35 ms).
    if (env_int("WB_GEMM_FORCE", 0) == 0) {
        const double bytes = (double)nrows * h->ld * 4.0;
        const double passes = (double)((nq + 7) / 8);
        if (passes * bytes / kK1BatchBytesPerS < kK2FixedSeconds + bytes / kK2StreamBytesPerS) return false;
    }
    *cap_out = (int)cap;
    return true;
}

template <int BN>
static int run_flat_gemm_t(wb_index* h, const float* rows, int64_t nrows, const float* q_ld, int64_t nq, int k, int cap,
                         const int64_t* ids, float* D, int64_t* I, cudaStream_t st, bool timed, bool* overflowed,
                         const RowMask* mask, const RangeOut* range) {
    // Filter-and-refine (rows of the store, or the compact copy of a filter's rows: norm2_max bounds both; not the
    // centroid table): after the first epoch the GEMM issues only the hi x hi term and the compaction re-scores the few
    // hundred candidates per query exactly in fp32.
    // A range search (`range`, k = 0) runs every epoch one-term: a 3xTF32 score is not the exact fp32 score, so it must
    // not decide membership.
    const bool filter = rows != h->centroids.get() && (range || env_int("WB_GEMM_FILTER", 1) != 0);
    constexpr bool kFold = kGemmFold<BN, false>;
    using Cfg = GemmCfg<BN, kFold>;
    constexpr int kGemmBN = BN;
    constexpr int kGemmBBytes = Cfg::kBBytes;
    constexpr size_t kGemmSmemBytes = Cfg::kSmemBytes;
    const int ld = h->ld;
    const int nchunks = (ld + kGemmBK - 1) / kGemmBK;
    const int nqb = (int)((nq + kGemmBN - 1) / kGemmBN);
    const int kstride = k + cap;
    // measured (10M x 768): 40 / 64 queries 5.9 / 6.3 ms on one CTA vs 6.2 / 6.4 ms on the pair; 128 queries 8.8 vs 8.1 ms
    const bool use2 = BN >= 128 && (h->sm_count % 2) == 0;
    // Batches above 128 queries run their filter epochs in 256-query blocks on the SS kernel (gemm_ss.cuh): half as many
    // passes over the rows and 1.5x fewer L2 bytes per MAC than 128-query blocks.
    const bool use_f2 = use2 && filter && nq > 128;
    // a single block of 65..128 queries: the same SS kernel with 64 queries per CTA (one pass over the rows, HBM-bound)
    const bool use_f2h = use2 && filter && nq <= 128;
    const int nqb2 = (int)((nq + kF2BN - 1) / kF2BN);
    const int nq_pad = use_f2 ? nqb2 * kF2BN : nqb * kGemmBN;  // thresholds / margins of padding queries: +inf / 0
    TRY(h->gimg.ensure((size_t)nqb * nchunks * kGemmBBytes));
    TRY(h->gkeys.ensure((size_t)nq * kstride * sizeof(uint64_t)));
    // thr | cnt | overflow | one work dispenser per epoch | range: overflow flag and candidate count of each epoch
    TRY(h->gstate.ensure((size_t)nq_pad * 4 + (size_t)nq * 4 + 64 + 64 * 4 + (range ? 2 * kRangeEpochs * 4 : 0)));
    float* thr = h->gstate.as<float>();
    float* margin = nullptr;
    if (filter) {
        TRY(h->gmargin.ensure((size_t)nq_pad * 4));
        margin = h->gmargin.as<float>();
        // |exact - hi.hi| <= 2^-9 |x||q| (two truncations to tf32, Cauchy-Schwarz) + fp32 accumulation slack
        // (n-term fp32 accumulation: <= n * 2^-23 * sum |x_i q_i| even if the tensor core truncates)
        const float c_margin = 1.953125e-3f + (float)ld * 1.1920929e-7f * 1.1f + 1e-5f;
        query_margin_kernel<<<(unsigned)((nq_pad * 32 + 255) / 256), 256, 0, st>>>(q_ld, (int)nq, nq_pad, ld, h->norm2_max.get(),
                                                                                 c_margin, margin);
        CK(cudaGetLastError());
        h->launches++;
    }
    if (use_f2) {
        TRY(h->gimg2.ensure((size_t)nqb2 * 2 * nchunks * kF2BBytes));
        const int64_t n4 = (int64_t)nqb2 * 2 * nchunks * 8 * kF2Half;
        image_queries_f2_kernel<128><<<(unsigned)((n4 + 255) / 256), 256, 0, st>>>(q_ld, (int)nq, ld, nchunks, nqb2,
                                                                                  h->gimg2.as<float>());
        CK(cudaGetLastError());
        h->launches++;
    } else if (use_f2h) {
        TRY(h->gimg2.ensure((size_t)nqb * 2 * nchunks * F2Cfg<64>::kBBytes));
        const int64_t n4 = (int64_t)nqb * 2 * nchunks * 8 * 64;
        image_queries_f2_kernel<64><<<(unsigned)((n4 + 255) / 256), 256, 0, st>>>(q_ld, (int)nq, ld, nchunks, nqb,
                                                                                 h->gimg2.as<float>());
        CK(cudaGetLastError());
        h->launches++;
    }
    int* cnt = reinterpret_cast<int*>(thr + (size_t)nq_pad);
    int* overflow = cnt + nq;
    unsigned int* dispensers = reinterpret_cast<unsigned int*>(overflow + 16);  // [64], zeroed once per search
    int* rflags = range ? reinterpret_cast<int*>(dispensers + 64) : nullptr;  // [kRangeEpochs] flags, then counts
    CK(cudaMemsetAsync(dispensers, 0, 64 * sizeof(unsigned int) + (range ? 2 * kRangeEpochs * 4 : 0), st));
    int epoch_no = 0;
    uint64_t* keys = h->gkeys.as<uint64_t>();
    {
        const int64_t n1 = std::max<int64_t>((int64_t)nq_pad, nq * (int64_t)k);
        if (range)
            range_gemm_init_kernel<<<(unsigned)((nq_pad + 255) / 256), 256, 0, st>>>(thr, (int)nq, nq_pad, range->thresh, cnt);
        else
            init_gemm_state_kernel<<<(unsigned)((n1 + 255) / 256), 256, 0, st>>>(thr, (int)nq, nq_pad, cnt, keys, k,
                                                                                kstride, overflow);
        CK(cudaGetLastError());
        const int64_t n2 = (int64_t)nqb * nchunks * 8 * kGemmBN;
        if constexpr (BN >= 128) {
            if (use2) {  // the 2-CTA kernel wants one image per 64 queries (each CTA of a pair holds half a block)
                const int64_t n3 = (int64_t)(2 * nqb) * nchunks * 8 * (BN / 2);
                split_queries_kernel<BN / 2><<<(unsigned)((n3 + 255) / 256), 256, 0, st>>>(q_ld, (int)nq, ld, nchunks,
                                                                                      2 * nqb, h->gimg.as<float>());
            }
        }
        if (!use2) {
            split_queries_kernel<BN, kFold><<<(unsigned)((n2 + 255) / 256), 256, 0, st>>>(q_ld, (int)nq, ld, nchunks, nqb,
                                                                                     h->gimg.as<float>());
            if (kFold && filter) {  // the one-term epochs read a plain image (hi half only), the first epoch the folded one
                TRY(h->gimg2.ensure((size_t)nqb * nchunks * kGemmBBytes));
                split_queries_kernel<BN, false><<<(unsigned)((n2 + 255) / 256), 256, 0, st>>>(q_ld, (int)nq, ld, nchunks, nqb,
                                                                                         h->gimg2.as<float>());
                h->launches++;
            }
        }
        CK(cudaGetLastError());
        h->launches += 2;
    }
    CUtensorMap tmap;
    TRY(encode_rows_tmap(rows, ld, nrows, &tmap));
    if constexpr (BN >= 128) {  // the CTA pair exists for 128-query blocks only
        if (use2) {
            CK(smem_optin<gemm2_topk_kernel<BN, false>>((int)Gemm2Cfg<BN>::kSmemBytes));
            if (use_f2) CK(smem_optin<filter2_topk_kernel<128, false, false>>((int)kF2SmemBytes));
            if (use_f2h) CK(smem_optin<filter2_topk_kernel<64, false, false>>((int)F2Cfg<64>::kSmemBytes));
        }
    }
    if (!use2) {
        CK(smem_optin<gemm_topk_kernel<BN, false>>((int)kGemmSmemBytes));
        CK(smem_optin<gemm_topk_kernel<BN, false, 1>>((int)GemmCfg<BN, false>::kSmemBytes));
    }
    CK(smem_optin<merge_topk_kernel<true>>(8192 * 8));
    CK(smem_optin<compact_topk_kernel>(8192 * 8));
    GemmParams g{};
    g.nchunks = nchunks;
    g.nq = (int)nq;
    g.nqb = nqb;
    g.bimg = h->gimg.as<float>();
    g.thr = thr;
    g.margin = margin;
    g.keys = keys;
    g.cnt = cnt;
    g.overflow = overflow;
    g.k = k;
    g.cap = cap;
    g.kstride = kstride;
    g.allow = mask ? mask->allow : nullptr;
    CompactParams c{};
    c.k = k;
    c.cap = cap;
    c.kstride = kstride;
    {
        const int64_t mmax = (int64_t)k + cap;
        const int full = pow2_ceil(k + 2 * kMergeThreads);
        c.S = mmax <= full ? pow2_ceil((int)mmax) : full;
    }
    c.keys = keys;
    c.cnt = cnt;
    c.thr = thr;
    c.ids = ids;
    c.rows = rows;
    c.q = q_ld;
    c.ld = ld;
    // next epoch = growth x (rows seen so far): a query then collects ~k*ln(1+growth) survivors per epoch, far
    // below `cap`; fewer, larger epochs mean fewer launch gaps and compactions (each costs ~50 us)
    const double growth = std::min(12.0, std::max(0.25, (double)cap / (4.0 * k)));
    // one epoch over rows [r0, r1): the K2 launch, the exact re-scoring of its candidates and their compaction
    auto run_epoch = [&](int64_t r0, int64_t r1) -> int {
        g.row_begin = r0;
        g.row_end = r1;
        const int64_t nwork = ((r1 - r0 + kGemmBM - 1) / kGemmBM) * nqb;
        const unsigned grid = (unsigned)std::min<int64_t>(nwork, h->sm_count);
        // first epoch: 3xTF32 scores select, the winners are re-scored; later epochs: one-term filter, candidates re-scored
        const bool one_term = filter && (r0 > 0 || range);
        c.rescore = filter ? (r0 == 0 && !range ? 2 : 1) : 0;
        if (range) g.overflow = rflags + epoch_no;
        if constexpr (BN >= 128) {
            // with the pair, every filter epoch (one_term) goes to the SS kernel: use_f2 or use_f2h is set
            const int64_t ntp = ((r1 - r0 + kGemmBM - 1) / kGemmBM + 1) / 2;
            if (use_f2 && one_term) {  // 256-query blocks, both operands from shared memory
                GemmParams g2 = g;
                g2.nqb = nqb2;
                g2.bimg = h->gimg2.as<float>();
                const unsigned grid3 = 2u * (unsigned)std::min<int64_t>(ntp * nqb2, h->sm_count / 2);
                filter2_topk_kernel<128, false, false><<<grid3, kF2Threads, kF2SmemBytes, st>>>(tmap, g2);
            } else if (use_f2h && one_term) {
                GemmParams g2 = g;
                g2.bimg = h->gimg2.as<float>();
                const unsigned grid3 = 2u * (unsigned)std::min<int64_t>(ntp * nqb, h->sm_count / 2);
                filter2_topk_kernel<64, false, false><<<grid3, kF2Threads, F2Cfg<64>::kSmemBytes, st>>>(tmap, g2);
            } else if (use2) {
                const unsigned grid2 = 2u * (unsigned)std::min<int64_t>(ntp * nqb, h->sm_count / 2);
                gemm2_topk_kernel<BN, false><<<grid2, kGemmThreads, Gemm2Cfg<BN>::kSmemBytes, st>>>(tmap, g);
            }
        }
        if (!use2) {
            // SMs stream at different rates: (tile, block) items are drawn from a dispenser, not dealt out statically
            g.work_counter = epoch_no < 64 ? dispensers + epoch_no : nullptr;
            if (one_term) {
                GemmParams g1 = g;
                if (kFold) g1.bimg = h->gimg2.as<float>();
                gemm_topk_kernel<BN, false, 1><<<grid, kGemmThreads, GemmCfg<BN, false>::kSmemBytes, st>>>(tmap, g1);
            } else {
                gemm_topk_kernel<BN, false><<<grid, kGemmThreads, kGemmSmemBytes, st>>>(tmap, g);
            }
        }
        CK(cudaGetLastError());
        const bool last = r1 >= nrows;
        c.D = last ? D : nullptr;
        c.I = last ? I : nullptr;
        if (c.rescore == 1) {
            const unsigned gy = (unsigned)std::max<int64_t>(1, std::min<int64_t>(64, (int64_t)h->sm_count * 4 / nq));
            rescore_candidates_kernel<<<dim3((unsigned)nq, gy), 256, 0, st>>>(c);
            CK(cudaGetLastError());
            h->launches++;
        }
        if (range) {
            const RangeCollect rc{keys, cnt, g.cap, g.kstride, rflags + epoch_no, rflags + kRangeEpochs + epoch_no, *range};
            range_collect_kernel<<<(unsigned)nq, kRangeThreads, 0, st>>>(rc);
        } else {
            compact_topk_kernel<<<(unsigned)nq, kMergeThreads, (size_t)c.S * 8, st>>>(c);
        }
        CK(cudaGetLastError());
        h->launches += 2;
        h->gemm_launches++;
        epoch_no++;
        return 0;
    };
    TRY(timing_begin(h, timed && h->timing, st));
    std::vector<std::pair<int64_t, int64_t>> spans;  // range: the row span of every epoch (overflow repair)
    int64_t r0 = 0;
    while (r0 < nrows) {
        if (range && epoch_no >= kRangeEpochs / 2) {  // (not reached: 12x growth; K1 takes the batch)
            *overflowed = true;
            return 0;
        }
        int64_t r1;
        if (mask) {
            // the same schedule in SELECTED rows: epoch 0 ends before its selected rows (every one of them a candidate)
            // exceed `cap`, later epochs take growth x the selected rows seen so far.  Counting all rows instead, a
            // filter that keeps 13 % of the rows leaves fewer than k = 1000 of them in a 4096-row epoch 0, the
            // threshold stays -inf and the next epoch's candidates overflow `cap`.  (A filter that keeps every row
            // gets exactly the unfiltered epochs.)
            const int64_t t0 = r0 / kGemmBM, nt = (nrows + kGemmBM - 1) / kGemmBM;
            const int64_t seen = mask->sel[t0];
            const int64_t grow = (int64_t)((double)seen * growth);
            const int64_t want = seen + (r0 == 0 ? cap : (grow + kGemmBM - 1) / kGemmBM * kGemmBM);
            const int64_t t1 = std::upper_bound(mask->sel + t0 + 1, mask->sel + nt + 1, want) - mask->sel - 1;
            r1 = std::min(nrows, std::max(t1, t0 + 1) * kGemmBM);
        } else {
            int64_t len = r0 == 0 ? cap : (int64_t)((double)r0 * growth);
            len = std::max<int64_t>(kGemmBM, (len + kGemmBM - 1) / kGemmBM * kGemmBM);
            r1 = std::min(nrows, r0 + len);
        }
        TRY(run_epoch(r0, r1));
        if (range) spans.emplace_back(r0, r1);
        r0 = r1;
    }
    TRY(timing_end(h, timed && h->timing, st));
    if (range) {
        // An epoch whose candidate list overflowed contributed nothing; its exact candidate count is known, so it is
        // re-run once with a list that holds them all.  *overflowed: the enlarged lists would exceed the budget (the
        // caller runs the batch on K1 instead).
        *overflowed = false;
        std::vector<int> fl(2 * kRangeEpochs);
        CK(cudaMemcpyAsync(fl.data(), rflags, fl.size() * sizeof(int), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        const int first = epoch_no;
        for (size_t e = 0; e < spans.size(); ++e) {
            if (!fl[e]) continue;
            const int64_t want = ((int64_t)fl[kRangeEpochs + e] + 127) / 128 * 128;
            if (nq * want > kRangeBudgetHits || epoch_no >= kRangeEpochs) {
                *overflowed = true;
                return 0;
            }
            TRY(h->gkeys.ensure((size_t)nq * want * sizeof(uint64_t)));
            keys = h->gkeys.as<uint64_t>();
            g.keys = c.keys = keys;
            g.cap = g.kstride = c.cap = c.kstride = (int)want;
            TRY(run_epoch(spans[e].first, spans[e].second));
        }
        if (epoch_no > first) {
            CK(cudaMemcpyAsync(fl.data(), rflags, kRangeEpochs * sizeof(int), cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            for (int e = first; e < epoch_no; ++e) *overflowed |= fl[e] != 0;
        }
        return 0;
    }
    int ovf = 0;
    CK(cudaMemcpyAsync(&ovf, overflow, sizeof(int), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    *overflowed = ovf != 0;
    return 0;
}

static int run_flat_gemm(wb_index* h, const float* rows, int64_t nrows, const float* q_ld, int64_t nq, int k, int cap,
                         const int64_t* ids, float* D, int64_t* I, cudaStream_t st, bool timed, bool* overflowed,
                         const RowMask* mask, const RangeOut* range = nullptr) {
    // 16-query blocks halve the image traffic and the MMA work of a half-empty 32-query block (K2 is power-capped at
    // small batches: 992 W and 1.37 GHz at batch 16)
    if (nq <= 16) return run_flat_gemm_t<16>(h, rows, nrows, q_ld, nq, k, cap, ids, D, I, st, timed, overflowed, mask, range);
    if (nq <= 32) return run_flat_gemm_t<32>(h, rows, nrows, q_ld, nq, k, cap, ids, D, I, st, timed, overflowed, mask, range);
    if (nq <= 64) return run_flat_gemm_t<64>(h, rows, nrows, q_ld, nq, k, cap, ids, D, I, st, timed, overflowed, mask, range);
    return run_flat_gemm_t<128>(h, rows, nrows, q_ld, nq, k, cap, ids, D, I, st, timed, overflowed, mask, range);
}

// K4/K6 on the tensor cores: argmax over the centroid table for n device-resident points (row stride ld).
// One launch, no epochs, no host synchronisation: the points are the A operand (streamed once from HBM), the
// centroids are the query images (L2 resident), each row keeps its running maximum in the epilogue.
static bool assign_gemm_eligible(const wb_index* h, int64_t n) {
    return n >= 1024 && h->nlist >= 64 && n < ((int64_t)1 << 31) - 256;
}

static int run_assign_gemm(wb_index* h, const float* x_ld, int64_t n, int32_t* assign_out, float* best_out,
                           cudaStream_t st, bool tf32 = false) {
    constexpr int BN = 128;
    using Cfg = GemmCfg<BN>;
    const int ld = h->ld;
    const int nchunks = (ld + kGemmBK - 1) / kGemmBK;
    const bool use2 = (h->sm_count % 2) == 0;
    CUtensorMap tmap;
    if (tf32 && use2) {
        // k-means TRAINING assignment: plain TF32 on the SS pair kernel, 256 centroids per block (gemm_ss.cuh)
        const int nqb2 = (int)((h->nlist + kF2BN - 1) / kF2BN);
        TRY(h->gimg2.ensure((size_t)nqb2 * 2 * nchunks * kF2BBytes));
        const int64_t n4 = (int64_t)nqb2 * 2 * nchunks * 8 * kF2Half;
        image_queries_f2_kernel<<<(unsigned)((n4 + 255) / 256), 256, 0, st>>>(h->centroids.get(), (int)h->nlist, ld, nchunks, nqb2,
                                                                             h->gimg2.as<float>());
        CK(cudaGetLastError());
        TRY(encode_rows_tmap(x_ld, ld, n, &tmap));
        CK(smem_optin<filter2_topk_kernel<128, true, false>>((int)kF2SmemBytes));
        GemmParams g{};
        g.row_begin = 0;
        g.row_end = n;
        g.nchunks = nchunks;
        g.nq = (int)h->nlist;
        g.nqb = nqb2;
        g.bimg = h->gimg2.as<float>();
        g.assign_out = assign_out;
        g.best_out = best_out;
        const int64_t ntp = ((n + kGemmBM - 1) / kGemmBM + 1) / 2;
        filter2_topk_kernel<128, true, false><<<2u * (unsigned)std::min<int64_t>(ntp, h->sm_count / 2), kF2Threads, kF2SmemBytes, st>>>(tmap, g);
        CK(cudaGetLastError());
        h->launches += 2;
        h->gemm_launches++;
        return 0;
    }
    const int nqb = (int)((h->nlist + BN - 1) / BN);
    TRY(h->gimg.ensure((size_t)nqb * nchunks * Cfg::kBBytes));
    const int64_t n2 = (int64_t)nqb * nchunks * 8 * BN;
    if (use2) {
        const int64_t n3 = (int64_t)(2 * nqb) * nchunks * 8 * (BN / 2);
        split_queries_kernel<BN / 2><<<(unsigned)((n3 + 255) / 256), 256, 0, st>>>(h->centroids.get(), (int)h->nlist, ld, nchunks,
                                                                              2 * nqb, h->gimg.as<float>());
    } else {
        split_queries_kernel<BN><<<(unsigned)((n2 + 255) / 256), 256, 0, st>>>(h->centroids.get(), (int)h->nlist, ld, nchunks, nqb,
                                                                              h->gimg.as<float>());
    }
    CK(cudaGetLastError());
    TRY(encode_rows_tmap(x_ld, ld, n, &tmap));
    GemmParams g{};
    g.row_begin = 0;
    g.row_end = n;
    g.nchunks = nchunks;
    g.nq = (int)h->nlist;
    g.nqb = nqb;
    g.bimg = h->gimg.as<float>();
    g.assign_out = assign_out;
    g.best_out = best_out;
    const int64_t ntiles = (n + kGemmBM - 1) / kGemmBM;
    if (use2) {
        CK(smem_optin<gemm2_topk_kernel<BN, true>>((int)Gemm2Cfg<BN>::kSmemBytes));
        const int64_t ntp = (ntiles + 1) / 2;
        gemm2_topk_kernel<BN, true><<<2u * (unsigned)std::min<int64_t>(ntp, h->sm_count / 2), kGemmThreads,
                                     Gemm2Cfg<BN>::kSmemBytes, st>>>(tmap, g);
    } else {
        CK(smem_optin<gemm_topk_kernel<BN, true>>((int)Cfg::kSmemBytes));
        gemm_topk_kernel<BN, true><<<(unsigned)std::min<int64_t>(ntiles, h->sm_count), kGemmThreads, Cfg::kSmemBytes, st>>>(tmap, g);
    }
    CK(cudaGetLastError());
    h->launches += 2;
    h->gemm_launches++;
    return 0;
}

// Exhaustive top-k, any batch size: tensor cores (K2) when the batch is big enough, else the
// bandwidth-bound CUDA-core scan (K1).  A candidate-list overflow in K2 (adversarially ordered data)
// is repaired by re-running the batch through K1.
static int run_flat_any(wb_index* h, const float* rows, int64_t nrows, const float* q_dev, int64_t nq, int k,
                        const int64_t* ids, float* D, int64_t* I, cudaStream_t st, bool timed,
                        const ExchParams* ex = nullptr, bool* exchanged = nullptr, const RowMask* mask = nullptr) {
    if (exchanged) *exchanged = false;
    int cap = 0;
    if (gemm_eligible(h, nrows, nq, k, &cap)) {
        const int64_t max_q = 65536;  // bounds the candidate buffers
        bool any_overflow = false;
        for (int64_t q0 = 0; q0 < nq; q0 += max_q) {
            const int64_t nqc = std::min(max_q, nq - q0);
            bool ovf = false;
            TRY(run_flat_gemm(h, rows, nrows, q_dev + (size_t)q0 * h->ld, nqc, k, cap, ids, D + (size_t)q0 * k,
                              I + (size_t)q0 * k, st, timed, &ovf, mask));
            any_overflow |= ovf;
        }
        if (!any_overflow) return 0;
        h->gemm_fallbacks++;
    }
    return run_flat_scan(h, rows, nrows, q_dev, nq, k, ids, D, I, st, timed,
                         ex && nq <= kMaxGridY ? ex : nullptr, exchanged, mask);
}

// ---- K8: CSR inverted lists, built on the device (csr.cuh) -------------------------------------------------------
// Stable grouping of n items by list: list_off[nlist + 1], src[slot] = item index, pos_out[slot] = pos_in[item].
// Everything is enqueued on `st`; the only host involvement is reading one error word when `check` is set.
static int device_csr(wb_index* h, const int32_t* assign, int64_t n, const uint32_t* pos_in, int64_t* list_off,
                      uint32_t* src, uint32_t* pos_out, cudaStream_t st, bool check) {
    const int64_t nlist = h->nlist;
    if (n >= (int64_t)0xFFFFFFFFll) return fail("too many items to group");
    // B blocks of items: enough to fill the GPU, few enough for the [B][nlist] counter matrix to stay small
    int64_t B = std::min<int64_t>(1024, std::max<int64_t>(1, (n + 4095) / 4096));
    B = std::max<int64_t>(1, std::min<int64_t>(B, ((int64_t)64 << 20) / std::max<int64_t>(nlist, 1)));
    int64_t ipb = (n + B - 1) / B;
    ipb = std::max<int64_t>(kCsrTile, (ipb + kCsrTile - 1) / kCsrTile * kCsrTile);
    B = std::max<int64_t>(1, (n + ipb - 1) / ipb);
    TRY(h->ccnt.ensure((size_t)B * nlist * sizeof(uint32_t) + 64));
    TRY(h->ctot.ensure((size_t)nlist * sizeof(int64_t) + 64));
    uint32_t* cnt = h->ccnt.as<uint32_t>();
    int* bad = reinterpret_cast<int*>(h->ctot.as<unsigned char>() + (size_t)nlist * sizeof(int64_t));
    CK(cudaMemsetAsync(cnt, 0, (size_t)B * nlist * sizeof(uint32_t), st));
    CK(cudaMemsetAsync(bad, 0, sizeof(int), st));
    if (n > 0) {
        csr_hist_kernel<<<(unsigned)B, kCsrTile, 0, st>>>(assign, n, nlist, ipb, cnt, bad);
        CK(cudaGetLastError());
    }
    csr_colscan_kernel<<<(unsigned)((nlist + 255) / 256), 256, 0, st>>>(cnt, (int)B, nlist, h->ctot.as<int64_t>());
    CK(cudaGetLastError());
    csr_offsets_kernel<<<1, 1024, 0, st>>>(h->ctot.as<int64_t>(), nlist, list_off);
    CK(cudaGetLastError());
    if (n > 0) {
        csr_scatter_kernel<<<(unsigned)B, kCsrTile, 0, st>>>(assign, n, nlist, ipb, cnt, list_off, pos_in, src, pos_out);
        CK(cudaGetLastError());
    }
    h->launches += 4;
    if (check) {
        int hb = 0;
        CK(cudaMemcpyAsync(&hb, bad, sizeof(int), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        if (hb) return fail("a row has a list assignment outside [0, %lld)", (long long)nlist);
    }
    return 0;
}

// Build the inverted lists.  Default: PHYSICALLY group the row store by list (rows of a list become one
// contiguous span, insertion order kept inside a list), so the list scan is a sequential HBM stream instead of
// a gather of 2-3 KB rows (measured 3.3-4.3 TB/s gathered).  Needs a second copy of the rows while it runs; if
// that does not fit, the lists stay a CSR of row indices (slot_row) over the store as it is.
// A failure leaves the store as it was and the lists dirty (list_off and slot_row describe nothing until then).
static int ensure_csr(wb_index* h) {
    if (!h->csr_dirty) return 0;
    cudaStream_t st = h->stream;
    const int64_t n = h->n;
    h->slot_row.reset();
    if (n == 0) {
        CK(cudaMemsetAsync(h->list_off.get(), 0, (size_t)(h->nlist + 1) * sizeof(int64_t), st));
        CK(cudaStreamSynchronize(st));
        h->csr_dirty = false;
        return 0;
    }
    DevPtr<uint32_t> src, pos_out;
    const int64_t mcap = std::max<int64_t>(h->cap, n);
    CK(dev_alloc(&src, (size_t)n * sizeof(uint32_t)));
    CK(dev_alloc(&pos_out, (size_t)mcap * sizeof(uint32_t)));
    TRY(device_csr(h, h->assign.get(), n, h->row_pos.get(), h->list_off.get(), src.get(), pos_out.get(), st, true));
    if (env_int("WB_IVF_CONTIGUOUS", 1)) {
        const int64_t ncap = std::max<int64_t>(h->cap, std::max<int64_t>(n, 1024));
        const size_t need = (size_t)ncap * h->ld * 4 + (size_t)ncap * 4;
        size_t free_b = 0, total_b = 0;
        CK(cudaMemGetInfo(&free_b, &total_b));
        if (free_b > need + kMemReserve) {
            DevPtr<float> nrows;
            DevPtr<int32_t> nas;
            DevPtr<int64_t> nids;  // ids keep their insertion order; they only follow the capacity
            CK(dev_alloc(&nrows, (size_t)ncap * h->ld * 4));
            CK(dev_alloc(&nas, (size_t)ncap * 4));
            if (ncap > h->cap) CK(dev_alloc(&nids, (size_t)ncap * 8));
            const int ld4 = h->ld / 4;
            const int64_t tot = n * ld4;
            permute_rows_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(
                reinterpret_cast<const float4*>(h->rows.get()), reinterpret_cast<float4*>(nrows.get()), src.get(), n, ld4);
            CK(cudaGetLastError());
            permute_i32_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(h->assign.get(), nas.get(), src.get(), n);
            CK(cudaGetLastError());
            h->launches += 2;
            if (nids) CK(cudaMemcpyAsync(nids.get(), h->ids.get(), (size_t)n * 8, cudaMemcpyDeviceToDevice, st));
            CK(cudaStreamSynchronize(st));
            h->rows = std::move(nrows);
            h->assign = std::move(nas);
            if (nids) h->ids = std::move(nids);
            h->cap = ncap;
            h->row_pos = std::move(pos_out);  // storage row -> insertion position
            h->map_cap = mcap;
            h->csr_dirty = false;
            return 0;
        }
    }
    // rows stay put: lists are row indices, row_pos (if any) still describes the storage
    CK(cudaStreamSynchronize(st));
    h->slot_row = std::move(src);
    h->csr_dirty = false;
    return 0;
}

// ---- add -----------------------------------------------------------------------------------
// assign rows [n0, n0+n) of the store to their max-inner-product centroid (K4 with k = 1)
static int assign_rows(wb_index* h, const float* x_dev, int64_t n, int32_t* assign_out, float* best_out,
                       cudaStream_t st, bool tf32 = false) {
    if (assign_gemm_eligible(h, n)) return run_assign_gemm(h, x_dev, n, assign_out, best_out, st, tf32);
    TRY(h->pD.ensure((size_t)n * sizeof(float)));
    TRY(h->pI.ensure((size_t)n * sizeof(int64_t)));
    float* D = best_out ? best_out : h->pD.as<float>();
    TRY(run_flat_any(h, h->centroids.get(), h->nlist, x_dev, n, 1, nullptr, D, h->pI.as<int64_t>(), st, false));
    labels_to_lists_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(h->pI.as<int64_t>(), assign_out, n);
    CK(cudaGetLastError());
    h->launches++;
    return 0;
}

static int add_common(wb_index* h, int64_t n, const float* x, const int64_t* ids, bool host, const int32_t* preassign,
                      cudaStream_t st, bool sync_host = true) {
    if (!h) return fail("NULL index");
    if (n < 0) return fail("negative n");
    if (n == 0) return 0;
    if (!x) return fail("x is NULL");
    TRY(set_dev(h));
    if (h->ivf && !h->trained) return fail("IndexIVFFlat must be trained before adding vectors");
    if (h->n + n > h->cap && st != h->stream) CK(cudaStreamSynchronize(st));  // growth copies run on the handle's stream
    TRY(ensure_capacity(h, h->n + n));
    const int64_t n0 = h->n;
    float* dst = h->rows.get() + (size_t)n0 * h->ld;
    const cudaMemcpyKind kind = host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
    if (h->ld == h->d) {
        CK(cudaMemcpyAsync(dst, x, (size_t)n * h->d * sizeof(float), kind, st));
    } else {
        const float* src = x;
        if (host) {
            TRY(h->xbuf.ensure((size_t)n * h->d * sizeof(float)));
            CK(cudaMemcpyAsync(h->xbuf.get(), x, (size_t)n * h->d * sizeof(float), kind, st));
            src = h->xbuf.as<float>();
        }
        const int64_t tot = n * h->ld;
        pad_rows_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(src, dst, n, h->d, h->ld);
        CK(cudaGetLastError());
        h->launches++;
    }
    {   // running max of |row|^2: the K2 filter epochs derive their safety margin from it
        const unsigned blocks = (unsigned)std::min<int64_t>((n + 7) / 8, (int64_t)h->sm_count * 8);
        row_norm2_max_kernel<<<blocks, 256, 0, st>>>(dst, n, h->ld, h->norm2_max.get());
        CK(cudaGetLastError());
        h->launches++;
    }
    if (ids) {
        CK(cudaMemcpyAsync(h->ids.get() + n0, ids, (size_t)n * sizeof(int64_t), kind, st));
    } else {
        iota_ids_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(h->ids.get() + n0, n0, n);
        CK(cudaGetLastError());
        h->launches++;
    }
    if (h->row_pos) {  // the store has been grouped before: new rows sit at their insertion position
        iota_u32_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(h->row_pos.get(), n0, n);
        CK(cudaGetLastError());
        h->launches++;
    }
    if (h->ivf) {
        if (preassign) {
            CK(cudaMemcpyAsync(h->assign.get() + n0, preassign, (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        } else {
            TRY(assign_rows(h, dst, n, h->assign.get() + n0, nullptr, st));
        }
        h->csr_dirty = true;
    }
    h->n += n;
    if (host && sync_host) CK(cudaStreamSynchronize(st));  // the caller may reuse its buffers on return
    return 0;
}

extern "C" int wb_add_with_ids(wb_index* h, int64_t n, const float* x_host, const int64_t* ids_host) {
    return add_common(h, n, x_host, ids_host, true, nullptr, h ? h->stream : nullptr);
}
// ---- pinned, overlapped ingest (FeatureStore shards -> HBM) ------------------------------------------------------
// The loader decodes shard i+1 into one pinned buffer while the copy engine moves shard i out of another and the
// SMs assign its rows to their lists: wb_add_with_ids_pinned enqueues (H2D, norms, ids, IVF assignment) on the
// handle's stream and returns at once; `slot` names the pinned buffer, wb_add_slot_wait(slot) blocks until the GPU has
// finished reading it.  Replaces the synchronous per-batch add of feature_search_index.py:79-82.
extern "C" int wb_pinned_alloc(int64_t bytes, void** out) {
    if (!out || bytes <= 0) return fail("bad arguments");
    *out = nullptr;
    CK(cudaHostAlloc(out, (size_t)bytes, cudaHostAllocDefault));
    return 0;
}
extern "C" int wb_pinned_free(void* p) {
    if (p) CK(cudaFreeHost(p));
    return 0;
}
static int add_pinned(wb_index* h, int64_t n, const float* x_pinned, const int64_t* ids_pinned, const int32_t* preassign,
                      int slot) {
    if (slot < 0 || slot >= wb_index::kAddSlots) return fail("slot %d out of range [0, %d)", slot, wb_index::kAddSlots);
    TRY(set_dev(h));
    if (!h->add_ev[slot]) CK(cudaEventCreateWithFlags(&h->add_ev[slot], cudaEventDisableTiming));
    TRY(add_common(h, n, x_pinned, ids_pinned, true, preassign, h->stream, false));
    CK(cudaEventRecord(h->add_ev[slot], h->stream));
    h->add_pending[slot] = true;
    return 0;
}
extern "C" int wb_add_with_ids_pinned(wb_index* h, int64_t n, const float* x_pinned, const int64_t* ids_pinned, int slot) {
    if (!h) return fail("NULL index");
    return add_pinned(h, n, x_pinned, ids_pinned, nullptr, slot);
}
// Same for rows whose list is already known (faiss.read_index of an IndexIVFFlat file): no coarse quantisation.
extern "C" int wb_ivf_add_preassigned_pinned(wb_index* h, int64_t n, const float* x_pinned, const int64_t* ids_pinned,
                                             const int32_t* assign_pinned, int slot) {
    if (!h || !h->ivf) return fail("not an IVF index");
    if (!assign_pinned) return fail("assign is NULL");
    return add_pinned(h, n, x_pinned, ids_pinned, assign_pinned, slot);
}
extern "C" int wb_add_slot_wait(wb_index* h, int slot) {
    if (!h) return fail("NULL index");
    if (slot < 0 || slot >= wb_index::kAddSlots) return fail("slot %d out of range [0, %d)", slot, wb_index::kAddSlots);
    if (!h->add_pending[slot]) return 0;
    TRY(set_dev(h));
    CK(cudaEventSynchronize(h->add_ev[slot]));
    h->add_pending[slot] = false;
    return 0;
}
extern "C" int wb_sync(wb_index* h) {
    if (!h) return fail("NULL index");
    TRY(set_dev(h));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

extern "C" int wb_add_with_ids_dev(wb_index* h, int64_t n, const float* x_dev, const int64_t* ids_dev, void* stream) {
    return add_common(h, n, x_dev, ids_dev, false, nullptr, (cudaStream_t)stream);
}
extern "C" int wb_ivf_add_preassigned(wb_index* h, int64_t n, const float* x_host, const int64_t* ids_host,
                                      const int32_t* assign_host) {
    if (!h || !h->ivf) return fail("not an IVF index");
    if (!assign_host) return fail("assign is NULL");
    return add_common(h, n, x_host, ids_host, true, assign_host, h->stream);
}

// ---- K5 for batches: list-major scan (ivf_lm.cuh) ------------------------------------------------------------------
// Taken when the probes of the batch overlap enough for shared reads to pay (on average every list is probed at
// least once) and the rows are physically grouped by list.  WB_IVF_LISTMAJOR=0 / 1 forces it off / on.
static int run_ivf_listmajor(wb_index* h, int64_t nq, const float* q_ld, int k, int np, float* D, int64_t* I,
                             cudaStream_t st, const uint32_t* allow, bool* done) {
    *done = false;
    const int mode = env_int("WB_IVF_LISTMAJOR", -1);
    if (mode == 0 || h->slot_row != nullptr || h->n == 0) return 0;
    const int64_t npairs = nq * (int64_t)np;
    if (mode < 0 && (nq < 8 || npairs < h->nlist)) return 0;
    if (npairs >= ((int64_t)1 << 31) || (double)npairs * k * 8.0 > 2e9) return 0;
    ScanCfg c;
    if (plan_scan(h, 8, k, false, 0, &c) != 0 || c.NQ != 8 || !c.single_copy) return 0;
    const int64_t nlist = h->nlist;
    const int64_t max_items = npairs / 8 + nlist + 1;
    TRY(h->lmA.ensure((size_t)npairs * 4));              // list of every (query, probe) pair
    TRY(h->lmB.ensure((size_t)npairs * 4));              // pairs grouped by list
    TRY(h->lmC.ensure((size_t)(nlist + 1) * 8));         // pairs per list (CSR offsets)
    TRY(h->lmD.ensure((size_t)(nlist + 1) * 8));         // work items per list
    TRY(h->lmE.ensure((size_t)(nlist + 1) * 8));         // first work item of every list
    TRY(h->lmF.ensure((size_t)max_items * 4));           // list of every work item
    TRY(h->lmG.ensure((size_t)nq * 4 + 64));             // shared thresholds + the work counter
    TRY(h->parts.ensure((size_t)npairs * k * sizeof(uint64_t)));
    probes_to_pairs_kernel<<<(unsigned)((npairs + 255) / 256), 256, 0, st>>>(h->pI.as<int64_t>(), h->lmA.as<int32_t>(), npairs, k,
                                                                            h->parts.as<uint64_t>());
    CK(cudaGetLastError());
    TRY(device_csr(h, h->lmA.as<int32_t>(), npairs, nullptr, h->lmC.as<int64_t>(), h->lmB.as<uint32_t>(), nullptr, st, false));
    lm_item_count_kernel<<<(unsigned)((nlist + 255) / 256), 256, 0, st>>>(h->lmC.as<int64_t>(), nlist, 8, h->lmD.as<int64_t>());
    CK(cudaGetLastError());
    csr_offsets_kernel<<<1, 1024, 0, st>>>(h->lmD.as<int64_t>(), nlist, h->lmE.as<int64_t>());
    CK(cudaGetLastError());
    lm_item_fill_kernel<<<(unsigned)((nlist + 255) / 256), 256, 0, st>>>(h->lmE.as<int64_t>(), nlist, h->lmF.as<int32_t>());
    CK(cudaGetLastError());
    CK(cudaMemsetAsync(h->lmG.get(), 0, (size_t)nq * 4 + 64, st));
    LmParams p{};
    p.rows = h->rows.get();
    p.ld = h->ld;
    p.queries = q_ld;
    p.nq = (int)nq;
    p.k = k;
    p.P = c.P;
    p.stages = c.stages;
    p.nprobe = np;
    p.nlist = nlist;
    p.list_off = h->list_off.get();
    p.row_pos = h->row_pos.get();
    p.allow = allow;
    p.pl_off = h->lmC.as<int64_t>();
    p.pair_src = h->lmB.as<uint32_t>();
    p.item_off = h->lmE.as<int64_t>();
    p.item_list = h->lmF.as<int32_t>();
    p.gthr = h->lmG.as<uint32_t>();
    p.counter = reinterpret_cast<unsigned int*>(h->lmG.as<unsigned char>() + (size_t)nq * 4 + 16);
    p.parts = h->parts.as<uint64_t>();
    TRY(timing_begin(h, h->timing, st));
    const int grid = (int)std::min<int64_t>(h->sm_count, max_items);
    TRY(with_rw(c.RW, [&](auto RW) { return launch<ivf_listmajor_kernel<8, RW>>(grid, kScanThreads, c.smem, st, p); }));
    TRY(timing_end(h, h->timing, st));
    h->launches += 4;
    TRY(launch_merge_keys(h, nq, k, np, h->parts.as<uint64_t>(), h->ids.get(), D, I, st));
    *done = true;
    return 0;
}

// ---- IVF set-up shared by search and range search ------------------------------------------------------------------
// The lists to probe per query, nprobe clamped to [1, min(nlist, WB_MAX_K)], and the inverted lists made current.
// ensure_csr works on the handle's stream, so rows added on `st` are waited for first.
static int ivf_prepare(wb_index* h, int64_t nprobe, cudaStream_t st, int* np) {
    *np = (int)std::min<int64_t>(std::max<int64_t>(nprobe, 1), std::min<int64_t>(h->nlist, WB_MAX_K));
    if (h->csr_dirty) {
        if (st != h->stream) CK(cudaStreamSynchronize(st));
        TRY(ensure_csr(h));
    }
    return 0;
}

// K4: the coarse quantizer, an exhaustive top-`np` scan of the centroids, into the probe table (h->pD, h->pI).
static int ivf_probes(wb_index* h, int64_t nq, const float* q_ld, int np, cudaStream_t st) {
    TRY(h->pD.ensure((size_t)nq * np * sizeof(float)));
    TRY(h->pI.ensure((size_t)nq * np * sizeof(int64_t)));
    return run_flat_any(h, h->centroids.get(), h->nlist, q_ld, nq, np, nullptr, h->pD.as<float>(), h->pI.as<int64_t>(), st, false);
}

// The fields of a K5 list scan that describe the inverted lists; `allow` as in RowMask.
static ScanParams ivf_scan_params(const wb_index* h, int np, const uint32_t* allow) {
    ScanParams p{};
    p.rows = h->rows.get();
    p.ld = h->ld;
    p.perm = h->slot_row.get();
    p.row_pos = h->row_pos.get();
    p.list_off = h->list_off.get();
    p.nprobe = np;
    p.allow = allow;
    return p;
}

// ---- filters (faiss SearchParameters.sel): a bitmap over insertion positions, DESIGN.md "Filtered search" ---------
struct wb_filter {
    wb_index* h = nullptr;          // the index whose rows the filter selects
    DevPtr<int64_t> set;            // the sorted, unique ids of an id set; null: the range [imin, imax)
    int64_t nset = 0, imin = 0, imax = 0;
    bool invert = false;            // IDSelectorNot
    DevPtr<uint32_t> bits;          // one bit per insertion position
    DevPtr<uint32_t> tile_cnt;      // selected positions per kFilterTile positions (evaluation output)
    int64_t words_cap = 0;          // capacity of `bits`, in 32-bit words (tile_cnt holds words_cap / 4)
    std::vector<int64_t> sel;       // [tiles + 1] selected positions before each tile (host)
    int64_t count = 0;              // selected rows
    int64_t built_n = -1;           // ntotal the bitmap describes; a search after an add re-evaluates it
    DevPtr<float> crows;            // flat sparse path: the selected rows [count, ld] in insertion order ...
    DevPtr<int64_t> cids;           // ... and their ids
    int64_t compact_n = -1;         // built_n the compact copy was made at (-1: none)
};
static_assert(kFilterTile == kGemmBM, "the K2 epoch schedule reads the per-tile counts of the filter evaluation");

// Below this selected fraction a flat search scans a compact copy of the selected rows instead of masking the full
// store.  Measured on a B200 (1000 W, 1965 MHz max SM clock; profiles/filtered/bench_filtered.jsonl, 10M x 768, k 100):
// the mask path costs the unfiltered time (batch 1: 4.05 ms at 1, 1/2 and 1/8 selected vs 4.05 unfiltered); the
// compact path costs about the selected fraction of it (1/64: 0.087 ms at batch 1, 0.40 ms at 16, 2.2 ms at 1024 vs
// 4.05 / 4.34 / 24.6 ms) plus a one-time gather (2.3-2.5 ms at batch 1 for 1/64).  Per search the copy wins at every
// measured fraction; the cutoff bounds the extra memory the copy takes to 1/8 of the store.
constexpr int64_t kSparseCutoffDen = 8;

// Evaluate the selector over the index's current rows (on the handle's stream, one synchronisation to read the
// per-tile counts the host needs for dispatch).
static int filter_eval(wb_filter* f) {
    wb_index* h = f->h;
    cudaStream_t st = h->stream;
    const int64_t n = h->n, ntiles = (n + kFilterTile - 1) / kFilterTile;
    const int64_t words = ntiles * (kFilterTile / 32);
    if (words > f->words_cap) {
        const int64_t cap = std::max<int64_t>(words, (std::max<int64_t>(h->cap, n) + kFilterTile - 1) / kFilterTile *
                                                         (kFilterTile / 32));
        DevPtr<uint32_t> bits, cnt;
        CK(dev_alloc(&bits, (size_t)cap * 4));
        CK(dev_alloc(&cnt, (size_t)cap / (kFilterTile / 32) * 4));
        f->bits = std::move(bits);
        f->tile_cnt = std::move(cnt);
        f->words_cap = cap;
    }
    std::vector<uint32_t> cnt((size_t)ntiles);
    if (n > 0) {
        filter_eval_kernel<<<(unsigned)ntiles, kFilterTile, 0, st>>>(h->ids.get(), n, f->set.get(), f->nset, f->imin,
                                                                    f->imax, f->invert, f->bits.get(), f->tile_cnt.get());
        CK(cudaGetLastError());
        h->launches++;
        CK(cudaMemcpyAsync(cnt.data(), f->tile_cnt.get(), (size_t)ntiles * 4, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
    }
    f->sel.assign((size_t)ntiles + 1, 0);
    for (int64_t t = 0; t < ntiles; ++t) f->sel[t + 1] = f->sel[t] + cnt[t];
    f->count = f->sel[ntiles];
    f->built_n = n;
    f->crows.reset();
    f->cids.reset();
    f->compact_n = -1;
    return 0;
}

// Bring the bitmap up to date with rows added since it was evaluated.  An add on `st` may still be writing the ids:
// `st` is synchronised first (this is the one synchronisation a _dev search with a stale filter makes).
static int filter_current(wb_filter* f, cudaStream_t st) {
    if (f->built_n == f->h->n) return 0;
    if (st != f->h->stream) CK(cudaStreamSynchronize(st));
    return filter_eval(f);
}

// Flat sparse path: the selected rows gathered, in insertion order, into [count, ld] with their ids, so that index
// order in the copy is insertion order and ties resolve as in the full store.  Built once per evaluation (repeated
// searches with one filter pay for it once).  *ok = false when it does not fit in memory: the caller masks instead.
static int filter_compact(wb_filter* f, bool* ok) {
    *ok = true;
    if (f->compact_n == f->built_n) return 0;
    wb_index* h = f->h;
    cudaStream_t st = h->stream;
    const int64_t m = f->count, ntiles = (int64_t)f->sel.size() - 1;
    DevPtr<float> rows;
    DevPtr<int64_t> ids, pos, off;
    if (dev_alloc(&rows, (size_t)m * h->ld * 4) != cudaSuccess || dev_alloc(&ids, (size_t)m * 8) != cudaSuccess ||
        dev_alloc(&pos, (size_t)m * 8) != cudaSuccess || dev_alloc(&off, (size_t)(ntiles + 1) * 8) != cudaSuccess) {
        cudaGetLastError();  // (clear the allocation error: the next launch check would report it)
        *ok = false;
        return 0;
    }
    CK(cudaMemcpyAsync(off.get(), f->sel.data(), (size_t)(ntiles + 1) * 8, cudaMemcpyHostToDevice, st));
    filter_positions_kernel<<<(unsigned)ntiles, kFilterTile, 0, st>>>(f->bits.get(), h->n, off.get(), h->ids.get(),
                                                                     pos.get(), ids.get());
    CK(cudaGetLastError());
    const int64_t tot = m * h->ld;  // whole rows, padding columns included: the copy has the store's stride
    gather_rows_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(h->rows.get(), h->ld, h->ld, pos.get(), m, rows.get());
    CK(cudaGetLastError());
    h->launches += 2;
    CK(cudaStreamSynchronize(st));  // a search on another stream reads the copy next; `off` and `pos` are freed on return
    f->crows = std::move(rows);
    f->cids = std::move(ids);
    f->compact_n = f->built_n;
    return 0;
}

static int check_filter(const wb_index* h, const wb_filter* f) {
    if (f && f->h != h) return fail("the filter was created for another index");
    return 0;
}

// The rows a search scans: without a filter the whole store.  With filter `f`, once it is current: nothing (`none`),
// the compact copy of its rows (a flat store of which fewer than 1/kSparseCutoffDen are selected, when the copy fits in
// memory) or the store under its bitmap (`mask`).
struct RowSel {
    bool none;
    const float* rows;
    int64_t nrows;
    const int64_t* ids;
    RowMask mask;  // mask.allow null: every row of `rows`
    const RowMask* masked() const { return mask.allow ? &mask : nullptr; }
};

static int select_rows(wb_index* h, wb_filter* f, cudaStream_t st, RowSel* s) {
    *s = RowSel{false, h->rows.get(), h->n, h->ids.get(), RowMask{}};
    if (!f) return 0;
    TRY(filter_current(f, st));
    if (f->count == 0) {
        s->none = true;
        return 0;
    }
    if (!h->ivf && f->count * kSparseCutoffDen < h->n) {
        bool ok = false;
        TRY(filter_compact(f, &ok));
        if (ok) {
            s->rows = f->crows.get();
            s->nrows = f->count;
            s->ids = f->cids.get();
            return 0;
        }
    }
    s->mask = RowMask{f->bits.get(), f->sel.data()};
    return 0;
}

// ---- search --------------------------------------------------------------------------------
constexpr int64_t kIvfFuseCoarseMaxQ = 4;  // largest IVF batch that runs the coarse quantizer inside the list-scan launch

// Every search entry point ends here.  `f` (may be null) restricts the result to the rows it selects.
static int search_dev_impl(wb_index* h, wb_filter* f, int64_t nq, const float* q_ld /* [nq, ld] */, int64_t k,
                           int64_t nprobe, float* D, int64_t* I, cudaStream_t st, const ExchParams* ex = nullptr,
                           bool* exchanged = nullptr) {
    if (exchanged) *exchanged = false;
    if (h->ivf && !h->trained) return fail("IndexIVFFlat is not trained");
    RowSel s;
    TRY(select_rows(h, f, st, &s));
    if (s.none) {  // all padding; a sharded search still takes part in the exchange (*exchanged stays false)
        const int64_t tot = nq * k;
        pad_results_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(D, I, tot);
        CK(cudaGetLastError());
        h->launches++;
        return 0;
    }
    if (!h->ivf) return run_flat_any(h, s.rows, s.nrows, q_ld, nq, (int)k, s.ids, D, I, st, true, ex, exchanged, s.masked());
    int np = 0;
    TRY(ivf_prepare(h, nprobe, st, &np));
    // K5 plan: gather-scan of the probed lists, S CTAs per query
    ScanCfg c;
    TRY(plan_scan(h, 1, (int)k, true, np, &c));
    const int64_t S = ivf_ctas(h, nq);
    if (ex && nq > kMaxGridY) ex = nullptr;
    int S_merge = 0, heads_bytes = 0;
    const bool fuse = tail_fusable(c, (int)k, S, ex ? ex->world : 1, &S_merge, &heads_bytes);
    // K4 + K5 in one launch (coarse.cuh): a few queries, every CTA resident, the selection scratch fits the idle ring
    const size_t ring_bytes = (size_t)c.stages * kConsumerWarps * c.RW * c.ck * 4;
    bool fuse_coarse = fuse && h->coop_ok && nq <= kIvfFuseCoarseMaxQ && S * nq <= h->sm_count &&
                       h->nlist < ((int64_t)1 << 30) && coarse_smem_layout(h->nlist, np).total <= ring_bytes &&
                       env_int("WB_IVF_FUSE_COARSE", 1) && env_int("WB_IVF_LISTMAJOR", -1) != 1;
    for (int attempt = 0; attempt < 2; ++attempt) {
        if (!fuse_coarse) {
            TRY(ivf_probes(h, nq, q_ld, np, st));
            // K5, batches: list-major - the probe table is inverted on the device and every probed list is streamed once
            // per group of 8 of the queries that probe it (ivf_lm.cuh)
            bool done = false;
            TRY(run_ivf_listmajor(h, nq, q_ld, (int)k, np, D, I, st, s.mask.allow, &done));
            if (done) return 0;
        }
        TRY(h->parts.ensure((size_t)nq * S * k * sizeof(uint64_t)));
        ScanParams p = ivf_scan_params(h, np, s.mask.allow);
        p.k = (int)k;
        p.nparts = (int)S;
        if (fuse) {
            TRY(ensure_tail_counters(h, st));
            set_tail(p, h, c, S_merge, heads_bytes, h->ids.get(), ex ? ex->D : D, ex ? ex->I : I, (int)k, ex);
        }
        if (fuse_coarse) {
            TRY(h->ckeys.ensure((size_t)nq * h->nlist * sizeof(uint32_t)));
            p.centroids = h->centroids.get();
            p.nlist = h->nlist;
            p.coarse_keys = h->ckeys.as<uint32_t>();
            p.coarse_count = h->tailcnt.as<unsigned int>() + 2 * kMaxGridY;
            p.queries = q_ld;
            p.nq = (int)nq;
            p.parts = h->parts.as<uint64_t>();
            TRY(timing_begin(h, h->timing, st));
            const cudaError_t e = launch_scan_coop(c, p, dim3((unsigned)S, (unsigned)nq), st);
            if (e != cudaSuccess) {
                // (a partitioned device can refuse a full-width cooperative grid: two launches from now on)
                cudaGetLastError();
                h->coop_ok = false;
                fuse_coarse = false;
                continue;
            }
            TRY(timing_end(h, h->timing, st));
            h->launches++;
            h->coarse_fused++;
            if (ex && exchanged) *exchanged = true;
            return 0;
        }
        return run_scan_groups(h, c, true, p, nq, q_ld, h->ids.get(), D, I, st, true, ex, exchanged);
    }
    return fail("unreachable");
}

// ---- multi-GPU exchange over peer memory ----------------------------------------------------------
struct wb_exchange {
    int device = 0, rank = 0, world = 1;
    size_t region_bytes = 0, flags_bytes = 0, cap_entries = 0, nq_cap = 0, total_bytes = 0;
    DevPtr<unsigned char> local;
    unsigned char* peers[kExchMaxWorld] = {};
    bool opened[kExchMaxWorld] = {};
    uint32_t seq = 0;       // sequence number of the last exchange that was LAUNCHED (all ranks advance in lockstep)
    PinPtr<int> status;     // pinned (device-visible) host word raised by a kernel whose wait for the peers timed out
    int64_t launches = 0;   // exchange_merge_kernel launches (the fused path needs none)
};

extern "C" int wb_exch_create(int device, int rank, int world, int64_t max_queries, int64_t max_entries,
                              wb_exchange** out) {
    if (!out) return fail("out is NULL");
    *out = nullptr;
    if (world < 1 || world > kExchMaxWorld || rank < 0 || rank >= world) return fail("bad rank/world %d/%d", rank, world);
    if (max_queries < 1 || max_entries < max_queries) return fail("bad exchange capacity");
    CK(cudaSetDevice(device));
    std::unique_ptr<wb_exchange> ex(new wb_exchange());
    ex->device = device;
    ex->rank = rank;
    ex->world = world;
    ex->nq_cap = (size_t)max_queries;
    ex->cap_entries = ((size_t)max_entries + 3) & ~(size_t)3;
    ex->flags_bytes = ((size_t)max_queries * 4 + 255) & ~(size_t)255;
    ex->region_bytes = (ex->flags_bytes + ex->cap_entries * 12 + 255) & ~(size_t)255;
    ex->total_bytes = ex->region_bytes * 2 * world;
    CK(dev_alloc(&ex->local, ex->total_bytes));
    CK(cudaMemset(ex->local.get(), 0, ex->total_bytes));
    int* status = nullptr;
    CK(cudaHostAlloc(&status, sizeof(int), cudaHostAllocMapped | cudaHostAllocPortable));
    ex->status.reset(status);
    *status = 0;
    CK(cudaDeviceSynchronize());
    ex->peers[rank] = ex->local.get();
    *out = ex.release();
    return 0;
}

extern "C" int wb_exch_local_handle(wb_exchange* ex, void* handle64) {
    if (!ex || !handle64) return fail("NULL argument");
    CK(cudaSetDevice(ex->device));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    cudaIpcMemHandle_t hnd;
    CK(cudaIpcGetMemHandle(&hnd, ex->local.get()));
    memcpy(handle64, &hnd, 64);
    return 0;
}

extern "C" int wb_exch_open_peers(wb_exchange* ex, const void* handles /* [world][64] */) {
    if (!ex || !handles) return fail("NULL argument");
    CK(cudaSetDevice(ex->device));
    for (int r = 0; r < ex->world; ++r) {
        if (r == ex->rank) continue;
        cudaIpcMemHandle_t hnd;
        memcpy(&hnd, (const char*)handles + (size_t)r * 64, 64);
        void* ptr = nullptr;
        CK(cudaIpcOpenMemHandle(&ptr, hnd, cudaIpcMemLazyEnablePeerAccess));
        ex->peers[r] = (unsigned char*)ptr;
        ex->opened[r] = true;
    }
    return 0;
}

extern "C" int wb_exch_free(wb_exchange* ex) {
    if (!ex) return 0;
    cudaSetDevice(ex->device);
    cudaDeviceSynchronize();
    for (int r = 0; r < ex->world; ++r)
        if (ex->opened[r]) cudaIpcCloseMemHandle(ex->peers[r]);
    delete ex;
    return 0;
}

// Parameters of the NEXT exchange (sequence number ex->seq + 1).  The caller commits the sequence number with
// exch_commit() only after the kernel that carries these parameters has been launched successfully: a rank whose
// launch failed must not drift out of lockstep with its peers.
static int exch_prepare(wb_exchange* ex, int64_t nq, int64_t k, float* D_dev, int64_t* I_dev, ExchParams* out) {
    if (!ex) return fail("NULL exchange");
    if (k < 1 || k > WB_MAX_K) return fail("k=%lld out of range [1, %d]", (long long)k, WB_MAX_K);
    if (nq < 1 || (size_t)nq > ex->nq_cap || (size_t)(nq * k) > ex->cap_entries)
        return fail("exchange capacity exceeded (nq=%lld, k=%lld)", (long long)nq, (long long)k);
    for (int r = 0; r < ex->world; ++r)
        if (!ex->peers[r]) return fail("peer %d is not mapped: call wb_exch_open_peers first", r);
    ExchParams p{};
    p.rank = ex->rank;
    p.world = ex->world;
    p.nq = nq;
    p.k = (int)k;
    p.S = merge_buffer_entries((int)k, ex->world);
    p.seq = ex->seq + 1;
    if (p.seq == 0) p.seq = 1;
    for (int r = 0; r < ex->world; ++r) p.mailbox[r] = ex->peers[r];
    p.region_bytes = ex->region_bytes;
    p.flags_bytes = ex->flags_bytes;
    p.cap_entries = ex->cap_entries;
    p.D = D_dev;
    p.I = I_dev;
    p.status = ex->status.get();
    *out = p;
    return 0;
}
static void exch_commit(wb_exchange* ex, const ExchParams& p) { ex->seq = p.seq; }

static int launch_exchange_kernel(wb_exchange* ex, ExchParams& p, const float* D_local, const int64_t* I_local,
                                  cudaStream_t st) {
    p.D_local = D_local;
    p.I_local = I_local;
    p.S = merge_buffer_entries(p.k, p.world);
    CK(smem_optin<exchange_merge_kernel>(8192 * 8));
    int sms = 148;
    CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ex->device));
    const unsigned grid = (unsigned)std::min<int64_t>(p.nq, sms);  // one resident CTA per SM at most (1024 threads)
    exchange_merge_kernel<<<grid, kMergeThreads, (size_t)p.S * 8, st>>>(p);
    CK(cudaGetLastError());
    exch_commit(ex, p);
    ex->launches++;
    return 0;
}

// Global top-k from this rank's local (D, I): one kernel does the NVLink exchange and the merge.
// Every rank must call this the same number of times with the same nq and k.
extern "C" int wb_exch_merge_dev(wb_exchange* ex, int64_t nq, int64_t k, const float* D_local_dev,
                                 const int64_t* I_local_dev, float* D_dev, int64_t* I_dev, void* stream) {
    ExchParams p;
    TRY(exch_prepare(ex, nq, k, D_dev, I_dev, &p));
    CK(cudaSetDevice(ex->device));
    return launch_exchange_kernel(ex, p, D_local_dev, I_local_dev, (cudaStream_t)stream);
}

// 1 when a kernel of this exchange gave up waiting for a peer (a rank that never launched): the results of that
// search are invalid.  The word lives in pinned host memory that the kernels write through; it is current for every
// kernel the caller has synchronised with.
extern "C" int64_t wb_exch_launch_count(const wb_exchange* ex) { return ex ? ex->launches : -1; }

extern "C" int wb_exch_status(wb_exchange* ex, int* timed_out) {
    if (!ex || !timed_out) return fail("NULL argument");
    *timed_out = *reinterpret_cast<volatile int*>(ex->status.get());
    return 0;
}

// Search over a row-sharded index, device buffers: local search + NVLink exchange + merge.  Batches that run the
// scan kernel (flat batch <= 4, every IVF list scan) do all of it in ONE launch (scan.cuh, fused tail); the others
// run the local search and then exchange_merge_kernel.  Every rank calls it with the same queries.
static int exch_search_dev_impl(wb_index* h, wb_exchange* ex, wb_filter* f, int64_t nq, const float* q_ld, int64_t k,
                                int64_t nprobe, float* D_dev, int64_t* I_dev, cudaStream_t st) {
    if (ex->device != h->device) return fail("index and exchange live on different devices");
    ExchParams p;
    TRY(exch_prepare(ex, nq, k, D_dev, I_dev, &p));
    TRY(h->dbuf.ensure((size_t)nq * k * sizeof(float)));
    TRY(h->ibuf.ensure((size_t)nq * k * sizeof(int64_t)));
    bool exchanged = false;
    TRY(search_dev_impl(h, f, nq, q_ld, k, nprobe, h->dbuf.as<float>(), h->ibuf.as<int64_t>(), st, &p, &exchanged));
    if (exchanged) {
        exch_commit(ex, p);
        return 0;
    }
    return launch_exchange_kernel(ex, p, h->dbuf.as<float>(), h->ibuf.as<int64_t>(), st);
}

// ---- search entry points -------------------------------------------------------------------
static int check_search_args(const wb_index* h, int64_t nq, const void* q, int64_t k, const void* D, const void* I) {
    if (!h) return fail("NULL index");
    if (nq < 0) return fail("negative nq");
    if (k < 1 || k > WB_MAX_K) return fail("k=%lld out of range [1, %d]", (long long)k, WB_MAX_K);
    if (nq > 0 && (!q || !D || !I)) return fail("NULL buffer");
    return 0;
}

constexpr size_t kPinStageMax = (size_t)4 << 20;  // larger transfers are bandwidth-bound anyway: copy them directly

// The scan, list-major, SS-image and re-scoring kernels load query rows 16 bytes at a time, and the assignment GEMM
// maps the points with TMA (16-byte base): a caller's device buffer goes to them as is only when it is 16-byte
// aligned.  The C API asks for no more than the alignment of a float, so other buffers are staged like padded ones.
static bool aligned16(const void* p) { return ((uintptr_t)p & 15) == 0; }

// queries arrive with row stride d; the kernels want stride ld
static int stage_queries(wb_index* h, int64_t nq, const float* q, bool host, cudaStream_t st, const float** out) {
    if (!host && h->ld == h->d && aligned16(q)) {
        *out = q;
        return 0;
    }
    const size_t qbytes = (size_t)nq * h->d * sizeof(float);
    if (host && qbytes <= kPinStageMax) {  // pageable -> pinned (host memcpy) -> device (async)
        PinBuf& pb = h->pin_q;
        TRY(pb.ensure(qbytes));
        memcpy(pb.get(), q, qbytes);
        q = reinterpret_cast<const float*>(pb.get());
    }
    TRY(h->qbuf.ensure((size_t)nq * h->ld * sizeof(float)));
    if (h->ld == h->d) {  // (device queries get here only when unaligned: a copy takes any alignment)
        CK(cudaMemcpyAsync(h->qbuf.get(), q, qbytes, host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, st));
    } else {
        const float* src = q;
        if (host) {
            TRY(h->xbuf.ensure(qbytes));
            CK(cudaMemcpyAsync(h->xbuf.get(), q, qbytes, cudaMemcpyHostToDevice, st));
            src = h->xbuf.as<float>();
        }
        const int64_t tot = nq * h->ld;
        pad_rows_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(src, h->qbuf.as<float>(), nq, h->d, h->ld);
        CK(cudaGetLastError());
        h->launches++;
    }
    *out = h->qbuf.as<float>();
    return 0;
}

// (D, I) device -> caller's host buffers, then ONE synchronisation of the stream.
// `word_dev` (optional): one more device int fetched with the results (the exchange's time-out flag), so that reading
// it costs no synchronisation of its own.
static int fetch_results(wb_index* h, int64_t nq, int64_t k, const float* D_dev, const int64_t* I_dev, float* D_host,
                         int64_t* I_host, cudaStream_t st) {
    const size_t dbytes = (size_t)nq * k * sizeof(float), ibytes = (size_t)nq * k * sizeof(int64_t);
    PinBuf& pb = h->pin_o;
    if (dbytes + ibytes <= kPinStageMax) {
        TRY(pb.ensure(dbytes + ibytes));
        unsigned char* stage = reinterpret_cast<unsigned char*>(pb.get());
        CK(cudaMemcpyAsync(stage, I_dev, ibytes, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(stage + ibytes, D_dev, dbytes, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        memcpy(I_host, stage, ibytes);
        memcpy(D_host, stage + ibytes, dbytes);
    } else {
        CK(cudaMemcpyAsync(D_host, D_dev, dbytes, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(I_host, I_dev, ibytes, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
    }
    return 0;
}

// Runs `search(D, I)`, which enqueues a search on `st`, and delivers its results to the caller's host buffers.
// Small result sets skip the device buffer and its two D2H copies: the kernel that emits the final (D, I) rows writes
// them straight into the pinned staging buffer (a few KB of posted PCIe writes), which the host reads after the
// stream synchronisation.  At one query this takes ~10 us off a 60 us IVF call.  Larger ones go through
// (D_dev, I_dev) and fetch_results.
constexpr size_t kDirectResultMax = (size_t)64 << 10;
template <class Search>
static int search_to_host(wb_index* h, int64_t nq, int64_t k, DevBuf& D_dev, DevBuf& I_dev, float* D_host, int64_t* I_host,
                          cudaStream_t st, const Search& search) {
    const size_t dbytes = (size_t)nq * k * sizeof(float), ibytes = (size_t)nq * k * sizeof(int64_t);
    if (dbytes + ibytes <= kDirectResultMax && env_int("WB_DIRECT_RESULTS", 1)) {
        TRY(h->pin_o.ensure(dbytes + ibytes));
        int64_t* I_pin = h->pin_o.as<int64_t>();
        float* D_pin = reinterpret_cast<float*>(h->pin_o.as<unsigned char>() + ibytes);
        TRY(search(D_pin, I_pin));
        CK(cudaStreamSynchronize(st));
        memcpy(I_host, I_pin, ibytes);
        memcpy(D_host, D_pin, dbytes);
        return 0;
    }
    TRY(D_dev.ensure(dbytes));
    TRY(I_dev.ensure(ibytes));
    TRY(search(D_dev.as<float>(), I_dev.as<int64_t>()));
    return fetch_results(h, nq, k, D_dev.as<float>(), I_dev.as<int64_t>(), D_host, I_host, st);
}

// With an exchange `ex` (may be null) the search runs over a row-sharded index: every rank calls it with the same
// queries, and (D, I) receive the global result.
static int search_dev_entry(wb_index* h, wb_exchange* ex, wb_filter* f, int64_t nq, const float* q_dev, int64_t k,
                            int64_t nprobe, float* D_dev, int64_t* I_dev, void* stream) {
    TRY(check_search_args(h, nq, q_dev, k, D_dev, I_dev));
    TRY(check_filter(h, f));
    if (nq == 0) return 0;
    TRY(set_dev(h));
    cudaStream_t st = (cudaStream_t)stream;
    const float* q = nullptr;
    TRY(stage_queries(h, nq, q_dev, false, st, &q));
    if (ex) return exch_search_dev_impl(h, ex, f, nq, q, k, nprobe, D_dev, I_dev, st);
    return search_dev_impl(h, f, nq, q, k, nprobe, D_dev, I_dev, st);
}

// Host buffers: H2D of the queries, the search (with `ex`: local search, NVLink exchange + merge), D2H of (D, I) - one
// call, one stream, one synchronisation.
static int search_host_entry(wb_index* h, wb_exchange* ex, wb_filter* f, int64_t nq, const float* q_host, int64_t k,
                             int64_t nprobe, float* D_host, int64_t* I_host) {
    TRY(check_search_args(h, nq, q_host, k, D_host, I_host));
    TRY(check_filter(h, f));
    if (nq == 0) return 0;
    TRY(set_dev(h));
    cudaStream_t st = h->stream;
    const float* q = nullptr;
    TRY(stage_queries(h, nq, q_host, true, st, &q));
    if (!ex)
        return search_to_host(h, nq, k, h->dbuf, h->ibuf, D_host, I_host, st, [&](float* D, int64_t* I) {
            return search_dev_impl(h, f, nq, q, k, nprobe, D, I, st);
        });
    // (eD, eI): exch_search_dev_impl keeps this rank's local results in (dbuf, ibuf)
    TRY(search_to_host(h, nq, k, h->eD, h->eI, D_host, I_host, st, [&](float* D, int64_t* I) {
        return exch_search_dev_impl(h, ex, f, nq, q, k, nprobe, D, I, st);
    }));
    if (*reinterpret_cast<volatile int*>(ex->status.get())) return fail("sharded search: a peer GPU did not join the exchange within 20 s (results invalid)");
    return 0;
}

extern "C" int wb_search_dev(wb_index* h, int64_t nq, const float* q_dev, int64_t k, int64_t nprobe, float* D_dev,
                             int64_t* I_dev, void* stream) {
    return wb_search_filtered_dev(h, nullptr, nq, q_dev, k, nprobe, D_dev, I_dev, stream);
}
extern "C" int wb_search(wb_index* h, int64_t nq, const float* q_host, int64_t k, int64_t nprobe, float* D_host,
                         int64_t* I_host) {
    return wb_search_filtered(h, nullptr, nq, q_host, k, nprobe, D_host, I_host);
}
extern "C" int wb_search_filtered_dev(wb_index* h, wb_filter* f, int64_t nq, const float* q_dev, int64_t k, int64_t nprobe,
                                      float* D_dev, int64_t* I_dev, void* stream) {
    return search_dev_entry(h, nullptr, f, nq, q_dev, k, nprobe, D_dev, I_dev, stream);
}
extern "C" int wb_search_filtered(wb_index* h, wb_filter* f, int64_t nq, const float* q_host, int64_t k, int64_t nprobe,
                                  float* D_host, int64_t* I_host) {
    return search_host_entry(h, nullptr, f, nq, q_host, k, nprobe, D_host, I_host);
}
extern "C" int wb_exch_search_dev(wb_index* h, wb_exchange* ex, int64_t nq, const float* q_dev, int64_t k, int64_t nprobe,
                                  float* D_dev, int64_t* I_dev, void* stream) {
    return wb_exch_search_filtered_dev(h, ex, nullptr, nq, q_dev, k, nprobe, D_dev, I_dev, stream);
}
extern "C" int wb_exch_search(wb_index* h, wb_exchange* ex, int64_t nq, const float* q_host, int64_t k, int64_t nprobe,
                              float* D_host, int64_t* I_host) {
    return wb_exch_search_filtered(h, ex, nullptr, nq, q_host, k, nprobe, D_host, I_host);
}
extern "C" int wb_exch_search_filtered_dev(wb_index* h, wb_exchange* ex, wb_filter* f, int64_t nq, const float* q_dev,
                                           int64_t k, int64_t nprobe, float* D_dev, int64_t* I_dev, void* stream) {
    if (!ex) return fail("NULL exchange");
    return search_dev_entry(h, ex, f, nq, q_dev, k, nprobe, D_dev, I_dev, stream);
}
extern "C" int wb_exch_search_filtered(wb_index* h, wb_exchange* ex, wb_filter* f, int64_t nq, const float* q_host,
                                       int64_t k, int64_t nprobe, float* D_host, int64_t* I_host) {
    if (!ex) return fail("NULL exchange");
    return search_host_entry(h, ex, f, nq, q_host, k, nprobe, D_host, I_host);
}

// ---- in-process shard group (DESIGN.md "Shard group") ------------------------------------------------------------
// A host thread of a group: runs a non-root shard's search when that search synchronises its stream (K2 reads its
// overflow flag), so that the shards' searches overlap instead of running one GPU at a time.
struct GroupWorker {
    std::mutex mu;
    std::condition_variable cv;
    std::function<int()> job;
    bool busy = false, quit = false;
    int rc = 0;
    std::string err;
    std::thread th;  // declared last: the thread starts once the members above exist

    GroupWorker() : th([this] { loop(); }) {}
    ~GroupWorker() {
        {
            std::lock_guard<std::mutex> lk(mu);
            quit = true;
        }
        cv.notify_all();
        th.join();
    }
    void loop() {
        std::unique_lock<std::mutex> lk(mu);
        for (;;) {
            cv.wait(lk, [&] { return quit || (bool)job; });
            if (quit) return;
            std::function<int()> j = std::move(job);
            job = nullptr;
            lk.unlock();
            const int r = j();
            lk.lock();
            rc = r;
            err = r ? g_err : std::string();  // g_err is per thread: hand the message to the caller
            busy = false;
            cv.notify_all();
        }
    }
    void post(std::function<int()> j) {
        std::lock_guard<std::mutex> lk(mu);
        job = std::move(j);
        busy = true;
        cv.notify_all();
    }
    int wait() {
        std::unique_lock<std::mutex> lk(mu);
        cv.wait(lk, [&] { return !busy; });
        if (rc) g_err = err;
        return rc;
    }
};

struct wb_group {
    std::vector<wb_index*> shards;                      // [s] on its own GPU; [0] is the root
    bool p2p = true;                                    // every ordered pair of the GPUs has peer access
    std::vector<wb_exchange*> ex;                       // [s]: rank s of the group's exchange (p2p only)
    std::vector<std::unique_ptr<GroupWorker>> workers;  // [s >= 1]
    std::vector<DevBuf> qpeer;                          // [s >= 1]: the _dev queries, copied from the root
    std::vector<EventPtr> ev;                           // [0]: the caller's stream reached the call; [s]: shard s's copies
    DevBuf pD, pI;                                      // fallback merge: the shards' local results on the root, [n][nq][k]

    ~wb_group() {
        workers.clear();
        for (size_t s = 0; s < shards.size(); ++s) {
            cudaSetDevice(shards[s]->device);
            if (s < ex.size()) wb_exch_free(ex[s]);  // waits for the device
            if (s < qpeer.size()) qpeer[s].mem.reset();
            if (s < ev.size()) ev[s].reset();
        }
        if (!shards.empty()) cudaSetDevice(shards[0]->device);
    }
};

extern "C" int wb_group_create(int n, wb_index* const* shards, int64_t max_queries, int64_t max_entries, wb_group** out) {
    if (!out) return fail("out is NULL");
    *out = nullptr;
    if (n < 1 || n > kExchMaxWorld) return fail("a group holds 1 to %d shards (got %d)", kExchMaxWorld, n);
    if (!shards) return fail("NULL shards");
    for (int s = 0; s < n; ++s) {
        const wb_index* h = shards[s];
        if (!h) return fail("shard %d is NULL", s);
        if (h->ivf != shards[0]->ivf || h->d != shards[0]->d || h->nlist != shards[0]->nlist)
            return fail("shard %d differs from shard 0 in kind, d or nlist", s);
        for (int r = 0; r < s; ++r)
            if (shards[r]->device == h->device) return fail("shards %d and %d are both on GPU %d", r, s, h->device);
    }
    if (shards[0]->ivf) {  // every shard must probe the same lists: identical centroids, bit for bit
        const size_t row = (size_t)shards[0]->d * sizeof(float), bytes = (size_t)shards[0]->nlist * row;
        std::vector<unsigned char> c0(bytes), cs(bytes);
        for (int s = 0; s < n; ++s) {
            TRY(set_dev(shards[s]));
            CK(cudaStreamSynchronize(shards[s]->stream));
            CK(cudaMemcpy2D(s ? cs.data() : c0.data(), row, shards[s]->centroids.get(), (size_t)shards[s]->ld * sizeof(float),
                            row, (size_t)shards[0]->nlist, cudaMemcpyDeviceToHost));
            if (s && memcmp(c0.data(), cs.data(), bytes) != 0) return fail("shard %d has other centroids than shard 0", s);
        }
    }
    std::unique_ptr<wb_group> g(new wb_group());
    g->shards.assign(shards, shards + n);
    for (int s = 0; s < n; ++s)
        for (int r = 0; r < n; ++r) {
            if (r == s) continue;
            int can = 0;
            CK(cudaDeviceCanAccessPeer(&can, shards[s]->device, shards[r]->device));
            if (!can) {
                g->p2p = false;
                continue;
            }
            TRY(set_dev(shards[s]));
            const cudaError_t e = cudaDeviceEnablePeerAccess(shards[r]->device, 0);
            if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
            else CK(e);
        }
    g->qpeer.resize(n);
    g->ev.resize(n);
    g->workers.resize(n);
    for (int s = 0; s < n; ++s) {
        TRY(set_dev(shards[s]));
        cudaEvent_t e = nullptr;
        CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        g->ev[s].reset(e);
        if (s) {
            try {
                g->workers[s].reset(new GroupWorker());
            } catch (const std::exception& ex) {  // std::system_error when no thread can be started
                return fail("group: could not start a host thread for shard %d: %s", s, ex.what());
            }
        }
    }
    if (g->p2p && n > 1) {  // the mailboxes of the exchange are plain device pointers of the peers
        for (int s = 0; s < n; ++s) {
            wb_exchange* ex = nullptr;
            TRY(wb_exch_create(shards[s]->device, s, n, max_queries, max_entries, &ex));
            g->ex.push_back(ex);
        }
        for (int s = 0; s < n; ++s)
            for (int r = 0; r < n; ++r) g->ex[s]->peers[r] = g->ex[r]->local.get();
    }
    TRY(set_dev(shards[0]));
    *out = g.release();
    return 0;
}

extern "C" int wb_group_free(wb_group* g) {
    delete g;
    return 0;
}

// Shard s's part of an exchange.  A shard whose search fails before it has launched its part joins the exchange with
// padding, so that the shards already launched are not left waiting and every rank keeps its place in the sequence.
static int group_exch_part(wb_index* h, wb_exchange* ex, wb_filter* f, int64_t nq, const float* q, int64_t k,
                           int64_t nprobe, float* D, int64_t* I, cudaStream_t st) {
    const uint32_t seq0 = ex->seq;
    int rc = set_dev(h);
    if (rc == 0) rc = exch_search_dev_impl(h, ex, f, nq, q, k, nprobe, D, I, st);
    if (rc != 0 && ex->seq == seq0) {
        const std::string err = g_err;
        ExchParams p;
        if (cudaSetDevice(h->device) == cudaSuccess && exch_prepare(ex, nq, k, D, I, &p) == 0) {
            pad_results_kernel<<<(unsigned)((nq * k + 255) / 256), 256, 0, st>>>(h->dbuf.as<float>(), h->ibuf.as<int64_t>(),
                                                                              nq * k);
            launch_exchange_kernel(ex, p, h->dbuf.as<float>(), h->ibuf.as<int64_t>(), st);
        }
        g_err = err;
    }
    return rc;
}

// Batches above this may run K2 (flat search, or the coarse step of IVF), which synchronises its stream: they run each
// non-root shard on a host thread.  Smaller ones never synchronise and are enqueued from the calling thread.
constexpr int64_t kGroupInlineMaxQ = 4;

// Search of a group: `host` says whether q / D / I are host buffers (else device buffers of the root, ordered on
// `caller`).  Every shard gets the queries on its own stream (the root: `caller`, or its own for host buffers), then
// either every shard searches with the exchange in its tail (root: into D / I) or, when the mailbox is too small or a
// pair of GPUs has no peer access, every shard searches locally, copies its result to the root and the root merges.
static int group_search(wb_group* g, wb_filter* const* filters, int64_t nq, const float* q, bool host, int64_t k,
                        int64_t nprobe, float* D, int64_t* I, cudaStream_t caller) {
    if (!g) return fail("NULL group");
    const int n = (int)g->shards.size();
    wb_index* h0 = g->shards[0];
    auto filt = [&](int s) { return filters ? filters[s] : nullptr; };
    if (n == 1)
        return host ? search_host_entry(h0, nullptr, filt(0), nq, q, k, nprobe, D, I)
                    : search_dev_entry(h0, nullptr, filt(0), nq, q, k, nprobe, D, I, caller);
    // every check and allocation comes before the first launch: an argument error leaves no shard waiting
    for (int s = 0; s < n; ++s) {
        TRY(check_search_args(g->shards[s], nq, q, k, D, I));
        TRY(check_filter(g->shards[s], filt(s)));
        if (g->shards[s]->ivf && !g->shards[s]->trained) return fail("IndexIVFFlat is not trained");
    }
    if (nq == 0) return 0;
    const bool exch = g->p2p && (size_t)nq <= g->ex[0]->nq_cap && (size_t)(nq * k) <= g->ex[0]->cap_entries;
    const bool threaded = nq > kGroupInlineMaxQ;
    const size_t dbytes = (size_t)nq * k * sizeof(float), ibytes = (size_t)nq * k * sizeof(int64_t);
    cudaStream_t st[kExchMaxWorld];
    const float* qs[kExchMaxWorld];
    for (int s = 0; s < n; ++s) {
        wb_index* h = g->shards[s];
        st[s] = s ? h->stream : host ? h->stream : caller;
        TRY(set_dev(h));
        TRY(h->dbuf.ensure(dbytes));
        TRY(h->ibuf.ensure(ibytes));
        TRY(h->eD.ensure(dbytes));
        TRY(h->eI.ensure(ibytes));
    }
    TRY(set_dev(h0));
    if (!exch) {
        TRY(g->pD.ensure(n * dbytes));
        TRY(g->pI.ensure(n * ibytes));
    }
    if (!host) CK(cudaEventRecord(g->ev[0].get(), caller));
    for (int s = 0; s < n; ++s) {
        wb_index* h = g->shards[s];
        TRY(set_dev(h));
        if (host || s == 0) {
            TRY(stage_queries(h, nq, q, host, st[s], &qs[s]));
            continue;
        }
        // _dev: the copy waits for the caller's stream, and the caller's stream waits for the copy (so that a later
        // write of q_dev cannot race it)
        const size_t qbytes = (size_t)nq * h->d * sizeof(float);
        TRY(g->qpeer[s].ensure(qbytes));
        CK(cudaStreamWaitEvent(st[s], g->ev[0].get(), 0));
        CK(cudaMemcpyPeerAsync(g->qpeer[s].get(), h->device, q, h0->device, qbytes, st[s]));
        TRY(stage_queries(h, nq, g->qpeer[s].as<float>(), false, st[s], &qs[s]));
        CK(cudaEventRecord(g->ev[s].get(), st[s]));
    }
    if (!host) {
        TRY(set_dev(h0));
        for (int s = 1; s < n; ++s) CK(cudaStreamWaitEvent(caller, g->ev[s].get(), 0));
    }

    // Shard s's search.  Exchange: the global top-k lands in (D0, I0) on the root and in eD / eI elsewhere.  Fallback:
    // the local top-k lands in part s of (pD, pI) on the root.
    auto part = [&](int s, float* D0, int64_t* I0) -> int {
        wb_index* h = g->shards[s];
        if (exch)
            return group_exch_part(h, g->ex[s], filt(s), nq, qs[s], k, nprobe, s ? h->eD.as<float>() : D0,
                                   s ? h->eI.as<int64_t>() : I0, st[s]);
        TRY(set_dev(h));
        float* Dl = s ? h->eD.as<float>() : g->pD.as<float>();
        int64_t* Il = s ? h->eI.as<int64_t>() : g->pI.as<int64_t>();
        TRY(search_dev_impl(h, filt(s), nq, qs[s], k, nprobe, Dl, Il, st[s]));
        if (s == 0) return 0;
        CK(cudaMemcpyPeerAsync(g->pD.as<unsigned char>() + s * dbytes, h0->device, Dl, h->device, dbytes, st[s]));
        CK(cudaMemcpyPeerAsync(g->pI.as<unsigned char>() + s * ibytes, h0->device, Il, h->device, ibytes, st[s]));
        CK(cudaEventRecord(g->ev[s].get(), st[s]));
        return 0;
    };
    // Searches of 1-4 queries are enqueued on every GPU from this thread, root last (no thread hand-off on the latency
    // path); larger batches run each non-root shard on its own thread.  Every shard runs even when another one failed.
    auto run = [&](float* D0, int64_t* I0) -> int {
        int rc = 0;
        std::string err;
        auto keep = [&](int r) {
            if (r && !rc) {
                rc = r;
                err = g_err;
            }
        };
        if (threaded) {
            for (int s = 1; s < n; ++s) g->workers[s]->post([&part, s, D0, I0] { return part(s, D0, I0); });
            keep(part(0, D0, I0));
            for (int s = 1; s < n; ++s) keep(g->workers[s]->wait());
        } else {
            for (int s = n - 1; s >= 0; --s) keep(part(s, D0, I0));
        }
        if (rc) {
            g_err = err;
            return rc;
        }
        if (exch) return 0;
        TRY(set_dev(h0));
        for (int s = 1; s < n; ++s) CK(cudaStreamWaitEvent(st[0], g->ev[s].get(), 0));
        return wb_merge_topk_dev(h0->device, nq, k, n, g->pD.as<float>(), g->pI.as<int64_t>(), D0, I0, st[0]);
    };
    if (!host) {
        const int rc = run(D, I);
        if (set_dev(h0) != 0) return 1;
        return rc;
    }
    int rc = search_to_host(h0, nq, k, h0->eD, h0->eI, D, I, st[0], run);
    std::string err = g_err;
    for (int s = 1; s < n; ++s) {  // host calls return synchronised on every GPU
        const cudaError_t e = cudaStreamSynchronize(st[s]);
        if (e != cudaSuccess && !rc) {
            rc = fail("group search: shard %d: %s", s, cudaGetErrorString(e));
            err = g_err;
        }
    }
    if (!rc && exch)
        for (int s = 0; s < n; ++s)
            if (*reinterpret_cast<volatile int*>(g->ex[s]->status.get()))
                return fail("group search: GPU %d did not join the exchange within 20 s (results invalid)",
                            g->shards[s]->device);
    g_err = err;
    if (set_dev(h0) != 0) return 1;
    return rc;
}

extern "C" int wb_group_search(wb_group* g, wb_filter* const* filters, int64_t nq, const float* q_host, int64_t k,
                               int64_t nprobe, float* D_host, int64_t* I_host) {
    return group_search(g, filters, nq, q_host, true, k, nprobe, D_host, I_host, nullptr);
}
extern "C" int wb_group_search_dev(wb_group* g, wb_filter* const* filters, int64_t nq, const float* q_dev, int64_t k,
                                   int64_t nprobe, float* D_dev, int64_t* I_dev, void* stream) {
    return group_search(g, filters, nq, q_dev, false, k, nprobe, D_dev, I_dev, (cudaStream_t)stream);
}

// ---- range search (DESIGN.md "Range search") --------------------------------------------------------------------
// A result owns its (D, I): in host memory (wb_range_search) or, one part per query chunk with hits, in device memory of
// the index's GPU (wb_range_search_dev).  Either way it is independent of the index, its scratch and its lifetime.
struct wb_range_result {
    std::vector<float> D;
    std::vector<int64_t> I;
    int device = -1;  // >= 0: a device result on this GPU
    struct Part {
        DevPtr<float> D;
        DevPtr<int64_t> I;
        int64_t n = 0;
    };
    std::vector<Part> parts;
};

constexpr int64_t kRangeMaxQ = 32768;  // queries per chunk: one launch (grid.y) per scan

// K1 / K5 in range mode: `S` CTAs per query group, one launch per <= kMaxGridY groups.  Whole-row stages draw their
// row groups from the shared dispensers, which every launch leaves at zero as the fused tails do.
static int run_range_scan(wb_index* h, const ScanCfg& c, bool gather, ScanParams& p, int64_t S, int64_t nq,
                          const float* q_ld, const RangeOut& ro0, cudaStream_t st) {
    apply_scan_cfg(c, p);
    p.k = 0;
    p.nparts = (int)S;
    TRY(ensure_tail_counters(h, st));
    p.group_count = c.nchunks == 1 ? h->tailcnt.as<unsigned int>() + kMaxGridY : nullptr;
    const int64_t qgroups = (nq + c.NQ - 1) / c.NQ;
    TRY(timing_begin(h, h->timing, st));
    for (int64_t g0 = 0; g0 < qgroups; g0 += kMaxGridY) {
        const int64_t gy = std::min(kMaxGridY, qgroups - g0), qoff = g0 * c.NQ;
        p.queries = q_ld + (size_t)qoff * h->ld;
        p.nq = (int)std::min<int64_t>(nq - qoff, gy * c.NQ);
        if (gather) p.probes = h->pI.as<int64_t>() + (size_t)qoff * p.nprobe;
        RangeOut ro = ro0;
        ro.count += qoff;
        ro.qbase = (int)qoff;
        const dim3 grid((unsigned)S, (unsigned)gy);
        TRY(with_scan_instance(c.NQ, c.RW, gather, [&](auto NQ, auto RW, auto G) {
            return launch<scan_range_kernel<NQ, RW, G>>(grid, kScanThreads, c.smem, st, p, ro);
        }));
        h->launches++;
        if (p.group_count) CK(cudaMemsetAsync(p.group_count, 0, (size_t)gy * sizeof(unsigned int), st));
    }
    return timing_end(h, h->timing, st);
}

// Flat range hits of `nq` queries against `nrows` rows: K2 epochs when search would take K2 for this batch (the same
// cost model without its k terms), else K1.  A K2 batch whose candidate lists cannot be repaired goes to K1.
static int range_flat(wb_index* h, const float* rows, int64_t nrows, const float* q_ld, int64_t nq, const RowMask* mask,
                      const RangeOut& ro, cudaStream_t st) {
    int cap = 0;
    if (gemm_eligible(h, nrows, nq, 0, &cap)) {
        bool ovf = false;
        TRY(run_flat_gemm(h, rows, nrows, q_ld, nq, 0, cap, nullptr, nullptr, nullptr, st, true, &ovf, mask, &ro));
        if (!ovf) return 0;
        h->gemm_fallbacks++;
        CK(cudaMemsetAsync(ro.cursor, 0, (size_t)(1 + nq) * sizeof(unsigned long long), st));
    }
    ScanCfg c;
    TRY(plan_scan(h, nq, kRangeStage - kMinQueue, false, 0, &c));
    ScanParams p{};
    p.rows = rows;
    p.nrows = nrows;
    p.ld = h->ld;
    p.allow = mask ? mask->allow : nullptr;
    return run_range_scan(h, c, false, p, flat_ctas(h, c, nrows, nq), nq, q_ld, ro, st);
}

// IVF range hits: K4 picks the probes exactly as search does, then K5 scans them query-major in range mode.
static int range_ivf(wb_index* h, int64_t nq, const float* q_ld, int np, const uint32_t* allow, const RangeOut& ro,
                     cudaStream_t st) {
    TRY(ivf_probes(h, nq, q_ld, np, st));
    ScanCfg c;
    TRY(plan_scan(h, 1, kRangeStage - kMinQueue, true, np, &c));
    ScanParams p = ivf_scan_params(h, np, allow);
    return run_range_scan(h, c, true, p, ivf_ctas(h, nq), nq, q_ld, ro, st);
}

// Sort the `total` pooled hits of a chunk by query and key, emit them as (D, I) and append them to `res`: a host result
// gets them with one synchronisation, a device result gets a new part that the emit kernel writes on `st`.
// off[nq + 1]: exclusive prefix of the per-query counts.
static int range_assemble(wb_index* h, int64_t nq, const std::vector<int64_t>& off, const int64_t* ids,
                          wb_range_result* res, cudaStream_t st) {
    const int64_t total = off[nq];
    if (total == 0) return 0;
    uint64_t* pool = h->rpool.as<uint64_t>();
    TRY(h->rgrp.ensure((size_t)total * sizeof(uint64_t)));
    TRY(h->roff.ensure((size_t)(nq + 1) * sizeof(int64_t) + (size_t)nq * sizeof(unsigned int)));
    int64_t* off_dev = h->roff.as<int64_t>();
    unsigned int* fill = reinterpret_cast<unsigned int*>(off_dev + nq + 1);
    CK(cudaMemcpyAsync(off_dev, off.data(), (size_t)(nq + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
    CK(cudaMemsetAsync(fill, 0, (size_t)nq * sizeof(unsigned int), st));
    const unsigned blocks = (unsigned)((total + 255) / 256);
    uint64_t* cur = h->rgrp.as<uint64_t>();
    uint64_t* other = pool;
    range_scatter_kernel<<<blocks, 256, 0, st>>>(pool, h->rqid.as<uint32_t>(), total, off_dev, fill, cur);
    CK(cudaGetLastError());
    // runs of <= kRangeRun keys of one query, sorted in shared memory
    std::vector<int64_t> run_start;
    std::vector<int> run_len;
    int64_t longest = 0;
    for (int64_t q = 0; q < nq; ++q) {
        const int64_t n = off[q + 1] - off[q];
        longest = std::max(longest, n);
        for (int64_t s = 0; s < n; s += kRangeRun) {
            run_start.push_back(off[q] + s);
            run_len.push_back((int)std::min<int64_t>(kRangeRun, n - s));
        }
    }
    const size_t nruns = run_start.size();
    TRY(h->rrun.ensure(nruns * (sizeof(int64_t) + sizeof(int))));
    int64_t* rs_dev = h->rrun.as<int64_t>();
    int* rl_dev = reinterpret_cast<int*>(rs_dev + nruns);
    CK(cudaMemcpyAsync(rs_dev, run_start.data(), nruns * sizeof(int64_t), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(rl_dev, run_len.data(), nruns * sizeof(int), cudaMemcpyHostToDevice, st));
    CK(smem_optin<range_block_sort_kernel>(kRangeRun * 8));
    for (size_t r0 = 0; r0 < nruns; r0 += (size_t)1 << 30) {
        const size_t nr = std::min(nruns - r0, (size_t)1 << 30);
        range_block_sort_kernel<<<(unsigned)nr, kRangeThreads, (size_t)kRangeRun * 8, st>>>(cur, rs_dev + r0, rl_dev + r0);
        CK(cudaGetLastError());
    }
    h->launches += 2;
    for (int64_t w = kRangeRun; w < longest; w *= 2) {
        range_merge_kernel<<<blocks, 256, 0, st>>>(cur, other, off_dev, (int)nq, total, w);
        CK(cudaGetLastError());
        std::swap(cur, other);
        h->launches++;
    }
    // host result: (D, I) go to the two buffers the sorted keys no longer need, the query tags and the other key buffer
    float* D_dev = reinterpret_cast<float*>(h->rqid.get());
    int64_t* I_dev = reinterpret_cast<int64_t*>(other);
    if (res->device >= 0) {
        wb_range_result::Part part;
        CK(dev_alloc(&part.D, (size_t)total * sizeof(float)));
        CK(dev_alloc(&part.I, (size_t)total * sizeof(int64_t)));
        part.n = total;
        D_dev = part.D.get();
        I_dev = part.I.get();
        res->parts.push_back(std::move(part));
    }
    range_emit_kernel<<<blocks, 256, 0, st>>>(cur, total, ids, D_dev, I_dev);
    CK(cudaGetLastError());
    h->launches++;
    if (res->device >= 0) return 0;
    const size_t at = res->D.size();
    res->D.resize(at + (size_t)total);
    res->I.resize(at + (size_t)total);
    CK(cudaMemcpyAsync(res->D.data() + at, D_dev, (size_t)total * sizeof(float), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(res->I.data() + at, I_dev, (size_t)total * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return 0;
}

static int range_search_impl(wb_index* h, wb_filter* f, int64_t nq, const float* q, float thresh, int64_t nprobe,
                             int64_t* lims, wb_range_result* res, cudaStream_t st) {
    if (h->ivf && !h->trained) return fail("IndexIVFFlat is not trained");
    for (int64_t i = 0; i <= nq; ++i) lims[i] = 0;
    if (nq == 0 || h->n == 0) return 0;
    RowSel s;
    TRY(select_rows(h, f, st, &s));
    if (s.none) return 0;
    int np = 0;
    if (h->ivf) TRY(ivf_prepare(h, nprobe, st, &np));
    TRY(h->rstate.ensure((size_t)(1 + kRangeMaxQ) * sizeof(unsigned long long)));
    unsigned long long* cursor = h->rstate.as<unsigned long long>();
    std::vector<unsigned long long> cnt((size_t)(1 + kRangeMaxQ));
    for (int64_t q0 = 0; q0 < nq;) {
        int64_t nqc = std::min(kRangeMaxQ, nq - q0);
        const float* qc = q + (size_t)q0 * h->ld;
        // run the scan; if the hits exceed the pool, grow it to the exact count and run again
        for (int attempt = 0;; ++attempt) {
            TRY(h->rpool.ensure((size_t)std::min<int64_t>(kRangeBudgetHits, nqc * 64) * sizeof(uint64_t)));
            TRY(h->rqid.ensure(h->rpool.cap / 2));
            const RangeOut ro{thresh, cursor, cursor + 1, h->rpool.as<uint64_t>(), h->rqid.as<uint32_t>(),
                              (int64_t)(h->rpool.cap / sizeof(uint64_t)), 0};
            CK(cudaMemsetAsync(cursor, 0, (size_t)(1 + nqc) * sizeof(unsigned long long), st));
            if (h->ivf) TRY(range_ivf(h, nqc, qc, np, s.mask.allow, ro, st));
            else TRY(range_flat(h, s.rows, s.nrows, qc, nqc, s.masked(), ro, st));
            CK(cudaMemcpyAsync(cnt.data(), cursor, (size_t)(1 + nqc) * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            int64_t total = (int64_t)cnt[0];
            if (total <= ro.cap) break;
            if (attempt >= 3) return fail("range_search: the hit count of a chunk did not settle");
            if (total > kRangeBudgetHits) {  // fewer queries: the longest prefix whose hits fit the budget
                int64_t keep = 0, sum = 0;
                while (keep < nqc && sum + (int64_t)cnt[1 + keep] <= kRangeBudgetHits) sum += (int64_t)cnt[1 + keep++];
                if (keep == 0)
                    return fail("range_search: query %lld has %llu results, more than the %lld one call can hold",
                                (long long)q0, cnt[1], (long long)kRangeBudgetHits);
                nqc = keep;
                total = sum;
            }
            TRY(h->rpool.ensure((size_t)total * sizeof(uint64_t)));
            TRY(h->rqid.ensure((size_t)total * sizeof(uint32_t)));
        }
        std::vector<int64_t> off((size_t)nqc + 1, 0);
        for (int64_t i = 0; i < nqc; ++i) off[i + 1] = off[i] + (int64_t)cnt[1 + i];
        for (int64_t i = 1; i <= nqc; ++i) lims[q0 + i] = lims[q0] + off[i];
        TRY(range_assemble(h, nqc, off, s.ids, res, st));
        q0 += nqc;
    }
    return 0;
}

// `host`: q is host memory and the result a host result; else q is on the index's GPU and the result a device result.
static int range_search_entry(wb_index* h, wb_filter* f, int64_t nq, const float* q_in, bool host, float thresh,
                              int64_t nprobe, int64_t* lims_host, wb_range_result** out, cudaStream_t st) {
    if (!out) return fail("out is NULL");
    *out = nullptr;
    if (!h) return fail("NULL index");
    if (nq < 0) return fail("negative nq");
    if (!lims_host || (nq > 0 && !q_in)) return fail("NULL buffer");
    TRY(check_filter(h, f));
    TRY(set_dev(h));
    std::unique_ptr<wb_range_result> res(new wb_range_result());
    if (!host) res->device = h->device;
    const float* q = nullptr;
    if (nq > 0) TRY(stage_queries(h, nq, q_in, host, st, &q));
    TRY(range_search_impl(h, f, nq, q, thresh, nprobe, lims_host, res.get(), st));
    *out = res.release();
    return 0;
}

extern "C" int wb_range_search(wb_index* h, wb_filter* f, int64_t nq, const float* q_host, float thresh, int64_t nprobe,
                               int64_t* lims_host, wb_range_result** out) {
    return range_search_entry(h, f, nq, q_host, true, thresh, nprobe, lims_host, out, h ? h->stream : nullptr);
}

extern "C" int wb_range_search_dev(wb_index* h, wb_filter* f, int64_t nq, const float* q_dev, float thresh,
                                   int64_t nprobe, int64_t* lims_host, wb_range_result** out, void* stream) {
    return range_search_entry(h, f, nq, q_dev, false, thresh, nprobe, lims_host, out, (cudaStream_t)stream);
}

static int64_t range_result_size(const wb_range_result* r) {
    int64_t n = (int64_t)r->D.size();
    for (const auto& p : r->parts) n += p.n;
    return n;
}

extern "C" int wb_range_result_copy(const wb_range_result* r, float* D_host, int64_t* I_host) {
    if (!r) return fail("NULL range result");
    if (range_result_size(r) == 0) return 0;
    if (!D_host || !I_host) return fail("NULL buffer");
    if (r->device < 0) {
        memcpy(D_host, r->D.data(), r->D.size() * sizeof(float));
        memcpy(I_host, r->I.data(), r->I.size() * sizeof(int64_t));
        return 0;
    }
    CK(cudaSetDevice(r->device));
    CK(cudaDeviceSynchronize());  // the result was written on the caller's stream, which this call does not know
    for (const auto& p : r->parts) {
        CK(cudaMemcpy(D_host, p.D.get(), (size_t)p.n * sizeof(float), cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(I_host, p.I.get(), (size_t)p.n * sizeof(int64_t), cudaMemcpyDeviceToHost));
        D_host += p.n;
        I_host += p.n;
    }
    return 0;
}

extern "C" int wb_range_result_copy_dev(const wb_range_result* r, float* D_dev, int64_t* I_dev, void* stream) {
    if (!r) return fail("NULL range result");
    if (range_result_size(r) == 0) return 0;
    if (!D_dev || !I_dev) return fail("NULL buffer");
    cudaStream_t st = (cudaStream_t)stream;
    if (r->device < 0) {  // (pageable source: the call returns once the driver has staged it)
        CK(cudaMemcpyAsync(D_dev, r->D.data(), r->D.size() * sizeof(float), cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(I_dev, r->I.data(), r->I.size() * sizeof(int64_t), cudaMemcpyHostToDevice, st));
        return 0;
    }
    CK(cudaSetDevice(r->device));
    for (const auto& p : r->parts) {
        CK(cudaMemcpyAsync(D_dev, p.D.get(), (size_t)p.n * sizeof(float), cudaMemcpyDeviceToDevice, st));
        CK(cudaMemcpyAsync(I_dev, p.I.get(), (size_t)p.n * sizeof(int64_t), cudaMemcpyDeviceToDevice, st));
        D_dev += p.n;
        I_dev += p.n;
    }
    return 0;
}

extern "C" int wb_range_result_free(wb_range_result* r) {
    if (r && r->device >= 0) cudaSetDevice(r->device);  // the device memory is freed on its own GPU
    delete r;
    return 0;
}

// ---- filter objects --------------------------------------------------------------------------
static int filter_create(wb_index* h, std::unique_ptr<wb_filter> f, wb_filter** out) {
    TRY(set_dev(h));
    f->h = h;
    TRY(filter_eval(f.get()));
    *out = f.release();
    return 0;
}

extern "C" int wb_filter_create_ids(wb_index* h, int64_t n, const int64_t* ids_host, int invert, wb_filter** out) {
    if (!out) return fail("out is NULL");
    *out = nullptr;
    if (!h) return fail("NULL index");
    if (n < 0 || (n > 0 && !ids_host)) return fail("bad id set");
    std::vector<int64_t> s(ids_host, ids_host + n);
    if (!std::is_sorted(s.begin(), s.end())) std::sort(s.begin(), s.end());
    s.erase(std::unique(s.begin(), s.end()), s.end());
    TRY(set_dev(h));
    std::unique_ptr<wb_filter> f(new wb_filter());
    f->nset = (int64_t)s.size();
    f->invert = invert != 0;
    CK(dev_alloc(&f->set, std::max<size_t>(s.size(), 1) * 8));  // (an empty set still has a pointer: it is a set)
    if (!s.empty()) {
        CK(cudaMemcpyAsync(f->set.get(), s.data(), s.size() * 8, cudaMemcpyHostToDevice, h->stream));
        CK(cudaStreamSynchronize(h->stream));  // `s` is freed on return
    }
    return filter_create(h, std::move(f), out);
}

extern "C" int wb_filter_create_range(wb_index* h, int64_t imin, int64_t imax, int invert, wb_filter** out) {
    if (!out) return fail("out is NULL");
    *out = nullptr;
    if (!h) return fail("NULL index");
    std::unique_ptr<wb_filter> f(new wb_filter());
    f->imin = imin;
    f->imax = imax;  // imin >= imax: the empty set
    f->invert = invert != 0;
    return filter_create(h, std::move(f), out);
}

extern "C" int64_t wb_filter_count(const wb_filter* f) { return f ? f->count : -1; }

extern "C" int wb_filter_free(wb_filter* f) {
    if (!f) return 0;
    cudaSetDevice(f->h->device);
    delete f;
    return 0;
}

extern "C" int wb_merge_topk_dev(int device, int64_t nq, int64_t k, int64_t nparts, const float* D_parts_dev,
                                 const int64_t* I_parts_dev, float* D_dev, int64_t* I_dev, void* stream) {
    if (k < 1 || k > WB_MAX_K) return fail("k=%lld out of range [1, %d]", (long long)k, WB_MAX_K);
    if (nq <= 0 || nparts <= 0) return fail("empty merge");
    if (nparts * k >= (int64_t)0xFFFFFFFFll) return fail("too many candidates to merge");
    CK(cudaSetDevice(device));
    MergeParams m{};
    m.nq = nq;
    m.k = (int)k;
    m.nparts = nparts;
    m.S = merge_buffer_entries((int)k, nparts);
    m.Dp = D_parts_dev;
    m.Ip = I_parts_dev;
    m.D = D_dev;
    m.I = I_dev;
    CK(smem_optin<merge_topk_kernel<false>>(8192 * 8));
    merge_topk_kernel<false><<<(unsigned)nq, kMergeThreads, (size_t)m.S * 8, (cudaStream_t)stream>>>(m);
    CK(cudaGetLastError());
    return 0;
}

extern "C" int wb_range_merge_dev(int device, int64_t nq, int64_t nparts, const int64_t* lims_parts_dev,
                                  int64_t part_stride, const float* D_parts_dev, const int64_t* I_parts_dev,
                                  const int64_t* lims_dev, float* D_dev, int64_t* I_dev, void* stream) {
    if (nq < 0) return fail("negative nq");
    if (nparts < 1 || nparts > kMaxGridY) return fail("nparts=%lld out of range [1, %lld]", (long long)nparts,
                                                      (long long)kMaxGridY);
    if (part_stride < 0) return fail("negative part stride");
    if (nq == 0 || part_stride == 0) return 0;  // nothing to merge
    if (!lims_parts_dev || !D_parts_dev || !I_parts_dev || !lims_dev || !D_dev || !I_dev) return fail("NULL buffer");
    const int64_t bx = (part_stride + 255) / 256;
    if (bx > INT32_MAX) return fail("part stride %lld too large", (long long)part_stride);
    CK(cudaSetDevice(device));
    range_merge_parts_kernel<<<dim3((unsigned)bx, (unsigned)nparts), 256, 0, (cudaStream_t)stream>>>(
        lims_parts_dev, nq, part_stride, D_parts_dev, I_parts_dev, lims_dev, D_dev, I_dev);
    CK(cudaGetLastError());
    return 0;
}

// ---- IVF: make the inverted lists current (K8) and describe them ---------------------------------------------------
// faiss keeps its inverted lists current on every add; this backend groups the row store lazily, at the first search
// after an add.  write_index calls this first so that every list is one contiguous run of storage rows.
extern "C" int wb_ivf_finalize(wb_index* h) {
    if (!h || !h->ivf) return fail("not an IVF index");
    TRY(set_dev(h));
    return ensure_csr(h);
}
// list_off_host[nlist + 1]: list l holds the storage rows [list_off[l], list_off[l+1]) once wb_ivf_finalize has run
// and *grouped_out is 1 (0: the rows could not be regrouped for lack of memory; use wb_export_rows + assignments).
extern "C" int wb_ivf_list_offsets(wb_index* h, int64_t* list_off_host, int* grouped_out) {
    if (!h || !h->ivf) return fail("not an IVF index");
    if (!list_off_host) return fail("NULL buffer");
    TRY(set_dev(h));
    TRY(ensure_csr(h));
    CK(cudaMemcpyAsync(list_off_host, h->list_off.get(), (size_t)(h->nlist + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (grouped_out) *grouped_out = h->slot_row == nullptr;
    return 0;
}

// ---- row access ----------------------------------------------------------------------------
// pos[j] = the index of tgt[j] in keys[0, h->n), all ones when it is absent; `kernel` (find_ids_kernel<T>) takes 64
// targets per launch
template <class T>
static int find_positions(wb_index* h, void (*kernel)(const T*, int64_t, const int64_t*, int, unsigned long long*),
                          const T* keys, const int64_t* tgt, int64_t m, unsigned long long* pos, cudaStream_t st) {
    CK(cudaMemsetAsync(pos, 0xFF, (size_t)m * sizeof(int64_t), st));
    for (int64_t j0 = 0; j0 < m; j0 += 64) {
        const int mm = (int)std::min<int64_t>(64, m - j0);
        const unsigned grid = (unsigned)std::min<int64_t>(std::max<int64_t>((h->n + 255) / 256, 1), h->sm_count * 8);
        kernel<<<grid, 256, 0, st>>>(keys, h->n, tgt + j0, mm, pos + j0);
        CK(cudaGetLastError());
        h->launches++;
    }
    return 0;
}
// Insertion positions of ids_host[0, m) into hpos (-1: absent), and on the device into h->idbuf[m, 2m).
static int lookup_ids(wb_index* h, int64_t m, const int64_t* ids_host, int64_t* hpos) {
    TRY(set_dev(h));
    cudaStream_t st = h->stream;
    TRY(h->idbuf.ensure((size_t)m * 2 * sizeof(int64_t)));
    int64_t* tgt = h->idbuf.as<int64_t>();
    unsigned long long* pos = reinterpret_cast<unsigned long long*>(tgt + m);
    CK(cudaMemcpyAsync(tgt, ids_host, (size_t)m * sizeof(int64_t), cudaMemcpyHostToDevice, st));
    TRY(find_positions(h, find_ids_kernel<int64_t>, h->ids.get(), tgt, m, pos, st));
    CK(cudaMemcpyAsync(hpos, pos, (size_t)m * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return 0;
}

extern "C" int wb_lookup_ids(wb_index* h, int64_t m, const int64_t* ids_host, int64_t* pos_host) {
    if (!h) return fail("NULL index");
    if (m < 0) return fail("negative m");
    if (m == 0) return 0;
    if (!ids_host || !pos_host) return fail("NULL buffer");
    return lookup_ids(h, m, ids_host, pos_host);
}

extern "C" int wb_reconstruct_batch(wb_index* h, int64_t m, const int64_t* ids_host, float* out_host) {
    if (!h) return fail("NULL index");
    if (m < 0) return fail("negative m");
    if (m == 0) return 0;
    if (!ids_host || !out_host) return fail("NULL buffer");
    std::vector<int64_t> hpos((size_t)m);
    TRY(lookup_ids(h, m, ids_host, hpos.data()));
    cudaStream_t st = h->stream;
    TRY(h->xbuf.ensure((size_t)m * h->d * sizeof(float)));
    int64_t* tgt = h->idbuf.as<int64_t>();
    unsigned long long* pos = reinterpret_cast<unsigned long long*>(tgt + m);
    for (int64_t j = 0; j < m; ++j)
        if (hpos[j] < 0) return fail("reconstruct: id %lld not found in the index", (long long)ids_host[j]);
    if (h->row_pos) {  // grouped IVF store: insertion position -> storage row
        CK(cudaMemcpyAsync(tgt, pos, (size_t)m * sizeof(int64_t), cudaMemcpyDeviceToDevice, st));
        TRY(find_positions(h, find_ids_kernel<uint32_t>, h->row_pos.get(), tgt, m, pos, st));
    }
    const int64_t tot = m * h->d;
    gather_rows_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(h->rows.get(), h->ld, h->d, (const int64_t*)pos, m,
                                                                       h->xbuf.as<float>());
    CK(cudaGetLastError());
    h->launches++;
    CK(cudaMemcpyAsync(out_host, h->xbuf.get(), (size_t)tot * sizeof(float), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return 0;
}

extern "C" int wb_export_rows(wb_index* h, int64_t start, int64_t n, float* x_host, int64_t* ids_host,
                              int32_t* assign_host) {
    if (!h) return fail("NULL index");
    if (start < 0 || n < 0 || start + n > h->n) return fail("export range [%lld,%lld) outside [0,%lld)",
                                                            (long long)start, (long long)(start + n), (long long)h->n);
    if (n == 0) return 0;
    TRY(set_dev(h));
    cudaStream_t st = h->stream;
    if (x_host)
        CK(cudaMemcpy2DAsync(x_host, (size_t)h->d * 4, h->rows.get() + (size_t)start * h->ld, (size_t)h->ld * 4,
                             (size_t)h->d * 4, (size_t)n, cudaMemcpyDeviceToHost, st));
    if (ids_host) {
        if (h->row_pos) {  // grouped IVF store: the id of storage row r is ids[row_pos[r]]
            TRY(h->idbuf.ensure((size_t)n * 8));
            gather_ids_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(h->ids.get(), h->row_pos.get(), start, n, h->idbuf.as<int64_t>());
            CK(cudaGetLastError());
            h->launches++;
            CK(cudaMemcpyAsync(ids_host, h->idbuf.get(), (size_t)n * 8, cudaMemcpyDeviceToHost, st));
        } else {
            CK(cudaMemcpyAsync(ids_host, h->ids.get() + start, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
        }
    }
    if (assign_host) {
        if (!h->ivf) return fail("assignments exist only for IVF indices");
        CK(cudaMemcpyAsync(assign_host, h->assign.get() + start, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
    }
    CK(cudaStreamSynchronize(st));
    return 0;
}

// ---- IVF quantizer / k-means -----------------------------------------------------------------
extern "C" int wb_ivf_set_centroids(wb_index* h, const float* c) {
    if (!h || !h->ivf) return fail("not an IVF index");
    if (!c) return fail("NULL centroids");
    if (h->n > 0) return fail("cannot replace the centroids of a non-empty index");
    TRY(set_dev(h));
    CK(cudaMemsetAsync(h->centroids.get(), 0, (size_t)h->nlist * h->ld * 4, h->stream));
    CK(cudaMemcpy2DAsync(h->centroids.get(), (size_t)h->ld * 4, c, (size_t)h->d * 4, (size_t)h->d * 4, (size_t)h->nlist,
                         cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->trained = true;
    return 0;
}

// faiss ClusteringParameters::spherical.  Default 0: an IndexIVFFlat built with the plain constructor, as the
// reference does (feature_search_index.py:60), trains with spherical = false [faiss-upstream]; index_factory is what
// switches it on for inner-product indices.
extern "C" int wb_ivf_set_spherical(wb_index* h, int on) {
    if (!h || !h->ivf) return fail("not an IVF index");
    h->spherical = on != 0;
    return 0;
}

extern "C" int wb_ivf_mark_trained(wb_index* h) {
    if (!h || !h->ivf) return fail("not an IVF index");
    h->trained = true;
    return 0;
}

extern "C" int wb_ivf_get_centroids(const wb_index* h, float* c) {
    if (!h || !h->ivf) return fail("not an IVF index");
    if (!c) return fail("NULL centroids");
    TRY(set_dev(h));
    CK(cudaMemcpy2DAsync(c, (size_t)h->d * 4, h->centroids.get(), (size_t)h->ld * 4, (size_t)h->d * 4, (size_t)h->nlist,
                         cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

// x_dev has row stride d; kernels need stride ld and a 16-byte aligned base (see stage_queries)
static int stage_points(wb_index* h, int64_t n, const float* x_dev, cudaStream_t st, const float** out) {
    if (h->ld == h->d && aligned16(x_dev)) {
        *out = x_dev;
        return 0;
    }
    TRY(h->xbuf.ensure((size_t)n * h->ld * sizeof(float)));
    if (h->ld == h->d) {
        CK(cudaMemcpyAsync(h->xbuf.get(), x_dev, (size_t)n * h->d * sizeof(float), cudaMemcpyDeviceToDevice, st));
    } else {
        const int64_t tot = n * h->ld;
        pad_rows_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(x_dev, h->xbuf.as<float>(), n, h->d, h->ld);
        CK(cudaGetLastError());
        h->launches++;
    }
    *out = h->xbuf.as<float>();
    return 0;
}

static int kmeans_assign_impl(wb_index* h, int64_t n, const float* x_dev, int32_t* assign_dev, double* objective_host,
                              void* stream, bool tf32);
extern "C" int wb_kmeans_assign_dev(wb_index* h, int64_t n, const float* x_dev, int32_t* assign_dev,
                                    double* objective_host, void* stream) {
    return kmeans_assign_impl(h, n, x_dev, assign_dev, objective_host, stream, false);
}
// TRAINING-only variant: plain-TF32 scores (one tensor-core term instead of three), ~3x less tensor work.
extern "C" int wb_kmeans_assign_fast_dev(wb_index* h, int64_t n, const float* x_dev, int32_t* assign_dev,
                                         double* objective_host, void* stream) {
    return kmeans_assign_impl(h, n, x_dev, assign_dev, objective_host, stream, env_int("WB_KMEANS_EXACT", 0) == 0);
}
static int kmeans_assign_impl(wb_index* h, int64_t n, const float* x_dev, int32_t* assign_dev, double* objective_host,
                              void* stream, bool tf32) {
    if (!h || !h->ivf) return fail("not an IVF index");
    if (n <= 0 || !x_dev || !assign_dev) return fail("bad arguments");
    TRY(set_dev(h));
    cudaStream_t st = (cudaStream_t)stream;
    const float* x = nullptr;
    TRY(stage_points(h, n, x_dev, st, &x));
    TRY(h->dbuf.ensure((size_t)n * sizeof(float)));
    TRY(assign_rows(h, x, n, assign_dev, h->dbuf.as<float>(), st, tf32));
    if (objective_host) {
        TRY(h->misc.ensure(sizeof(double)));
        CK(cudaMemsetAsync(h->misc.get(), 0, sizeof(double), st));
        sum_f32_kernel<<<(unsigned)std::min<int64_t>((n + 255) / 256, 1024), 256, 0, st>>>(h->dbuf.as<float>(), n,
                                                                                          h->misc.as<double>());
        CK(cudaGetLastError());
        h->launches++;
        CK(cudaMemcpyAsync(objective_host, h->misc.get(), sizeof(double), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
    }
    return 0;
}

extern "C" int wb_kmeans_accumulate_dev(wb_index* h, int64_t n, const float* x_dev, const int32_t* assign_dev,
                                        float* sums_dev, int64_t* counts_dev, void* stream) {
    if (!h || !h->ivf) return fail("not an IVF index");
    if (n < 0 || !sums_dev || !counts_dev) return fail("bad arguments");
    TRY(set_dev(h));
    cudaStream_t st = (cudaStream_t)stream;
    TRY(h->kperm.ensure(std::max<size_t>((size_t)n * 4, 16)));
    TRY(h->koff.ensure((size_t)(h->nlist + 1) * 8));
    // group the points by their centroid on the device (stable: every list is summed in insertion order, so the
    // result does not depend on the schedule); no host copy, no synchronisation
    TRY(device_csr(h, assign_dev, n, nullptr, h->koff.as<int64_t>(), h->kperm.as<uint32_t>(), nullptr, st, false));
    segment_sum_kernel<<<(unsigned)h->nlist, 256, 0, st>>>(x_dev, h->d, h->d, h->kperm.as<uint32_t>(),
                                                          h->koff.as<int64_t>(), sums_dev, counts_dev);
    CK(cudaGetLastError());
    h->launches++;
    return 0;
}

extern "C" int wb_kmeans_update_dev(wb_index* h, const float* sums_dev, const int64_t* counts_dev, int64_t n_total,
                                    int64_t seed, int64_t* nsplit_host, void* stream) {
    if (!h || !h->ivf) return fail("not an IVF index");
    TRY(set_dev(h));
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t k = h->nlist;
    const int d = h->d, ld = h->ld;
    const int64_t tot = k * d;
    centroid_mean_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(sums_dev, counts_dev, h->centroids.get(), ld, d, k);
    CK(cudaGetLastError());
    h->launches++;
    // split_clusters [faiss-upstream]: an empty list takes a perturbed copy of a list picked with probability ~ its
    // size; eps = 1/1024.  The pick is a sequential draw over the list sizes (host, k counters); the copies are applied
    // on the device (split_apply_kernel) - the centroid table never leaves HBM.
    std::vector<int64_t> cnt((size_t)k);
    CK(cudaMemcpyAsync(cnt.data(), counts_dev, (size_t)k * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    int64_t nsplit = 0;
    bool any_empty = false;
    for (int64_t c = 0; c < k; ++c) any_empty |= cnt[c] == 0;
    if (any_empty && n_total > k) {
        std::mt19937 mt((uint32_t)seed);
        std::vector<double> hass(cnt.begin(), cnt.end());
        const double denom = (double)(n_total - k);
        std::vector<float> prob((size_t)k);  // acceptance probability of every list, kept current
        for (int64_t c = 0; c < k; ++c) prob[c] = (float)((hass[c] - 1.0) / denom);
        std::vector<int32_t> pairs;
        for (int64_t ci = 0; ci < k; ++ci) {
            if (hass[ci] != 0) continue;
            int64_t cj = 0;
            for (int64_t guard = 0;; cj = (cj + 1 == k ? 0 : cj + 1)) {
                // (float)mt() / (float)mt.max(): the divisor is 2^32 as a float, so the product below is the same bits
                const float r = (float)mt() * 2.3283064365386963e-10f;
                if (r < prob[cj]) break;
                if (++guard > k * 1000) return fail("split_clusters did not converge");
            }
            pairs.push_back((int32_t)ci);
            pairs.push_back((int32_t)cj);
            hass[ci] = (double)((int64_t)hass[cj] / 2);
            hass[cj] -= hass[ci];
            prob[ci] = (float)((hass[ci] - 1.0) / denom);
            prob[cj] = (float)((hass[cj] - 1.0) / denom);
            nsplit++;
        }
        TRY(h->misc.ensure(pairs.size() * sizeof(int32_t) + 16));
        CK(cudaMemcpyAsync(h->misc.get(), pairs.data(), pairs.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        split_apply_kernel<<<(unsigned)((d + 255) / 256), 256, 0, st>>>(h->centroids.get(), ld, d, h->misc.as<int32_t>(), (int)nsplit);
        CK(cudaGetLastError());
        h->launches++;
        CK(cudaStreamSynchronize(st));  // `pairs` (host) is read by the copy above
    }
    if (h->spherical) {
        renorm_rows_kernel<<<(unsigned)k, 256, 0, st>>>(h->centroids.get(), ld, d);
        CK(cudaGetLastError());
        h->launches++;
    }
    if (nsplit_host) *nsplit_host = nsplit;
    return 0;
}

// The k-means iterations of wb_ivf_train, on device buffers that the caller owns: x [n, d], assign [n],
// sums [nlist, d], counts [nlist] and the non-finite flag.
static int kmeans_train(wb_index* h, int64_t n, const float* x_host, int niter, int64_t seed, float* x, int32_t* assign,
                        float* sums, int64_t* counts, int* nonfinite) {
    cudaStream_t st = h->stream;
    const int64_t k = h->nlist;
    const int d = h->d;
    CK(cudaMemcpyAsync(x, x_host, (size_t)n * d * 4, cudaMemcpyHostToDevice, st));
    // faiss Clustering::train: "input contains NaN's or Inf's" - checked on the device, read at the first sync
    CK(cudaMemsetAsync(nonfinite, 0, sizeof(int), st));
    nonfinite_flag_kernel<<<(unsigned)(h->sm_count * 8), 256, 0, st>>>(x, n * (int64_t)d, nonfinite);
    CK(cudaGetLastError());
    // initial centroids: first k rows of the faiss-style random permutation, seed + 1
    std::mt19937 mt((uint32_t)(seed + 1));
    std::vector<int64_t> perm((size_t)n);
    for (int64_t i = 0; i < n; ++i) perm[i] = i;
    for (int64_t i = 0; i + 1 < n; ++i) {
        const int64_t i2 = i + (int64_t)(mt() % (uint64_t)(n - i));
        std::swap(perm[i], perm[i2]);
    }
    CK(cudaMemsetAsync(h->centroids.get(), 0, (size_t)k * h->ld * 4, st));
    {   // the k picked rows, gathered by one kernel
        TRY(h->idbuf.ensure((size_t)k * 8));
        CK(cudaMemcpyAsync(h->idbuf.get(), perm.data(), (size_t)k * 8, cudaMemcpyHostToDevice, st));
        if (h->ld == d) {
            gather_rows_kernel<<<(unsigned)((k * d + 255) / 256), 256, 0, st>>>(x, d, d, h->idbuf.as<int64_t>(), k, h->centroids.get());
            CK(cudaGetLastError());
        } else {
            TRY(h->xbuf.ensure((size_t)k * d * 4));
            gather_rows_kernel<<<(unsigned)((k * d + 255) / 256), 256, 0, st>>>(x, d, d, h->idbuf.as<int64_t>(), k, h->xbuf.as<float>());
            CK(cudaGetLastError());
            pad_rows_kernel<<<(unsigned)((k * h->ld + 255) / 256), 256, 0, st>>>(h->xbuf.as<float>(), h->centroids.get(), k, d, h->ld);
            CK(cudaGetLastError());
        }
        h->launches++;
        CK(cudaStreamSynchronize(st));  // perm (host) is read by the copy above
        int bad = 0;
        CK(cudaMemcpy(&bad, nonfinite, sizeof(int), cudaMemcpyDeviceToHost));
        if (bad) return fail("input contains NaN's or Inf's");
    }
    if (h->spherical) {
        renorm_rows_kernel<<<(unsigned)k, 256, 0, st>>>(h->centroids.get(), h->ld, d);
        CK(cudaGetLastError());
        h->launches++;
    }
    for (int it = 0; it < niter; ++it) {
        double obj = 0;
        TRY(wb_kmeans_assign_fast_dev(h, n, x, assign, &obj, st));
        TRY(wb_kmeans_accumulate_dev(h, n, x, assign, sums, counts, st));
        int64_t nsplit = 0;
        TRY(wb_kmeans_update_dev(h, sums, counts, n, 1234, &nsplit, st));
    }
    return 0;
}

extern "C" int wb_ivf_train(wb_index* h, int64_t n, const float* x_host, int niter, int64_t seed) {
    if (!h || !h->ivf) return fail("not an IVF index");
    if (h->n > 0) return fail("cannot train a non-empty index");
    if (n < h->nlist) return fail("Number of training points (%lld) should be at least as large as number of clusters (%lld)",
                                   (long long)n, (long long)h->nlist);
    if (!x_host) return fail("NULL training set");
    TRY(set_dev(h));
    const int64_t k = h->nlist;
    const int d = h->d;
    DevPtr<float> x, sums;
    DevPtr<int32_t> assign;
    DevPtr<int64_t> counts;
    DevPtr<int> nonfinite;
    CK(dev_alloc(&x, (size_t)n * d * 4));
    CK(dev_alloc(&assign, (size_t)n * 4));
    CK(dev_alloc(&sums, (size_t)k * d * 4));
    CK(dev_alloc(&counts, (size_t)k * 8));
    CK(dev_alloc(&nonfinite, sizeof(int)));
    const int rc = kmeans_train(h, n, x_host, niter, seed, x.get(), assign.get(), sums.get(), counts.get(), nonfinite.get());
    const cudaError_t e = cudaStreamSynchronize(h->stream);  // the buffers are freed on return
    if (rc) return rc;
    if (e != cudaSuccess) return fail("k-means training failed: %s", cudaGetErrorString(e));
    h->trained = true;
    return 0;
}

// ---- TF32 tensor-pipe peak of this GPU, measured with the library's own MMA shape (gemm_ss.cuh) -----------------
// Denominator for the batched-search roofline in bench.py: `iters` x 4 back-to-back
// tcgen05.mma.cta_group::2.kind::tf32 (M = 256, N = 256, K = 8) per CTA pair, no loads, best of `reps` launches.
extern "C" int wb_tf32_peak(int device, int iters, int reps, double* tflops_burst_out, double* tflops_sustained_out) {
    if (iters < 1 || reps < 1 || !tflops_burst_out) return fail("bad arguments");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) return fail("no CUDA device available (%s)", cudaGetErrorString(e));
    if (device < 0 || device >= ndev) return fail("device %d out of range", device);
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return fail("device %d is not sm_100", device);
    const int npairs = prop.multiProcessorCount / 2;
    const int constant_ops = env_int("WB_PEAK_CONSTANT", 0);  // 1: all-ones operands (no bit toggling: less power, higher clock)
    const size_t smem = (size_t)kF2StageBytes + 1024;
    CK(cudaFuncSetAttribute(tf32_peak_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    CK(cudaEventCreate(&e0));
    const EventPtr own_e0(e0);
    CK(cudaEventCreate(&e1));
    const EventPtr own_e1(e1);
    const double flop = (double)npairs * iters * 4.0 * 2.0 * 256.0 * 256.0 * 8.0;
    float best = 1e30f;
    for (int r = 0; r < 4; ++r) {  // burst: best single launch (the first one is the warm-up)
        CK(cudaEventRecord(e0, 0));
        tf32_peak_kernel<<<2 * npairs, 128, smem, 0>>>(iters, constant_ops);
        CK(cudaGetLastError());
        CK(cudaEventRecord(e1, 0));
        CK(cudaEventSynchronize(e1));
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, e0, e1));
        if (r > 0) best = std::min(best, ms);
    }
    *tflops_burst_out = flop / (best * 1e-3) / 1e12;
    if (tflops_sustained_out) {  // sustained: `reps` launches back to back, the second half timed (power cap settled)
        const int half = std::max(1, reps / 2);
        for (int r = 0; r < reps - half; ++r) tf32_peak_kernel<<<2 * npairs, 128, smem, 0>>>(iters, constant_ops);
        CK(cudaEventRecord(e0, 0));
        for (int r = 0; r < half; ++r) tf32_peak_kernel<<<2 * npairs, 128, smem, 0>>>(iters, constant_ops);
        CK(cudaGetLastError());
        CK(cudaEventRecord(e1, 0));
        CK(cudaEventSynchronize(e1));
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, e0, e1));
        *tflops_sustained_out = flop * half / (ms * 1e-3) / 1e12;
    }
    return 0;
}

// ---- FeatureStore fast ingest (host only) ------------------------------------------------------------
// Count the feature rows of one WebdatasetStore shard and report their dimension.
extern "C" int wb_tar_scan(const char* path, int64_t* rows_out, int64_t* members_out, int64_t* d_out) {
    if (!path) return fail("NULL path");
    int64_t rows = 0, members = 0, d = -1;
    std::string why;
    {   // fixed-stride shards (what WebdatasetStore writes): the layout is derived from the first member and checked
        // on up to 64 evenly spaced members - a handful of pages per shard, like the reference, which counts members
        // without reading payloads (webdataset_store.py:83-91; its count is an estimate too).  wb_tar_read verifies
        // EVERY member when it decodes and reports the exact number of rows.
        wbtar::Mapped mp;
        wbtar::Plan pl;
        bool ok = mp.open(path, false) && wbtar::make_plan(mp, &pl);
        if (ok) {  // up to 64 evenly spaced members (all of them in a small shard)
            const int64_t S = std::min<int64_t>(pl.count, 64);
            for (int64_t i = 0; i < S && ok; ++i) {
                int64_t id = 0;
                ok = wbtar::check_member(mp, pl, S > 1 ? i * (pl.count - 1) / (S - 1) : 0, &id);
            }
        }
        if (ok) {
            if (rows_out) *rows_out = pl.count * pl.m;
            if (members_out) *members_out = pl.count;
            if (d_out) *d_out = pl.d;
            return 0;
        }
    }
    const int rc = wbtar::walk(path, [&](const wbtar::Sample& s) {
        if (d < 0) d = s.d;
        if (s.d != d) return 2;
        rows += s.m;
        members++;
        return 0;
    }, &why);
    if (rc) return fail("wb_tar_scan(%s): %s (code %d)", path, why.empty() ? "mixed dimensions" : why.c_str(), rc), rc + 1;
    if (rows_out) *rows_out = rows;
    if (members_out) *members_out = members;
    if (d_out) *d_out = d;
    return 0;
}

// Decode one shard into caller-owned host buffers: ids[cap] (the sample key, repeated for multi-row samples),
// x[cap*d] float32.  *rows_out = rows written.  Fails (non-zero) if the shard needs the python reader.
extern "C" int wb_tar_read(const char* path, int64_t d, int64_t cap, int64_t* ids, float* x, int64_t* rows_out) {
    if (!path || !ids || !x || !rows_out) return fail("NULL argument");
    int64_t n = 0;
    std::string why;
    {
        wbtar::Mapped mp;
        wbtar::Plan pl;
        if (mp.open(path) && wbtar::make_plan(mp, &pl) && pl.d == d && pl.count * pl.m <= cap) {
            const size_t row_bytes = (size_t)pl.m * (size_t)d * 4;
            const bool ok = wbtar::for_each_member(mp, pl, [&](int64_t j, int64_t id) {
                memcpy(reinterpret_cast<unsigned char*>(x) + (size_t)j * row_bytes,
                       mp.p + (size_t)j * pl.stride + pl.pre + 512 + pl.data_off, row_bytes);
                for (int64_t r = 0; r < pl.m; ++r) ids[j * pl.m + r] = id;
            });
            if (ok) {
                *rows_out = pl.count * pl.m;
                return 0;
            }
        }
    }
    const int rc = wbtar::walk(path, [&](const wbtar::Sample& s) {
        if (s.d != d) { why = "dimension changes inside the shard"; return 2; }
        if (n + s.m > cap) { why = "buffer too small"; return 1; }
        memcpy(x + (size_t)n * d, s.data, (size_t)s.m * d * 4);
        for (int64_t r = 0; r < s.m; ++r) ids[n + r] = s.id;
        n += s.m;
        return 0;
    }, &why);
    if (rc) return fail("wb_tar_read(%s): %s (code %d)", path, why.c_str(), rc), rc + 1;
    *rows_out = n;
    return 0;
}
