// scan.cuh - K1 flat_scan_topk and K5 ivf_list_scan_topk (one kernel, two row sources).
//
// Replaces faiss knn_inner_product/exhaustive_inner_product_seq + heap (IndexFlat::search) and
// IndexIVF::search_preassigned + IVFFlatScanner::scan_codes [faiss-upstream], reached from
// /root/reference/src/index/feature_search_index.py:113 and /root/reference/api/routes.py:1407.
//
// HBM-bound streaming kernel (DESIGN.md "K1"):
//   * one persistent CTA per SM: warp 0 is the producer, warps 1..8 are consumers;
//   * the producer streams "row groups" of 32 rows through a ring of shared-memory stages with
//     1-D bulk async copies (cp.async.bulk -> UBLKCP, the TMA engine), one copy per row chunk,
//     completion on an mbarrier (full[]); consumers hand stages back through empty[];
//   * each consumer warp owns 4 rows of the group and NQ (1/2/4/8) queries: 128-bit LDS of the
//     row chunk and of the query chunk (queries are resident in shared memory), FMA into 4*NQ
//     register accumulators, then a transposing warp-shuffle reduction that leaves each
//     (row, query) score in one lane;
//   * fused top-k: a score survives only if it beats the CTA's current k-th best for that query
//     (register compare against a shared threshold); survivors go to a small shared-memory
//     queue; when a queue fills, the consumers bitonic-sort [top-k list | queue] in shared
//     memory and tighten the threshold.  Scores never go to HBM; each CTA writes k keys per
//     query at the end, merged by merge_topk_kernel (merge.cuh).
//   * range mode (scan_range_kernel, range search): the same scan with a fixed threshold; every hit is staged in the
//     shared lists and flushed to a global pool (RangeOut) instead of the fused top-k (DESIGN.md "Range search").
//   * int8 filter (flat top-k of 1-2 queries, DESIGN.md "K1"): the ring streams the int8 image of the rows instead,
//     the consumers score it approximately, and only the (row, query) pairs whose approximation can reach the
//     threshold are queued and re-scored from the fp32 rows with the arithmetic of the fp32 scan; every CTA's list is
//     therefore the top-k of the exact keys of its rows, as without the filter.
// Algorithmic bytes per launch: nrows * ld * 4 (the row store is read exactly once per pass); with the int8 filter
// nrows * img_row_bytes(ld) plus the re-scored rows.
#pragma once
#include <cuda_fp16.h>
#include "coarse.cuh"
#include "exchange.cuh"
#include "filter.cuh"

namespace wb {

constexpr int kConsumerWarps = 8;
constexpr int kMaxRowsPerWarp = 4;
constexpr int kMaxGroupRows = kConsumerWarps * kMaxRowsPerWarp;  // 32
constexpr int kConsumerThreads = kConsumerWarps * kWarp;   // 256
constexpr int kScanThreads = kConsumerThreads + kWarp;     // 288
constexpr int kBarConsumers = 1;
constexpr int kMinQueue = 64;  // queue capacity >= 2 * kMaxGroupRows

struct ScanParams {
    const float* rows;      // row store [*, ld]
    int64_t nrows;          // flat: rows to scan; gather: unused
    int ld;                 // row stride in floats (multiple of 4)
    const float* queries;   // [nq, ld]
    int nq;
    int k;
    int P;                  // per-query list size (power of two >= k + kMinQueue)
    int ck;                 // chunk width in floats (multiple of 4)
    int nchunks;            // ceil(ld / ck)
    int stages;
    int single_copy;        // flat && nchunks == 1: one bulk copy per group
    int rw;                 // rows per consumer warp (4, 2 or 1); a row group is 8 * rw rows
    uint64_t* parts;        // [nq][nparts][k] keys
    int nparts;             // == gridDim.x
    // gather mode (IVF): candidates = concatenation of the probed lists of query blockIdx.y
    const uint32_t* perm;     // CSR: row index per slot; null when the rows are physically grouped by list
    const uint32_t* row_pos;  // storage row -> insertion position (the tie rule and the id lookup); null: identity
    const int64_t* list_off;  // CSR: [nlist + 1]
    const int64_t* probes;    // [nq][nprobe] list ids (-1 = none); unused when the coarse quantizer is fused
    int nprobe;
    // fused coarse quantizer (coarse.cuh; gather mode, cooperative launch, fuse_tail set): the CTAs of a query group
    // score the centroid table, meet at coarse_count[blockIdx.y] and each select the top-nprobe lists themselves.
    const float* centroids;      // [nlist][ld]; null: the probes come from `probes`
    int64_t nlist;
    uint32_t* coarse_keys;       // [gridDim.y][nlist] scratch: ordered scores
    unsigned int* coarse_count;  // [gridDim.y] arrival counters, zero between launches (reset with tail_count)
    // fused tail (K3 inside K1/K5): the LAST CTA of a query group to finish merges the group's nparts lists and
    // emits (D, I) itself - a search is one launch instead of scan + merge.  With `exchange` set it also pushes the
    // merged rows to the peer GPUs' mailboxes, waits for theirs and emits the GLOBAL top-k (exchange.cuh).
    int fuse_tail;
    int S_merge;              // sort-buffer entries of the fused merge (the idle ring holds them)
    int heads_bytes;          // > 0: the fused merge tries block_merge_heads (merge.cuh) in this many bytes of the ring
    int rank_sort;            // 1: [list | queue] of one query is sorted by rank counting (P <= 512), not bitonic
    unsigned int* tail_count; // [gridDim.y] arrival counters, zero between launches (the last CTA resets its own)
    // dynamic row-group scheduling (fused-tail launches with whole-row stages): CTAs draw the next row group from
    // group_count[blockIdx.y] instead of striding by gridDim.x.  SMs stream at slightly different rates (ncu: the
    // fastest SM of a statically partitioned scan idles for 6-10 % of the kernel); with a shared dispenser every SM
    // works until the rows run out.  The result does not depend on who scans what: keys carry positions.
    unsigned int* group_count; // [gridDim.y], zero between launches (reset with tail_count); null: static partition
    const int64_t* ids;       // position -> external id (null: id = position)
    const uint32_t* allow;    // filtered search: bitmap over insertion positions (filter.cuh); null: every row
    float* D;                 // [nq][k]
    int64_t* I;
    int exchange;             // 0: emit local results; 1: exch holds the peer mailboxes
    // diagnostics (WB_PHASE_TS=1, scripts/phase_times.py): globaltimer stamps of the first consumer thread of every CTA
    // of query group 0 - [blockIdx.x][16]: 0 start, 1 centroids scored, 2 coarse barrier passed, 3 probes selected,
    // 4 prologue done, 5 rows done, 6 final sort done, 7 arrived, 8 merge selected (last CTA), 9 results written,
    // 10-13 inside block_merge_heads: staged, T0 found, candidates compacted, ranked
    unsigned long long* phase_ts;
    ExchParams exch;
    // int8 filter (scan_topk_kernel<..., IMG = true>): `img` is the int8 image of `rows` (int8_image_kernel), row
    // stride img_row_bytes(ld) = 4 * ck; `rows` is read only to re-score the queued candidates
    const uint8_t* img;
    unsigned long long* rescored;    // += (row, query) pairs re-scored by this launch
};

constexpr int kRescoreCap = 256;    // queued (row, query) pairs of the int8 filter per CTA
constexpr int kRescoreChunk = 32;   // pairs re-scored per insertion round: 4 rows in flight per consumer warp

// A row of the int8 image: a 16-byte header {s, resid, xhat, 0} (fp32) and the codes u_i = n_i + 128 (n_i in
// [-127, 127], offset binary), zero codes (128) up to a multiple of 16 bytes.  The row's approximation is s * n;
// resid >= |x - s n| and xhat >= |s n| (both rounded up); s is NaN for a row with a NaN or Inf element.
constexpr int kImgHeader = 16;
__host__ __device__ inline int img_row_bytes(int ld) { return kImgHeader + ((ld + 15) & ~15); }

struct ScanSmem {
    size_t ring, queries, lists, bars, misc, prefix, rescore, total;
};

// `ld`: stride of the queries in shared memory (floats).  `rescore`: the int8 filter's queue, per-query margin terms
// (8 floats) and fp16 queries (img_row_bytes(ld) - kImgHeader halves each).
__host__ __device__ inline ScanSmem scan_smem_layout(int NQ, int ld, int P, int ck, int stages, int nprobe,
                                                     int group_rows, bool rescore = false) {
    ScanSmem L;
    size_t o = 0;
    L.ring = o;    o += (size_t)stages * group_rows * ck * 4;
    L.queries = o; o += (size_t)NQ * ld * 4;
    o = (o + 15) & ~(size_t)15;
    L.lists = o;   o += (size_t)NQ * P * 8;
    L.bars = o;    o += (size_t)stages * 2 * 8 + (size_t)stages * 8;  // full[], empty[], group id of each stage
    L.misc = o;    o += (size_t)NQ * 12 + 16;  // qcnt[NQ] (int) + thr_s[NQ] (float) + 4 ints (fused tail / work item) + pair[NQ] (list-major)
    o = (o + 7) & ~(size_t)7;
    L.prefix = o;  o += nprobe > 0 ? (size_t)nprobe * 8 + (size_t)(nprobe + 1) * 4 : 0;  // pbase[np] i64 + prefix[np+1] u32
    o = (o + 15) & ~(size_t)15;
    L.rescore = o; o += rescore ? (size_t)kRescoreCap * 8 + (size_t)NQ * (32 + 2 * (img_row_bytes(ld) - kImgHeader)) + 16 : 0;
    L.total = (o + 15) & ~(size_t)15;
    return L;
}

// Sum V per-lane partials across the warp, V in {4,8,16,32}.  Returns the total of value
// index (lane >> (5 - log2 V)) - every lane of that index group holds the same sum.
template <int N, int OFF>
__device__ __forceinline__ void multi_reduce_step(float* v, int lane) {
    if constexpr (OFF >= 1) {
        if constexpr (N > 1) {
            constexpr int H = N / 2;
            const bool up = (lane & OFF) != 0;
#pragma unroll
            for (int i = 0; i < H; ++i) {
                const float keep = up ? v[i + H] : v[i];
                const float send = up ? v[i] : v[i + H];
                v[i] = keep + __shfl_xor_sync(0xffffffffu, send, OFF);
            }
            multi_reduce_step<H, OFF / 2>(v, lane);
        } else {
            v[0] += __shfl_xor_sync(0xffffffffu, v[0], OFF);
            multi_reduce_step<1, OFF / 2>(v, lane);
        }
    }
}

template <int V>
struct Log2 { static constexpr int value = 1 + Log2<V / 2>::value; };
template <>
struct Log2<1> { static constexpr int value = 0; };

struct GatherCtx {
    const uint32_t* prefix;  // smem [nprobe + 1] exclusive prefix of probed list sizes
    const int64_t* pbase;    // smem [nprobe] CSR offset of each probed list
    const uint32_t* perm;
    int nprobe;
};

__device__ __forceinline__ uint32_t gather_row(const GatherCtx& G, uint32_t cpos) {
    int lo = 0, hi = G.nprobe - 1;  // largest j with prefix[j] <= cpos
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (G.prefix[mid] <= cpos) lo = mid;
        else hi = mid - 1;
    }
    const int64_t slot = G.pbase[lo] + (int64_t)(cpos - G.prefix[lo]);
    return G.perm ? G.perm[slot] : (uint32_t)slot;  // perm == null: rows are physically grouped by list
}

// Range search (DESIGN.md "Range search"): where the result goes.  Every row with score > thresh (and allowed by the
// filter) is appended to `keys` / `qid` at a slot drawn from `cursor`; `count[q]` counts the hits of query q.  Both
// counters keep counting once `cap` slots are used, so the host learns the exact sizes from one read.
struct RangeOut {
    float thresh;
    unsigned long long* cursor;  // pool slots drawn so far
    unsigned long long* count;   // [nq of this launch] hits per query
    uint64_t* keys;              // [cap] pool: make_key(score, insertion position)
    uint32_t* qid;               // [cap] query of each pool entry (chunk-relative)
    int64_t cap;
    int qbase;                   // chunk-relative index of this launch's first query
};

// The scan (K1 flat, K5 gather) with its result stage as a compile-time mode: RANGE = false keeps the fused top-k,
// RANGE = true stages every hit in the per-query shared lists and flushes them to the range pool (RangeOut).
// Range mode: move the staged hits of every query of this CTA to the pool - one slot reservation and one count per
// query and flush - and empty the stages.  Called by all consumer threads at a consumer barrier.  The pool slot bases
// live in the misc region behind qcnt[] (the range kernel has no thresholds there): round8(4 NQ) + 8 NQ <= 12 NQ + 16.
template <int NQ>
__device__ __forceinline__ void range_flush(const ScanSmem& L, unsigned char* smem, const uint64_t* lists, int* qcnt,
                                            int P, int q0, int nqv, int ctid, const RangeOut& ro) {
    unsigned long long* base = reinterpret_cast<unsigned long long*>(smem + L.misc + ((NQ * 4 + 7) & ~7));
    if (ctid < nqv) {
        const int c = qcnt[ctid];
        if (c) {
            base[ctid] = atomicAdd(ro.cursor, (unsigned long long)c);
            atomicAdd(&ro.count[q0 + ctid], (unsigned long long)c);
        }
    }
    named_bar_sync(kBarConsumers, kConsumerThreads);
    for (int i = ctid; i < nqv * P; i += kConsumerThreads) {
        const int l = i / P, j = i - l * P;
        if (j < qcnt[l]) {
            const unsigned long long slot = base[l] + (unsigned long long)j;
            if (slot < (unsigned long long)ro.cap) {
                ro.keys[slot] = lists[i];
                ro.qid[slot] = (uint32_t)(ro.qbase + q0 + l);
            }
        }
    }
    named_bar_sync(kBarConsumers, kConsumerThreads);
    if (ctid < nqv) qcnt[ctid] = 0;
    named_bar_sync(kBarConsumers, kConsumerThreads);
}

// The exact fp32 score of J rows, each against its own query (queries in shared memory, stride dq4 float4), with the
// arithmetic of the fp32 scan's whole-row stages: lane l accumulates float4 l, l + 32, ... in order with fmaf in x, y,
// z, w order, then the xor butterfly 16, 8, 4, 2, 1 (the sums multi_reduce_step forms, so the same bits).  Every lane
// gets every score.  The loads of all J rows are in flight together.
template <int J>
__device__ __forceinline__ void exact_scores(const float* rows, int ld, const float4* q4, int dq4, const uint64_t* ent,
                                             const bool* valid, int lane, float* a) {
    const float4* xr[J];
    const float4* qr[J];
#pragma unroll
    for (int j = 0; j < J; ++j) {
        xr[j] = reinterpret_cast<const float4*>(rows + (size_t)(ent[j] >> 8) * ld);
        qr[j] = q4 + (size_t)(ent[j] & 0xff) * dq4;
        a[j] = 0.f;
    }
    const int d4 = ld >> 2;
#pragma unroll 2
    for (int i = lane; i < d4; i += 32) {
        float4 x[J];
#pragma unroll
        for (int j = 0; j < J; ++j) x[j] = valid[j] ? __ldg(xr[j] + i) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int j = 0; j < J; ++j) {
            const float4 q = qr[j][i];
            a[j] = fmaf(x[j].x, q.x, a[j]);
            a[j] = fmaf(x[j].y, q.y, a[j]);
            a[j] = fmaf(x[j].z, q.z, a[j]);
            a[j] = fmaf(x[j].w, q.w, a[j]);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
#pragma unroll
        for (int j = 0; j < J; ++j) a[j] += __shfl_xor_sync(0xffffffffu, a[j], o);
}

// a + the dot product of 8 image codes (offset binary, element 8i + j in byte j) with 8 fp16 query elements, in fp32.
// PRMT puts two codes u under the exponent byte of fp16 1024 (0x64: 1024 + u exactly), HADD2 subtracts 1152 (exact
// fp16 n = u - 128), and fma.rn.f32.f16 (FHFMA) adds the exact product n q to the fp32 sum with one rounding: 2
// instructions per element at one query, 3 at two (the unpack is shared).
__device__ __forceinline__ float fma_f32_f16(uint32_t a, uint32_t b, bool hi, float c) {
    const uint16_t x = (uint16_t)(hi ? a >> 16 : a), y = (uint16_t)(hi ? b >> 16 : b);
    float d;
    asm("fma.rn.f32.f16 %0, %1, %2, %3;" : "=f"(d) : "h"(x), "h"(y), "f"(c));
    return d;
}
__device__ __forceinline__ float dot8_i8_f16(uint2 x, uint4 q, float a) {
    const uint32_t w[2] = {x.x, x.y}, qw[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int h = 0; h < 4; ++h) {
        uint32_t v = __byte_perm(w[h >> 1], 0x64646464u, (h & 1) ? 0x7342 : 0x5140);
        const __half2 n = __hsub2(*reinterpret_cast<const __half2*>(&v), __half2half2(__ushort_as_half(0x6480)));
        v = *reinterpret_cast<const uint32_t*>(&n);
        a = fma_f32_f16(v, qw[h], false, a);
        a = fma_f32_f16(v, qw[h], true, a);
    }
    return a;
}

// 2^e as an fp32, e in [-126, 127]
__device__ __forceinline__ float pow2f(int e) { return __uint_as_float((uint32_t)(e + 127) << 23); }

template <int NQ, int RW, bool GATHER, bool RANGE, bool IMG = false>
__device__ __forceinline__ void scan_impl(const ScanParams& p, const RangeOut& ro) {
    static_assert(!(IMG && (GATHER || RANGE)), "the int8 filter serves flat top-k scans only");
    constexpr int kRowsPerWarp = RW;
    constexpr int kGroupRows = kConsumerWarps * RW;
    extern __shared__ __align__(128) unsigned char smem_scan[];
    unsigned char* smem = smem_scan;
    const int dq4 = p.ld >> 2;  // queries in shared memory: stride ld
    const ScanSmem L = scan_smem_layout(NQ, p.ld, p.P, p.ck, p.stages, GATHER ? p.nprobe : 0, kGroupRows, IMG);
    float* ring = reinterpret_cast<float*>(smem + L.ring);
    float* qs = reinterpret_cast<float*>(smem + L.queries);
    uint64_t* lists = reinterpret_cast<uint64_t*>(smem + L.lists);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + L.bars);
    uint64_t* empty = full + p.stages;
    long long* stage_group = reinterpret_cast<long long*>(empty + p.stages);  // dynamic mode: row group in each stage
    int* qcnt = reinterpret_cast<int*>(smem + L.misc);
    float* thr_s = reinterpret_cast<float*>(smem + L.misc) + NQ;
    int64_t* pbase = reinterpret_cast<int64_t*>(smem + L.prefix);
    uint32_t* prefix = reinterpret_cast<uint32_t*>(pbase + (GATHER ? p.nprobe : 0));
    uint64_t* rq = reinterpret_cast<uint64_t*>(smem + L.rescore);  // int8 filter: queued (row << 8 | query) pairs
    float* qc_s = reinterpret_cast<float*>(rq + kRescoreCap);       // [NQ][8] margin terms and scale of each query
    const int nc8 = (4 * p.ck - kImgHeader) >> 3;                   // int8 filter: 8-code words per image row
    uint4* qh_s = reinterpret_cast<uint4*>(qc_s + NQ * 8);          // [NQ][nc8] fp16 queries, 8 per uint4
    int* rq_cnt = reinterpret_cast<int*>(qh_s + NQ * nc8);

    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    auto stamp = [&](int i) {
        if (p.phase_ts && tid == kWarp && blockIdx.y == 0 && blockIdx.x < 1024) p.phase_ts[(size_t)blockIdx.x * 16 + i] = global_ns();
    };
    stamp(0);
    const int q0 = blockIdx.y * NQ;
    const int nqv = min(NQ, p.nq - q0);
    const int ld = p.ld, d4 = ld >> 2, ck = p.ck, ck4 = ck >> 2;
    const int k = p.k, P = p.P;
    const int qcap = P - k;
    // insertions into a queue between two checks: one per row of a group, or one per pair of a re-scoring round
    const int hw_mark = qcap - (IMG ? kRescoreChunk : kGroupRows);

    // ---- prologue: barriers, queries, empty lists ------------------------------------------
    if (tid == 0) {
        for (int s = 0; s < p.stages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], kConsumerWarps);
        }
        fence_mbar_init();
    }
    for (int i = tid; i < NQ * dq4; i += kScanThreads) {
        const int b = i / dq4, c = i - b * dq4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (b < nqv && c < d4) v = reinterpret_cast<const float4*>(p.queries + (size_t)(q0 + b) * ld)[c];
        reinterpret_cast<float4*>(qs)[i] = v;
    }
    for (int i = tid; i < NQ * P; i += kScanThreads) lists[i] = 0ull;
    if (tid < NQ) {
        qcnt[tid] = 0;
        thr_s[tid] = tid < nqv ? -INFINITY : INFINITY;
    }
    if (IMG && tid == 0) *rq_cnt = 0;
    int64_t total = p.nrows;
    GatherCtx G{prefix, pbase, p.perm, p.nprobe};
    if constexpr (GATHER && NQ == 1) {
        if (p.centroids) {
            // ---- fused K4: top-nprobe of the centroid scores, identical in every CTA of the group (coarse.cuh) ----
            const CoarseSmem CL = coarse_smem_layout(p.nlist, p.nprobe);
            unsigned char* scratch = reinterpret_cast<unsigned char*>(ring);  // the ring is idle until the producer starts
            uint32_t* ckeys = reinterpret_cast<uint32_t*>(scratch + CL.keys);
            uint64_t* sel = reinterpret_cast<uint64_t*>(scratch + CL.sel);
            const int nl = (int)p.nlist;
            __syncthreads();  // the query is in shared memory
            const int64_t per = (p.nlist + gridDim.x - 1) / gridDim.x;
            const int64_t c0 = (int64_t)blockIdx.x * per;
            uint32_t* gkeys = p.coarse_keys + (size_t)blockIdx.y * p.nlist;
            coarse_score_slice<kScanThreads>(p.centroids, ld, reinterpret_cast<const float4*>(qs), c0,
                                             min(p.nlist, c0 + per), gkeys, tid);
            stamp(1);
            group_arrive_wait(&p.coarse_count[blockIdx.y], gridDim.x);
            stamp(2);
            // (8 loads in flight per thread: one at a time, the L2 round trips of a 4096-list table alone took ~7 us)
            for (int base = 0; base < nl; base += kScanThreads * 8) {
                uint32_t v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const int i = base + u * kScanThreads + tid;
                    v[u] = i < nl ? __ldcg(gkeys + i) : 0u;
                }
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const int i = base + u * kScanThreads + tid;
                    if (i < nl) ckeys[i] = v[u];
                }
            }
            const int Pn = pow2_ceil(p.nprobe);
            for (int i = p.nprobe + tid; i < Pn; i += kScanThreads) sel[i] = 0ull;
            __syncthreads();
            block_radix_select<kScanThreads>(nl, p.nprobe, [&](int i) { return coarse_key64(ckeys[i], (uint32_t)i); },
                                             RadixScratch(scratch + CL.scratch), sel, tid, -1);
            auto probe_of = [](uint64_t key) { return (key >> 32) ? (int64_t)key_pos(key) : (int64_t)-1; };
            if (p.nprobe <= 128) {
                // few winners: the rank of a key among them (keys are distinct) is its place in the probe order
                for (int t0 = warp * 4; t0 < p.nprobe; t0 += (kScanThreads / 32) * 4) {
                    uint64_t key = 0ull;
                    if (lane < 4 && t0 + lane < p.nprobe) key = sel[t0 + lane];
                    const Rank4 rk = warp_rank4_desc(sel, p.nprobe, __shfl_sync(0xffffffffu, key, 0),
                                                     __shfl_sync(0xffffffffu, key, 1), __shfl_sync(0xffffffffu, key, 2),
                                                     __shfl_sync(0xffffffffu, key, 3));
                    const int myr = lane == 0 ? rk.r[0] : lane == 1 ? rk.r[1] : lane == 2 ? rk.r[2] : rk.r[3];
                    if (lane < 4 && t0 + lane < p.nprobe) pbase[myr] = probe_of(key);  // read back as the list id below
                }
            } else {
                bitonic_sort_desc<kScanThreads>(sel, Pn, 1, tid, -1);
                for (int j = tid; j < p.nprobe; j += kScanThreads) pbase[j] = probe_of(sel[j]);
            }
            fence_proxy_async();  // generic-proxy writes to the ring precede the bulk copies that will land there
            __syncthreads();
            stamp(3);
        }
    }
    if constexpr (GATHER) {
        if (warp == 0) {  // exclusive prefix sum of the probed list sizes
            uint32_t carry = 0;
            for (int base = 0; base < p.nprobe; base += 32) {
                const int j = base + lane;
                uint32_t sz = 0;
                if (j < p.nprobe) {
                    const int64_t lid = p.centroids ? pbase[j] : p.probes[(size_t)blockIdx.y * p.nprobe + j];
                    int64_t b = 0;
                    if (lid >= 0) {
                        b = p.list_off[lid];
                        sz = (uint32_t)(p.list_off[lid + 1] - b);
                    }
                    pbase[j] = b;
                }
                uint32_t inc = sz;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
                    if (lane >= o) inc += t;
                }
                if (j < p.nprobe) prefix[j] = carry + inc - sz;
                carry += __shfl_sync(0xffffffffu, inc, 31);
            }
            if (lane == 0) prefix[p.nprobe] = carry;
        }
    }
    __syncthreads();
    stamp(4);
    if constexpr (GATHER) total = prefix[p.nprobe];
    const int64_t ngroups = (total + kGroupRows - 1) / kGroupRows;
    const size_t stage_floats = (size_t)kGroupRows * ck;

    if (warp == 0) {
        // ================================ producer ==========================================
        int s = 0;
        uint32_t ph = 0;
        // Row index of this lane in group g.  Only the INDEX is produced here; the pointer arithmetic
        // that consumes the (global-memory) perm value happens one iteration later, so the load of
        // the next group's indices is in flight while this group's copies are issued.
        auto lookup = [&](int64_t g) -> int64_t {
            const int64_t pos = g * kGroupRows + lane;
            if (lane >= kGroupRows || pos >= total) return 0;
            return GATHER ? (int64_t)gather_row(G, (uint32_t)pos) : pos;
        };
        const bool dyn = p.group_count != nullptr;
        // next row group of this CTA: the shared dispenser (dynamic) or the static stride
        auto draw = [&](int64_t cur) -> int64_t {
            if (!dyn) return cur + gridDim.x;
            unsigned int v = 0;
            if (lane == 0) v = atomicAdd(&p.group_count[blockIdx.y], 1u);
            return (int64_t)__shfl_sync(0xffffffffu, v, 0);
        };
        int64_t g = dyn ? draw(0) : (int64_t)blockIdx.x;
        int64_t row_next = g < ngroups ? lookup(g) : 0;
        for (; g < ngroups;) {
            const int64_t p0 = g * kGroupRows;
            const int nvalid = (int)min((int64_t)kGroupRows, total - p0);
            const int64_t row = row_next;
            // the next group is drawn (and its row indices looked up) now, one iteration ahead: the atomic and the
            // CSR loads are in flight while this group's copies are issued
            const int64_t g_next = draw(g);
            if (g_next < ngroups) row_next = lookup(g_next);
            const float* src = IMG ? reinterpret_cast<const float*>(p.img) + (size_t)row * ck : p.rows + (size_t)row * ld;
            for (int ch = 0; ch < p.nchunks; ++ch) {
                if (lane == 0) {
                    mbar_wait(&empty[s], ph ^ 1u);
                    if (dyn) stage_group[s] = g;  // published to the consumers by the arrive below
                }
                __syncwarp();
                const int cfl = IMG ? ck : min(ck, ld - ch * ck);
                const uint32_t cbytes = (uint32_t)cfl * 4u;
                if (lane == 0) mbar_arrive_expect_tx(&full[s], cbytes * (uint32_t)nvalid);
                __syncwarp();
                float* dst = ring + (size_t)s * stage_floats;
                if (!GATHER && p.single_copy) {
                    if (lane == 0) bulk_g2s(dst, src, cbytes * (uint32_t)nvalid, &full[s]);
                } else if (GATHER && p.perm == nullptr && p.nchunks == 1) {
                    // rows are grouped by list: consecutive candidates are consecutive rows except at a list
                    // boundary, so each RUN of the group is one sequential copy (usually 1-2 per group)
                    const int64_t prev = __shfl_up_sync(0xffffffffu, row, 1);
                    const bool start = lane < nvalid && (lane == 0 || row != prev + 1);
                    const unsigned sm = __ballot_sync(0xffffffffu, start);
                    if (start) {
                        const unsigned higher = sm & ~((2u << lane) - 1u);
                        const int end = higher ? __ffs(higher) - 1 : nvalid;
                        bulk_g2s(dst + (size_t)lane * ck, src, cbytes * (uint32_t)(end - lane), &full[s]);
                    }
                } else if (lane < nvalid) {
                    bulk_g2s(dst + (size_t)lane * ck, src + (size_t)ch * ck, cbytes, &full[s]);
                }
                if (++s == p.stages) { s = 0; ph ^= 1u; }
            }
            g = g_next;
        }
        if (dyn && lane == 0) {  // end marker: the consumers learn that the dispenser is empty
            mbar_wait(&empty[s], ph ^ 1u);
            stage_group[s] = -1;
            mbar_arrive(&full[s]);
        }
    } else {
        // ================================ consumers =========================================
        const int cw = warp - 1;
        const int ctid = tid - kWarp;
        constexpr int V = kRowsPerWarp * NQ;
        constexpr int LV = Log2<V>::value;
        const float4* q4 = reinterpret_cast<const float4*>(qs);
        int s = 0;
        uint32_t ph = 0;
        const bool dyn = p.group_count != nullptr;
        // [list | queue] of every query sorted, queues emptied, thresholds tightened (all consumers, at a barrier)
        auto tighten = [&]() {
            if (NQ == 1 && p.rank_sort) rank_sort_desc<kConsumerThreads>(lists, P, ctid, kBarConsumers);
            else bitonic_sort_desc<kConsumerThreads>(lists, P, nqv, ctid, kBarConsumers);
            for (int i = ctid; i < nqv * qcap; i += kConsumerThreads) {
                const int l = i / qcap, j = i - l * qcap;
                lists[(size_t)l * P + k + j] = 0ull;
            }
            if (ctid < nqv) {
                qcnt[ctid] = 0;
                const uint64_t t = lists[(size_t)ctid * P + k - 1];
                thr_s[ctid] = t ? key_score(t) : -INFINITY;
            }
            named_bar_sync(kBarConsumers, kConsumerThreads);
        };
        // int8 filter.  Row x has the image s n (header: s, resid >= |x - s n|, xhat >= |s n|); query q is scaled by
        // 2^e (e per query: max |q_i| 2^e in [2^14, 2^15), e <= 126) and rounded to fp16, q^ = fp16(q 2^e), and the
        // approximation is approx = s 2^-e (q^ . n), the dot product summed in fp32 from exact products (FHFMA).  With
        // q' = 2^-e q^ and h = ld + 64 (the depth of every summation tree of the fp32 scan and of this sum, butterfly
        // included), gamma = 1.01 h 2^-24:
        //   |exact - approx| <= |q| resid                          quantisation residual: q . (x - s n)
        //                     + |q - q'| xhat                       query rounding: (q - q') . s n
        //                     + gamma |q| (resid + xhat)            the fp32 scan's sum (|x| <= resid + xhat)
        //                     + gamma |q'| xhat                     the fp32 sum of q^ . n (scaled by s 2^-e)
        //                     + 2^-21 |q'| xhat                     the two products forming approx, approx + margin
        //                     + h 2^-148                            underflow: every rounding above that lands below
        //                                                           2^-126 errs by at most 2^-150 absolute
        // With |q'| <= T = |q| + |q - q'| and g = 2 gamma + 2^-21 this is margin = A resid + B xhat + C, A = |q| + g T,
        // B = |q - q'| + g T, C = h 2^-148, all times 1.001 for the rounding of the norms (fp32 sums of squares, ld
        // 2^-149 added for the squares that underflowed), of A, B, C and of the margin itself.  The sum q^ . n cannot
        // underflow (its terms are multiples of 2^-24), and approx multiplies by 2^-e first when 2^-e > 1 (exactly) so
        // that an underflow of a product is never scaled up.  The bound assumes that no partial sum overflows: a pair
        // with T (resid + xhat) > 2^126 gets an infinite margin.  A NaN or Inf row (s = NaN) has a NaN approximation
        // and a NaN or Inf query a NaN or Inf margin: both are always re-scored.  One warp per query, before the first
        // group; qc_s[b] = {A, B, C, 2^-e, T}.
        unsigned long long nrescored = 0;
        if constexpr (IMG) {
            if (cw < NQ) {
                const float* qf = qs + (size_t)cw * ld;
                float s2 = 0.f, mx = 0.f;
                for (int t = lane; t < ld; t += 32) {
                    s2 = fmaf(qf[t], qf[t], s2);
                    mx = fmaxf(mx, fabsf(qf[t]));
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    s2 += __shfl_xor_sync(0xffffffffu, s2, o);
                    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
                }
                const int e = min(141 - (int)((__float_as_uint(mx) >> 23) & 0xffu), 126);
                float d2 = 0.f;
                __half* qh = reinterpret_cast<__half*>(qh_s + (size_t)cw * nc8);
                for (int t = lane; t < 8 * nc8; t += 32) {
                    const float x = t < ld ? qf[t] : 0.f;
                    const float v = e > 63 ? x * pow2f(63) * pow2f(e - 63) : x * pow2f(e);  // |v| < 2^15
                    const __half h = __float2half_rn(v);
                    qh[t] = h;
                    const float d = v - __half2float(h);  // exact
                    d2 = fmaf(d, d, d2);
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) d2 += __shfl_xor_sync(0xffffffffu, d2, o);
                if (lane == 0) {
                    const float h = (float)(ld + 64), lost = (float)ld * 0x1p-149f;
                    const float g = 2.f * 1.01f * h * 0x1p-24f + 0x1p-21f;
                    const float qs_e = pow2f(-e);
                    const float qn = sqrtf(s2 + lost);
                    // |q - q'|: the scaled rounding errors (v itself may have underflowed by 2^-150 when e <= 0), scaled
                    // back by 2^-e (that product may underflow by 2^-150 too).  2^-149 stands for 2^-150: nvcc folds the
                    // literal 0x1p-150f to +Inf.
                    const float dqn = (sqrtf(d2 + lost) + sqrtf((float)ld) * 0x1p-149f) * qs_e + 0x1p-149f;
                    const float T = qn + dqn;
                    float* c = qc_s + cw * 8;
                    c[0] = 1.001f * (qn + g * T);
                    c[1] = 1.001f * (dqn + g * T);
                    c[2] = 1.001f * h * 0x1p-148f;
                    c[3] = qs_e;
                    c[4] = T;
                }
            }
            named_bar_sync(kBarConsumers, kConsumerThreads);
        }
        // Re-score the queued pairs exactly, kRescoreChunk at a time (insertion as in the fp32 scan), and empty the
        // queue.  All consumers, at a barrier.
        auto rescore_queue = [&]() {
            const int n = *rq_cnt;
            nrescored += (unsigned long long)n;
            for (int c0 = 0; c0 < n; c0 += kRescoreChunk) {
                constexpr int J = kRescoreChunk / kConsumerWarps;
                uint64_t ent[J];
                bool valid[J];
#pragma unroll
                for (int j = 0; j < J; ++j) {
                    const int e = c0 + cw + kConsumerWarps * j;
                    valid[j] = e < n;
                    ent[j] = valid[j] ? rq[e] : 0ull;
                }
                float a[J];
                exact_scores<J>(p.rows, ld, q4, dq4, ent, valid, lane, a);
                bool hw = false;
#pragma unroll
                for (int j = 0; j < J; ++j) {
                    if (lane == j && valid[j]) {
                        const float score = a[j];
                        const int b = (int)(ent[j] & 0xff);
                        const uint32_t pos = (uint32_t)(ent[j] >> 8);
                        if (score >= thr_s[b]) {
                            const uint64_t key = make_key(score, pos);
                            if (key > lists[(size_t)b * P + k - 1] && row_allowed(p.allow, pos)) {
                                const int slot = atomicAdd(&qcnt[b], 1);
                                lists[(size_t)b * P + k + slot] = key;
                                hw = slot + 1 > hw_mark;
                            }
                        }
                    }
                }
                if (named_bar_or(kBarConsumers, kConsumerThreads, hw)) tighten();
            }
            if (ctid == 0 && n) *rq_cnt = 0;
            named_bar_sync(kBarConsumers, kConsumerThreads);
        };
        for (int64_t g = blockIdx.x; dyn || g < ngroups; g += gridDim.x) {
            float acc[V];
            float4 hdr;  // int8 filter: header {s, resid, xhat, 0} of this lane's row
#pragma unroll
            for (int i = 0; i < V; ++i) acc[i] = 0.f;
            if (dyn) {  // (whole-row stages only: one stage per group)
                mbar_wait(&full[s], ph);
                g = stage_group[s];
                if (g < 0) break;
            }
            for (int ch = 0; ch < p.nchunks; ++ch) {
                if (!dyn) mbar_wait(&full[s], ph);
                if constexpr (IMG) {  // whole image rows: 8 codes per 8-byte load, the header of this lane's row
                    const unsigned char* tile = reinterpret_cast<const unsigned char*>(ring + (size_t)s * stage_floats) +
                                                (size_t)(cw * kRowsPerWarp) * (4 * ck);
                    const uint2* codes = reinterpret_cast<const uint2*>(tile + kImgHeader);
#pragma unroll 2
                    for (int i = lane; i < nc8; i += 32) {
                        uint2 x[kRowsPerWarp];
#pragma unroll
                        for (int r = 0; r < kRowsPerWarp; ++r) x[r] = codes[r * (ck >> 1) + i];
#pragma unroll
                        for (int b = 0; b < NQ; ++b) {
                            const uint4 q = qh_s[b * nc8 + i];
#pragma unroll
                            for (int r = 0; r < kRowsPerWarp; ++r) acc[r * NQ + b] = dot8_i8_f16(x[r], q, acc[r * NQ + b]);
                        }
                    }
                    hdr = *reinterpret_cast<const float4*>(tile + (size_t)(((lane >> (5 - LV)) / NQ) * (4 * ck)));
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&empty[s]);
                    if (++s == p.stages) { s = 0; ph ^= 1u; }
                    continue;
                }
                const float4* tile =
                    reinterpret_cast<const float4*>(ring + (size_t)s * stage_floats) + (size_t)(cw * kRowsPerWarp) * ck4;
                const int c4n = min(ck4, d4 - ch * ck4);
                const float4* qb = q4 + ch * ck4;
#pragma unroll 2
                for (int i = lane; i < c4n; i += 32) {
                    float4 x[kRowsPerWarp];
#pragma unroll
                    for (int r = 0; r < kRowsPerWarp; ++r) x[r] = tile[r * ck4 + i];
#pragma unroll
                    for (int b = 0; b < NQ; ++b) {
                        const float4 q = qb[b * d4 + i];
#pragma unroll
                        for (int r = 0; r < kRowsPerWarp; ++r) {
                            float a = acc[r * NQ + b];
                            a = fmaf(x[r].x, q.x, a);
                            a = fmaf(x[r].y, q.y, a);
                            a = fmaf(x[r].z, q.z, a);
                            a = fmaf(x[r].w, q.w, a);
                            acc[r * NQ + b] = a;
                        }
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty[s]);
                if (++s == p.stages) { s = 0; ph ^= 1u; }
            }
            multi_reduce_step<V, 16>(acc, lane);
            const float score = acc[0];
            const int vi = lane >> (5 - LV);
            const bool owner = (lane & ((32 >> LV) - 1)) == 0;
            const int r = vi / NQ, b = vi % NQ;
            bool hw = false;
            if constexpr (RANGE) {
                if (owner && b < nqv) {
                    const int64_t cpos = g * kGroupRows + cw * kRowsPerWarp + r;
                    if (cpos < total && score > ro.thresh) {
                        uint32_t pos = GATHER ? gather_row(G, (uint32_t)cpos) : (uint32_t)cpos;
                        if (GATHER && p.row_pos) pos = p.row_pos[pos];
                        if (row_allowed(p.allow, pos)) {
                            const int slot = atomicAdd(&qcnt[b], 1);
                            lists[(size_t)b * P + slot] = make_key(score, pos);
                            hw = slot + 1 > hw_mark;
                        }
                    }
                }
                if (named_bar_or(kBarConsumers, kConsumerThreads, hw)) range_flush<NQ>(L, smem, lists, qcnt, P, q0, nqv, ctid, ro);
                continue;
            }
            if constexpr (IMG) {
                // queue the pair unless the bound shows that its exact score is below the threshold (a NaN or Inf
                // approximation, a non-finite margin and a threshold of -inf all queue it)
                bool full_q = false;
                if (owner && b < nqv) {
                    const int64_t cpos = g * kGroupRows + cw * kRowsPerWarp + r;
                    const float* c = qc_s + b * 8;
                    const float approx = c[3] > 1.f ? score * c[3] * hdr.x : score * hdr.x * c[3];
                    float margin = fmaf(c[0], hdr.y, fmaf(c[1], hdr.z, c[2]));
                    if (!(c[4] * (hdr.y + hdr.z) <= 0x1p126f)) margin = INFINITY;
                    if (cpos < total && row_allowed(p.allow, (uint32_t)cpos) &&
                        !(fabsf(approx) <= FLT_MAX && approx + margin < thr_s[b])) {
                        const int slot = atomicAdd(rq_cnt, 1);
                        rq[slot] = (uint64_t)cpos << 8 | (uint64_t)b;
                        full_q = slot + 1 > kRescoreCap - kGroupRows * NQ;
                    }
                }
                if (named_bar_or(kBarConsumers, kConsumerThreads, full_q)) rescore_queue();
                continue;
            }
            if (owner) {
                const int64_t cpos = g * kGroupRows + cw * kRowsPerWarp + r;
                if (cpos < total && score >= thr_s[b]) {
                    uint32_t pos = GATHER ? gather_row(G, (uint32_t)cpos) : (uint32_t)cpos;
                    if (GATHER && p.row_pos) pos = p.row_pos[pos];  // grouped store: ties go by INSERTION position
                    const uint64_t key = make_key(score, pos);
                    if (key > lists[(size_t)b * P + k - 1] && row_allowed(p.allow, pos)) {
                        const int slot = atomicAdd(&qcnt[b], 1);
                        lists[(size_t)b * P + k + slot] = key;
                        hw = slot + 1 > hw_mark;
                    }
                }
            }
            if (named_bar_or(kBarConsumers, kConsumerThreads, hw)) tighten();
        }
        // ---- epilogue: final sort, k best keys of this CTA for each query -------------------
        named_bar_sync(kBarConsumers, kConsumerThreads);
        stamp(5);
        if constexpr (RANGE) {
            range_flush<NQ>(L, smem, lists, qcnt, P, q0, nqv, ctid, ro);
            return;
        }
        if constexpr (IMG) {
            rescore_queue();
            if (ctid == 0 && nrescored) atomicAdd(p.rescored, nrescored);
        }
        if (NQ == 1 && p.rank_sort) rank_sort_desc<kConsumerThreads>(lists, P, ctid, kBarConsumers);
        else bitonic_sort_desc<kConsumerThreads>(lists, P, nqv, ctid, kBarConsumers);
        stamp(6);
        for (int i = ctid; i < nqv * k; i += kConsumerThreads) {
            const int l = i / k, j = i - l * k;
            p.parts[((size_t)(q0 + l) * p.nparts + blockIdx.x) * k + j] = lists[(size_t)l * P + j];
        }
        if (!p.fuse_tail) return;
        // ---- fused K3: the last CTA of this query group merges all nparts lists --------------------
        int& tail_last = reinterpret_cast<int*>(thr_s + NQ)[0];  // (no static shared memory: the layout fills the SM)
        int& tail_cnt = reinterpret_cast<int*>(thr_s + NQ)[1];
        __threadfence();  // my keys are visible device-wide before my arrival is
        named_bar_sync(kBarConsumers, kConsumerThreads);
        if (ctid == 0) {
            const unsigned int prev = atomicAdd(&p.tail_count[blockIdx.y], 1u);
            tail_last = prev == gridDim.x - 1;
            if (tail_last) {  // ready for the next launch on this stream (every CTA has drawn its last group by now)
                p.tail_count[blockIdx.y] = 0;
                if (p.group_count) p.group_count[blockIdx.y] = 0;
                if (p.coarse_count) p.coarse_count[blockIdx.y] = 0;  // every CTA of the group left that barrier long ago
            }
        }
        named_bar_sync(kBarConsumers, kConsumerThreads);
        stamp(7);
        if (!tail_last) return;
        __threadfence();
        uint64_t* buf = reinterpret_cast<uint64_t*>(ring);  // the ring is idle: every copy has landed and been consumed
        for (int l = 0; l < nqv; ++l) {
            const int64_t q = q0 + l;
            const uint64_t* src = p.parts + (size_t)q * p.nparts * k;
            const int64_t M = (int64_t)p.nparts * k;
            const uint64_t* best = buf;
            auto load2 = [&](int li, int r) { return __ldcg(src + (size_t)li * k + r); };
            if (!(p.heads_bytes && block_merge_heads<kConsumerThreads, GATHER>(reinterpret_cast<unsigned char*>(ring), k, p.nparts, load2,
                                                                       &tail_cnt, ctid, kBarConsumers, &best,
                                                                       p.phase_ts && blockIdx.y == 0 && blockIdx.x < 1024
                                                                           ? p.phase_ts + (size_t)blockIdx.x * 16 + 10
                                                                           : nullptr))) {
                best = buf;
                named_bar_sync(kBarConsumers, kConsumerThreads);
                if (!block_select_topk_lists<kConsumerThreads>(buf, p.S_merge, k, p.nparts, load2, &tail_cnt, ctid,
                                                               kBarConsumers)) {
                    named_bar_sync(kBarConsumers, kConsumerThreads);
                    block_select_topk<kConsumerThreads>(buf, p.S_merge, k, M, [&](int64_t c) { return __ldcg(src + c); },
                                                        &tail_cnt, ctid, kBarConsumers);
                }
            }
            if (l == 0) stamp(8);
            auto local = [&](int j, float& d, int64_t& id) {
                const uint64_t key = best[j];
                d = -FLT_MAX;
                id = -1;
                if (key) {
                    d = key_score(key);
                    const uint32_t pos = key_pos(key);
                    id = p.ids ? p.ids[pos] : (int64_t)pos;
                }
            };
            if (!p.exchange) {
                for (int j = ctid; j < k; j += kConsumerThreads) {
                    float d;
                    int64_t id;
                    local(j, d, id);
                    p.D[q * k + j] = d;
                    p.I[q * k + j] = id;
                }
                named_bar_sync(kBarConsumers, kConsumerThreads);  // buf is reused by the next query
            } else {
                // the local winners move to the second half of the buffer region: the exchange merge sorts in `buf`
                float* ld_s = reinterpret_cast<float*>(reinterpret_cast<unsigned char*>(ring) +
                                                       max((size_t)p.S_merge * 8, (size_t)p.heads_bytes));
                int64_t* li_s = reinterpret_cast<int64_t*>(ld_s + ((k + 1) & ~1));
                for (int j = ctid; j < k; j += kConsumerThreads) local(j, ld_s[j], li_s[j]);
                named_bar_sync(kBarConsumers, kConsumerThreads);
                exch_push_wait_merge<kConsumerThreads>(p.exch, q, buf, &tail_cnt, ctid, kBarConsumers,
                                                       [&](int j, float& d, int64_t& id) {
                                                           d = ld_s[j];
                                                           id = li_s[j];
                                                       });
            }
        }
        stamp(9);
    }
}

// The int8 image of n rows (row layout at kImgHeader), one warp per row.  s = max |x_i| / 127 (at least the smallest
// subnormal), n_i = rint(x_i / s) clamped to [-127, 127]; resid = |x - s n| and xhat = s |n| are summed in fp64 (every
// term exact) and rounded up to fp32, so rounding can only make them larger; an xhat beyond FLT_MAX becomes +Inf.
// An all-zero row has s = 0, n = 0, resid = xhat = 0; a row with a NaN or Inf element has s = NaN, n = 0 and
// resid = +Inf.  `rb` = img_row_bytes(ld).
__global__ void int8_image_kernel(const float* rows, int ld, int rb, int64_t n, uint8_t* out) {
    const int64_t r = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (r >= n) return;
    const float4* x4 = reinterpret_cast<const float4*>(rows + (size_t)r * ld);
    const int d4 = ld >> 2, w4 = (rb - kImgHeader) >> 2;  // float4s of the row, 4-code words of the image row
    float mx = 0.f;
    bool bad = false;
    for (int t = lane; t < d4; t += 32) {
        const float4 v = x4[t];
        const float a[4] = {fabsf(v.x), fabsf(v.y), fabsf(v.z), fabsf(v.w)};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            bad |= !(a[e] <= FLT_MAX);
            mx = fmaxf(mx, a[e]);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    bad = __any_sync(0xffffffffu, bad);
    const float s = bad ? NAN : mx == 0.f ? 0.f : fmaxf(mx / 127.f, 0x1p-149f);
    double r2 = 0.0, n2 = 0.0;
    uint32_t* w = reinterpret_cast<uint32_t*>(out + (size_t)r * rb + kImgHeader);
    for (int t = lane; t < w4; t += 32) {
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (t < d4) v = x4[t];
        const float f[4] = {v.x, v.y, v.z, v.w};
        uint32_t u = 0;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const float c = s > 0.f ? fminf(fmaxf(rintf(f[e] / s), -127.f), 127.f) : 0.f;  // (s NaN: 0)
            const double d = (double)f[e] - (double)s * (double)c;
            r2 = fma(d, d, r2);
            n2 = fma((double)c, (double)c, n2);
            u |= (uint32_t)((int)c + 128) << (8 * e);
        }
        w[t] = u;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        r2 += __shfl_xor_sync(0xffffffffu, r2, o);
        n2 += __shfl_xor_sync(0xffffffffu, n2, o);
    }
    if (lane == 0) {
        constexpr double up = 1.0 + 0x1p-30;  // the fp64 sums' and square roots' rounding
        const float resid = bad ? INFINITY : __double2float_ru(sqrt(r2) * up);
        const float xhat = bad ? 0.f : __double2float_ru((double)s * sqrt(n2) * up);
        *reinterpret_cast<float4*>(out + (size_t)r * rb) = make_float4(s, resid, xhat, 0.f);
    }
}

template <int NQ, int RW, bool GATHER, bool IMG = false>
__global__ void __launch_bounds__(kScanThreads, 1) scan_topk_kernel(const ScanParams p) {
    scan_impl<NQ, RW, GATHER, false, IMG>(p, RangeOut{});
}

// Range mode: P = the staging capacity per query, p.k = 0; no parts, no fused tail.
template <int NQ, int RW, bool GATHER>
__global__ void __launch_bounds__(kScanThreads, 1) scan_range_kernel(const ScanParams p, const RangeOut ro) {
    scan_impl<NQ, RW, GATHER, true>(p, ro);
}

}  // namespace wb
