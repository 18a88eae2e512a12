// ivf_lm.cuh - K5 for BATCHES: list-major scan of the inverted lists.
//
// Replaces the batched form of faiss IndexIVF::search_preassigned + IVFFlatScanner::scan_codes [faiss-upstream]
// (reached from /root/reference/src/index/feature_search_index.py:113 with n > 1).  The query-major kernel
// (scan_topk_kernel<1, RW, true>) streams the probed lists of ONE query per CTA group, so a list probed by m queries
// is read m times: at nq = 256, nprobe = 128 over nlist = 4096 that is 8x the distinct bytes.  Here the probe table is
// inverted on the device (csr.cuh: the (query, probe) pairs grouped by list) and persistent CTAs pull work items
// (list, group of up to NQ of the queries that probe it): the rows of a list are streamed ONCE per group of 8 queries,
// with the same machinery as the flat scan - bulk async copies into a shared-memory ring, 128-bit LDS, register
// accumulators, fused top-k with a running threshold.
//   * every item writes the k best keys of each of its queries to parts[query][probe slot][k]; merge_topk_kernel then
//     merges the nprobe sorted lists of a query (K3), exactly as it merges per-CTA lists;
//   * thresholds are shared through global memory: a finished item publishes, per query, the k-th best score it found
//     (atomicMax) - a LOWER bound of the query's final k-th best score - and later items start from it, so almost every
//     row dies on one register compare.  Rows that tie with the bound are kept; publication order only changes how
//     much is pruned, never the result.
// HBM-bound; algorithmic bytes = sum over (list, query group) items of len(list) * ld * 4.
#pragma once
#include "scan.cuh"

namespace wb {

struct LmParams {
    const float* rows;        // row store, physically grouped by list
    int ld;
    const float* queries;     // [nq, ld]
    int nq, k, P, stages, nprobe;
    int64_t nlist;
    const int64_t* list_off;  // [nlist + 1] rows of each list
    const uint32_t* row_pos;  // storage row -> insertion position (null: identity)
    const uint32_t* allow;    // filtered search: bitmap over insertion positions (filter.cuh); null: every row
    const int64_t* pl_off;    // [nlist + 1] (query, probe) pairs of each list
    const uint32_t* pair_src; // [npairs] pair = query * nprobe + probe slot, grouped by list (queries ascending)
    const int64_t* item_off;  // [nlist + 1] first work item of each list; item_off[nlist] = number of items
    const int32_t* item_list; // [items] list of each work item
    uint32_t* gthr;           // [nq] order_f32 bits of the best known lower bound of the final k-th score (0: none)
    unsigned int* counter;    // work-item dispenser (zero at launch)
    uint64_t* parts;          // [nq][nprobe][k] keys
};

// nitems[l] = ceil(pairs of list l / NQ)
__global__ void lm_item_count_kernel(const int64_t* pl_off, int64_t nlist, int nqg, int64_t* nitems) {
    const int64_t l = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (l < nlist) nitems[l] = (pl_off[l + 1] - pl_off[l] + nqg - 1) / nqg;
}
__global__ void lm_item_fill_kernel(const int64_t* item_off, int64_t nlist, int32_t* item_list) {
    const int64_t l = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (l < nlist)
        for (int64_t i = item_off[l]; i < item_off[l + 1]; ++i) item_list[i] = (int32_t)l;
}

template <int NQ, int RW>
__global__ void __launch_bounds__(kScanThreads, 1) ivf_listmajor_kernel(const LmParams p) {
    constexpr int kGroupRows = kConsumerWarps * RW;
    extern __shared__ __align__(128) unsigned char smem_lm[];
    const int ld = p.ld, d4 = ld >> 2;
    const ScanSmem L = scan_smem_layout(NQ, ld, p.P, ld, p.stages, 0, kGroupRows);
    float* ring = reinterpret_cast<float*>(smem_lm + L.ring);
    float* qs = reinterpret_cast<float*>(smem_lm + L.queries);
    uint64_t* lists = reinterpret_cast<uint64_t*>(smem_lm + L.lists);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem_lm + L.bars);
    uint64_t* empty = full + p.stages;
    int* qcnt = reinterpret_cast<int*>(smem_lm + L.misc);
    float* thr_s = reinterpret_cast<float*>(smem_lm + L.misc) + NQ;
    int* item_s = reinterpret_cast<int*>(thr_s + NQ);  // [0] current work item
    uint32_t* pair_s = reinterpret_cast<uint32_t*>(item_s + 4);  // [NQ] (query, probe) pair of each query of the item

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int k = p.k, P = p.P;
    const int qcap = P - k;
    const int hw_mark = qcap - kGroupRows;
    const size_t stage_floats = (size_t)kGroupRows * ld;

    if (tid == 0) {
        for (int s = 0; s < p.stages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], kConsumerWarps);
        }
        fence_mbar_init();
    }
    __syncthreads();
    const int64_t nitems = p.item_off[p.nlist];
    int s = 0;  // ring position and phase: producer and consumers walk the ring in lockstep across items
    uint32_t ph = 0;
    for (;;) {
        if (tid == 0) item_s[0] = (int)atomicAdd(p.counter, 1u);
        __syncthreads();
        const int64_t item = item_s[0];
        if (item >= nitems) break;
        const int64_t l = p.item_list[item];
        const int64_t first = p.pl_off[l] + (item - p.item_off[l]) * NQ;
        const int cnt = (int)min((int64_t)NQ, p.pl_off[l + 1] - first);
        const int64_t row0 = p.list_off[l];
        const int64_t total = p.list_off[l + 1] - row0;
        const int64_t ngroups = (total + kGroupRows - 1) / kGroupRows;
        // ---- item setup: the group's queries, empty lists, thresholds from the shared lower bounds ---------
        if (tid < NQ) {
            const uint32_t pair = tid < cnt ? p.pair_src[first + tid] : 0u;
            pair_s[tid] = pair;
            qcnt[tid] = 0;
            float t = INFINITY;  // padding slots admit nothing
            if (tid < cnt) {
                const uint32_t g = __ldcg(&p.gthr[pair / (uint32_t)p.nprobe]);
                t = g ? unorder_f32(g) : -INFINITY;
            }
            thr_s[tid] = t;
        }
        __syncthreads();
        for (int i = tid; i < NQ * d4; i += kScanThreads) {
            const int b = i / d4, c = i - b * d4;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (b < cnt) v = reinterpret_cast<const float4*>(p.queries + (size_t)(pair_s[b] / (uint32_t)p.nprobe) * ld)[c];
            reinterpret_cast<float4*>(qs)[i] = v;
        }
        for (int i = tid; i < NQ * P; i += kScanThreads) lists[i] = 0ull;
        __syncthreads();

        if (warp == 0) {
            // ================================ producer: one contiguous copy per row group ==============
            for (int64_t g = 0; g < ngroups; ++g) {
                const int nvalid = (int)min((int64_t)kGroupRows, total - g * kGroupRows);
                if (lane == 0) {
                    mbar_wait(&empty[s], ph ^ 1u);
                    const uint32_t bytes = (uint32_t)nvalid * (uint32_t)ld * 4u;
                    mbar_arrive_expect_tx(&full[s], bytes);
                    bulk_g2s(ring + (size_t)s * stage_floats, p.rows + (size_t)(row0 + g * kGroupRows) * ld, bytes, &full[s]);
                }
                __syncwarp();
                if (++s == p.stages) { s = 0; ph ^= 1u; }
            }
        } else {
            // ================================ consumers (as in scan_topk_kernel) ========================
            const int cw = warp - 1;
            const int ctid = tid - kWarp;
            constexpr int V = RW * NQ;
            constexpr int LV = Log2<V>::value;
            const float4* q4 = reinterpret_cast<const float4*>(qs);
            for (int64_t g = 0; g < ngroups; ++g) {
                float acc[V];
#pragma unroll
                for (int i = 0; i < V; ++i) acc[i] = 0.f;
                mbar_wait(&full[s], ph);
                const float4* tile = reinterpret_cast<const float4*>(ring + (size_t)s * stage_floats) + (size_t)(cw * RW) * d4;
#pragma unroll 2
                for (int i = lane; i < d4; i += 32) {
                    float4 x[RW];
#pragma unroll
                    for (int r = 0; r < RW; ++r) x[r] = tile[r * d4 + i];
#pragma unroll
                    for (int b = 0; b < NQ; ++b) {
                        const float4 q = q4[b * d4 + i];
#pragma unroll
                        for (int r = 0; r < RW; ++r) {
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
                multi_reduce_step<V, 16>(acc, lane);
                const float score = acc[0];
                const int vi = lane >> (5 - LV);
                const bool owner = (lane & ((32 >> LV) - 1)) == 0;
                const int r = vi / NQ, b = vi % NQ;
                bool hw = false;
                if (owner) {
                    const int64_t cpos = g * kGroupRows + cw * RW + r;
                    if (cpos < total && score >= thr_s[b]) {
                        uint32_t pos = (uint32_t)(row0 + cpos);
                        if (p.row_pos) pos = p.row_pos[pos];  // ties go by INSERTION position
                        const uint64_t key = make_key(score, pos);
                        if (key > lists[(size_t)b * P + k - 1] && row_allowed(p.allow, pos)) {
                            const int slot = atomicAdd(&qcnt[b], 1);
                            lists[(size_t)b * P + k + slot] = key;
                            hw = slot + 1 > hw_mark;
                        }
                    }
                }
                if (named_bar_or(kBarConsumers, kConsumerThreads, hw)) {
                    bitonic_sort_desc<kConsumerThreads>(lists, P, cnt, ctid, kBarConsumers);
                    for (int i = ctid; i < cnt * qcap; i += kConsumerThreads) {
                        const int li = i / qcap, j = i - li * qcap;
                        lists[(size_t)li * P + k + j] = 0ull;
                    }
                    if (ctid < cnt) {
                        qcnt[ctid] = 0;
                        const uint64_t t = lists[(size_t)ctid * P + k - 1];
                        // the list's own k-th best, but never below the shared bound the item started from
                        if (t) thr_s[ctid] = fmaxf(thr_s[ctid], key_score(t));
                    }
                    named_bar_sync(kBarConsumers, kConsumerThreads);
                }
            }
            // ---- item epilogue: k best keys of every query of the group, publish the bounds ---------------
            named_bar_sync(kBarConsumers, kConsumerThreads);
            bitonic_sort_desc<kConsumerThreads>(lists, P, cnt, ctid, kBarConsumers);
            for (int i = ctid; i < cnt * k; i += kConsumerThreads) {
                const int li = i / k, j = i - li * k;
                p.parts[(size_t)pair_s[li] * k + j] = lists[(size_t)li * P + j];
            }
            if (ctid < cnt) {
                const uint64_t kth = lists[(size_t)ctid * P + k - 1];
                if (kth) atomicMax(&p.gthr[pair_s[ctid] / (uint32_t)p.nprobe], (uint32_t)(kth >> 32));
            }
        }
        __syncthreads();  // item boundary: qs / lists / pair_s / item_s are rewritten by the next item
    }
}

}  // namespace wb
