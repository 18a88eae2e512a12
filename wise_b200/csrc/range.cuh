// range.cuh - range search (faiss Index::range_search [faiss-upstream]): every row whose inner product with the query
// is strictly above a threshold, in score-descending / insertion-position-ascending order (DESIGN.md "Range search").
//
// The scan kernels find the hits (scan.cuh scan_range_kernel for K1 / K5; the K2 epochs with range_collect_kernel
// below) and append make_key(score, pos) to a pool tagged with the query.  Then, per chunk of queries:
//   range_scatter_kernel      groups the pool by query (lims = exclusive prefix of the per-query counts);
//   range_block_sort_kernel   sorts runs of at most kRangeRun keys of one query in shared memory;
//   range_merge_kernel        merges pairs of sorted runs of a query, run width doubling per pass, until the
//                             longest query is one run (each key finds its rank in the other run by bisection:
//                             keys of one query are distinct, so ranks are unique and the result is deterministic);
//   range_emit_kernel         turns keys into (D, I).
// A sharded range search merges the per-rank (D, I) with range_merge_parts_kernel.
#pragma once
#include "merge.cuh"
#include "scan.cuh"

namespace wb {

// Keys one CTA sorts in shared memory (64 KB): the cut-off between the block sort and the merge passes.
constexpr int kRangeRun = 8192;
constexpr int kRangeThreads = 256;

// K2 range epoch set-up: every real query has threshold `thresh`, padding queries +inf; no candidates yet.
__global__ void range_gemm_init_kernel(float* thr, int nq, int nq_pad, float thresh, int* cnt) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nq_pad) thr[i] = i < nq ? thresh : INFINITY;
    if (i < nq) cnt[i] = 0;
}

// K2 range epoch boundary (replaces compact_topk_kernel): the candidates of query blockIdx.x carry exact fp32 scores
// (rescore_candidates_kernel ran first); those above the threshold go to the pool, and the candidate list is emptied.
// When a candidate list of this epoch overflowed (*overflow) the epoch contributes nothing: *need records the largest
// candidate count (counting continued past `cap`) and the host re-runs the epoch with that capacity.
struct RangeCollect {
    const uint64_t* keys;  // [nq][kstride] candidates
    int* cnt;              // [nq]
    int cap, kstride;
    const int* overflow;
    int* need;
    RangeOut out;
};

__global__ void __launch_bounds__(kRangeThreads) range_collect_kernel(const RangeCollect c) {
    __shared__ int wsum[kRangeThreads / 32];
    __shared__ unsigned long long sbase;
    const int q = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int n = c.cnt[q];
    __syncthreads();  // every thread has read the count before it is reset below
    if (*c.overflow) {
        if (tid == 0) {
            atomicMax(c.need, n);
            c.cnt[q] = 0;
        }
        return;
    }
    const uint64_t* cand = c.keys + (size_t)q * c.kstride;
    for (int i0 = 0; i0 < n; i0 += kRangeThreads) {
        const int i = i0 + tid;
        const uint64_t key = i < n ? cand[i] : 0ull;
        const bool pass = key != 0ull && key_score(key) > c.out.thresh;
        const unsigned m = __ballot_sync(0xffffffffu, pass);
        if (lane == 0) wsum[warp] = __popc(m);
        __syncthreads();
        int before = 0, tot = 0;
        for (int w = 0; w < kRangeThreads / 32; ++w) {
            before += w < warp ? wsum[w] : 0;
            tot += wsum[w];
        }
        if (tid == 0 && tot) {
            sbase = atomicAdd(c.out.cursor, (unsigned long long)tot);
            atomicAdd(&c.out.count[q], (unsigned long long)tot);
        }
        __syncthreads();
        if (pass) {
            const unsigned long long slot = sbase + (unsigned long long)(before + __popc(m & ((1u << lane) - 1u)));
            if (slot < (unsigned long long)c.out.cap) {
                c.out.keys[slot] = key;
                c.out.qid[slot] = (uint32_t)(c.out.qbase + q);
            }
        }
        __syncthreads();  // wsum / sbase are reused by the next round
    }
    if (tid == 0) c.cnt[q] = 0;
}

// Group the pool by query: out[off[q] + (arrival order)] = key.  The order inside a query is settled by the sort.
__global__ void range_scatter_kernel(const uint64_t* keys, const uint32_t* qid, int64_t total, const int64_t* off,
                                     unsigned int* fill, uint64_t* out) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= total) return;
    const uint32_t q = qid[i];
    out[off[q] + atomicAdd(&fill[q], 1u)] = keys[i];
}

// Sort run blockIdx.x - keys[run_start[b], run_start[b] + run_len[b]) - descending in shared memory.
__global__ void __launch_bounds__(kRangeThreads) range_block_sort_kernel(uint64_t* keys, const int64_t* run_start,
                                                                        const int* run_len) {
    extern __shared__ __align__(16) unsigned char smem_range[];
    uint64_t* buf = reinterpret_cast<uint64_t*>(smem_range);
    const int tid = threadIdx.x;
    const int n = run_len[blockIdx.x];
    uint64_t* src = keys + run_start[blockIdx.x];
    const int P = max(2, pow2_ceil(n));
    for (int i = tid; i < P; i += kRangeThreads) buf[i] = i < n ? src[i] : 0ull;  // 0 (empty) sorts last
    __syncthreads();
    bitonic_sort_desc<kRangeThreads>(buf, P, 1, tid, -1);
    __syncthreads();
    for (int i = tid; i < n; i += kRangeThreads) src[i] = buf[i];
}

// One merge pass: inside every query (off[nq + 1]), sorted runs of width w are merged pairwise into runs of 2w.
__global__ void range_merge_kernel(const uint64_t* in, uint64_t* out, const int64_t* off, int nq, int64_t total,
                                   int64_t w) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= total) return;
    int lo = 0, hi = nq - 1;  // the query of entry i: the largest s with off[s] <= i
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (off[mid] <= i) lo = mid;
        else hi = mid - 1;
    }
    const int64_t b = off[lo], n = off[lo + 1] - b, l = i - b;
    const uint64_t key = in[i];
    const int64_t r = l / w, pstart = (r ^ 1) * w;
    if (pstart >= n) {  // no partner run (this run is the last of the query, or the query is one run)
        out[i] = key;
        return;
    }
    int64_t a = pstart, e = min(pstart + w, n);  // keys of the partner run larger than `key`
    while (a < e) {
        const int64_t mid = (a + e) >> 1;
        if (in[b + mid] > key) a = mid + 1;
        else e = mid;
    }
    out[b + (r & ~(int64_t)1) * w + (l - r * w) + (a - pstart)] = key;
}

__global__ void range_emit_kernel(const uint64_t* keys, int64_t total, const int64_t* ids, float* D, int64_t* I) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= total) return;
    const uint64_t key = keys[i];
    const uint32_t pos = key_pos(key);
    D[i] = key_score(key);
    I[i] = ids ? ids[pos] : (int64_t)pos;
}

// Sharded range search: merge the range results of the same nq queries from gridDim.y parts (ranks).  Part p's hits
// for query q are entries p * stride + [lp[q], lp[q + 1]) of Dp / Ip, lp = lims_parts + p * (nq + 1), in the order
// range_emit_kernel writes them.  Entry i of part p goes to lims[q] + (i - lp[q]) plus, for every other part, the
// number of its entries of query q that come first: a larger score (parts after p) or a larger or equal score (parts
// before p).  Scores compare as order_f32 bits, the map make_key uses, so equal scores tie by part, then by position
// inside the part: the single-index order when part p holds the p-th contiguous slice of the rows.  The output is a
// permutation of the input, found by bisection alone.
__global__ void range_merge_parts_kernel(const int64_t* lims_parts, int64_t nq, int64_t stride, const float* Dp,
                                         const int64_t* Ip, const int64_t* lims, float* D, int64_t* I) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int p = blockIdx.y;
    const int64_t* lp = lims_parts + (size_t)p * (nq + 1);
    if (i >= stride || i >= lp[nq]) return;
    int64_t lo = 0, hi = nq - 1;  // the query of entry i: the largest q with lp[q] <= i
    while (lo < hi) {
        const int64_t mid = (lo + hi + 1) >> 1;
        if (lp[mid] <= i) lo = mid;
        else hi = mid - 1;
    }
    const int64_t q = lo;
    const float d = Dp[(size_t)p * stride + i];
    const uint32_t key = order_f32(d);
    int64_t out = lims[q] + (i - lp[q]);
    for (int o = 0; o < (int)gridDim.y; ++o) {
        if (o == p) continue;
        const int64_t* lo_lims = lims_parts + (size_t)o * (nq + 1);
        const float* Do = Dp + (size_t)o * stride;
        const int64_t b = lo_lims[q];
        int64_t a = b, e = lo_lims[q + 1];  // the run of part o is sorted: the entries before this one are a prefix
        while (a < e) {
            const int64_t mid = (a + e) >> 1;
            const uint32_t km = order_f32(Do[mid]);
            if (o < p ? km >= key : km > key) a = mid + 1;
            else e = mid;
        }
        out += a - b;
    }
    D[out] = d;
    I[out] = Ip[(size_t)p * stride + i];
}

}  // namespace wb
