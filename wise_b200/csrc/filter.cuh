// filter.cuh - filtered search (faiss SearchParameters with an IDSelector [faiss-upstream]): the selector evaluated
// into a bitmap over insertion positions, and the compaction of the selected rows for very selective filters.
//
// Every search kernel already knows the insertion position of each row it scores (it is the tie rule), so one bitmap
// over positions serves every path: the scan kernels test the bit of a row after its threshold compare, the
// tensor-core epilogues AND it into their row predicate (DESIGN.md "Filtered search").
#pragma once
#include <float.h>

#include "common.cuh"

namespace wb {

constexpr int kFilterTile = 128;  // positions per block of the evaluation kernel == rows per K2 tile (kGemmBM)

// bits[p / 32] bit p % 32 = selector(ids[p]) for p < n, one thread per position.  The selector is the sorted, unique
// id set set[0, nset) when `set` is given, else the range [imin, imax); `invert` negates it (IDSelectorNot).
// tile_cnt[t] = selected positions in [t * 128, (t + 1) * 128): the host's prefix of these drives the K2 epoch
// schedule and the compaction.
__global__ void __launch_bounds__(kFilterTile) filter_eval_kernel(const int64_t* ids, int64_t n, const int64_t* set,
                                                                  int64_t nset, int64_t imin, int64_t imax, int invert,
                                                                  uint32_t* bits, uint32_t* tile_cnt) {
    const int64_t pos = (int64_t)blockIdx.x * kFilterTile + threadIdx.x;
    bool in = false;
    if (pos < n) {
        const int64_t id = ids[pos];
        if (set) {
            int64_t lo = 0, hi = nset;  // first element >= id
            while (lo < hi) {
                const int64_t mid = (lo + hi) >> 1;
                if (set[mid] < id) lo = mid + 1;
                else hi = mid;
            }
            in = lo < nset && set[lo] == id;
        } else {
            in = id >= imin && id < imax;
        }
        in = in != (invert != 0);
    }
    const unsigned word = __ballot_sync(0xffffffffu, in);
    if ((threadIdx.x & 31) == 0 && pos < n) bits[pos >> 5] = word;
    const int cnt = __syncthreads_count(in);
    if (threadIdx.x == 0) tile_cnt[blockIdx.x] = (uint32_t)cnt;
}

// Stream compaction of the bitmap: selected position p goes to slot tile_off[p / 128] + (selected positions before p
// in its tile), so the slots keep insertion order.  pos_out[slot] = p, ids_out[slot] = ids[p].
__global__ void __launch_bounds__(kFilterTile) filter_positions_kernel(const uint32_t* bits, int64_t n,
                                                                       const int64_t* tile_off, const int64_t* ids,
                                                                       int64_t* pos_out, int64_t* ids_out) {
    const int64_t pos = (int64_t)blockIdx.x * kFilterTile + threadIdx.x;
    if (pos >= n) return;
    const uint32_t word = bits[pos >> 5];
    const int lane = threadIdx.x & 31;
    if (!((word >> lane) & 1u)) return;
    int before = __popc(word & ((1u << lane) - 1u));
    const int64_t w0 = (pos >> 5) & ~(int64_t)(kFilterTile / 32 - 1);  // first word of the tile
    for (int64_t w = w0; w < (pos >> 5); ++w) before += __popc(bits[w]);
    const int64_t slot = tile_off[blockIdx.x] + before;
    pos_out[slot] = pos;
    ids_out[slot] = ids[pos];
}

// (D, I)[n] <- (-FLT_MAX, -1): the result of a search whose filter selects no row
__global__ void pad_results_kernel(float* D, int64_t* I, int64_t n) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) {
        D[i] = -FLT_MAX;
        I[i] = -1;
    }
}

// Is insertion position `pos` selected?  (allow == null: no filter)
__device__ __forceinline__ bool row_allowed(const uint32_t* allow, uint32_t pos) {
    return !allow || ((allow[pos >> 5] >> (pos & 31)) & 1u);
}

}  // namespace wb
