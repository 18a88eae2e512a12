// gemm.cuh - K2 flat_gemm_topk: batched exhaustive inner product on the 5th-gen tensor cores
// (tcgen05.mma kind::tf32, 3xTF32 split for fp32 accuracy) with a fused top-k filter epilogue.
//
// Replaces faiss exhaustive_inner_product_blas (sgemm tiles + heap/reservoir add_results)
// [faiss-upstream], the n >= 20 branch of knn_inner_product reached from
// /root/reference/src/index/feature_search_index.py:113, and serves the same contraction for the
// IVF coarse quantizer / add-time assignment and the k-means assignment (k = 1).
//
// S[row, q] = sum_t X[row, t] * Q[q, t],  X = database rows (A operand, M = 128 rows per tile),
// Q = a block of BN = 16 / 32 / 64 / 128 queries (B operand), both K-major.  x*y ~= xh*yh + xh*yl + xl*yh with
// xh = tf32-truncated x, xl = x - xh (exact in fp32): three terms per k-step into one fp32 accumulator in TMEM
// (issued as two MMAs for BN <= 64, see FOLD); the dropped xl*yl term is < 2^-20 relative.
// TERMS = 1 ("filter" epochs of a search, see the kernel): only xh*yh, candidates re-scored exactly afterwards.
//
// One persistent CTA per SM, 16 warps:
//   warp 0      producer A: per 32-float k-chunk one 2-D TMA load of the raw fp32 row tile
//                          (128 x 128 B, SWIZZLE_128B) into a deep ring freed by the transform warps
//   warp 3      producer B: one bulk copy of the pre-split query image per chunk into the operand slots
//   warps 4-7, 12-15 transform (two sets on alternate chunks): thread = row; reads its 128 B of the swizzled tile
//                          (conflict-free), splits hi/lo and stores both straight into TENSOR MEMORY (tcgen05.st):
//                          the A operand never goes back to shared memory
//   warp 1      MMA      : waits on ONE barrier per slot (4 transform arrivals + the image's transaction bytes), one
//                          elected thread issues the chunk's tcgen05.mma (A from TMEM, B from a no-swizzle K-major
//                          shared-memory descriptor); tcgen05.commit releases the slot
//   warps 8-11  epilogue : tcgen05.ld of the finished tile (double-buffered in TMEM, so it overlaps the next
//                          tile's MMAs); a score survives only if it beats the query's current k-th best
//                          (minus the filter margin for TERMS = 1); survivors are appended to a per-query
//                          candidate list in global memory (warp-aggregated atomics)
//   warp 2      TMEM allocator.
// Scores never go to HBM.  The host runs the database in growing "epochs"; between epochs
// compact_topk_kernel (merge.cuh) folds the candidates into the per-query top-k and tightens the
// thresholds; an epoch yields ~k * growth (~1000) candidates per query.
// Algorithmic work: 2*nq*N*d flop (3x that is issued in 3xTF32 epochs, 1x in filter epochs).
#pragma once
#include <cuda.h>  // CUtensorMap (types only; the encoder is fetched with cudaGetDriverEntryPoint)

#include "common.cuh"
#include "filter.cuh"

namespace wb {

constexpr int kGemmBM = 128;      // database rows per tile (UMMA M)
constexpr int kGemmBK = 32;       // floats per k-chunk (128 B = one swizzle-128B row)
constexpr int kGemmThreads = 512;
constexpr int kGemmABytes = kGemmBM * kGemmBK * 4;       // 16 KB raw row tile
constexpr int kTmemCols = 512;
constexpr int kBarEpilogue = 2;
// Dynamic work distribution (search mode of the 1-CTA kernel): producer A draws (row tile, query block) items from a
// global dispenser and hands them to the other roles through a small shared-memory queue.  The kernel is HBM-bound at
// small batches and SMs stream at different rates: with the static interleave the fastest SM idled for a quarter of the
// kernel (ncu, batch 16: SMs active 87 % on average, 75 % minimum).
constexpr int kGemmWQ = 8;

// Per query-block width BN (UMMA N = 16 / 32 / 64 / 128): small batches use a narrow block so the kernel
// stays bound by the HBM stream of the rows instead of by padded MMAs and query-image traffic.
//
// Timing-only experiment knobs for the 1-CTA kernel (results are WRONG when set; never defined in the product build):
// bit 0: the transform skips LDS + split (stores zeros); bit 1: it also skips the TMEM stores; bit 2: the MMA thread
// skips the MMAs and only commits.  Used to locate the ~600-cycle per-chunk cost (profiles/r01/gemm_experiments.md).
#ifndef WB_GEMM_EXP
#define WB_GEMM_EXP 0
#endif
#ifndef WB_GEMM_SLOTS
#define WB_GEMM_SLOTS(BN) 7  // experiment knob: same-box A/B of 7/6, 6/5 and 5/4 slots (BN 32/64) showed no difference
#endif
// FOLD (search mode, BN <= 64): every tcgen05.mma costs the tensor pipe ~45 cycles however small N is (measured:
// 12 MMAs of N = 32 per chunk = 540 cycles > the 508 cycles HBM allows a chunk at 1.55 GHz), so the three split
// terms are issued as TWO instructions per k-step: A_hi x [Q_hi ; Q_lo] (N = 2*BN, the lo image stacked under the hi
// image as extra operand rows) and A_lo x Q_hi (N = BN, the first rows of the same descriptor).  The accumulator
// tile is then 2*BN columns wide - [hi.hi + lo.hi | hi.lo] - and the epilogue adds the two halves.
template <int BN, bool ARGMAX>
constexpr bool kGemmFold = !ARGMAX && BN <= 64;
template <int BN, bool FOLD = false>
struct GemmCfg {
    static constexpr int kBBytes = 2 * BN * kGemmBK * 4;             // hi image + lo image of one k-chunk
    static constexpr int kDCols = FOLD ? 2 * BN : BN;                 // accumulator columns per buffer
    static constexpr int kTmemAOff = 2 * kDCols;                      // TMEM: D0 | D1 | A ring (64 columns per slot)
    // Ring 2 ("operand slots"): query image chunk in shared memory + split A operand in TMEM.  ONE barrier per slot
    // collects the 4 transform-warp arrivals and the image copy's transaction bytes, so the MMA thread - a serial
    // instruction stream that is on the critical path at small BN - waits once per chunk; freed by tcgen05.commit.
    // (A deeper, separate image ring was measured and did not help: the refill latency is not the limiter.)
    // The slot count is not critical (measured: 5 slots + 11 raw stages == 7 slots + 10 raw stages at BN = 32).
    static constexpr int kSlotsTmem = (kTmemCols - kTmemAOff) / 64;  // 4 / 6 / 7 for BN = 128 / 64 / 32
    static constexpr int kSlots = kSlotsTmem < WB_GEMM_SLOTS(BN) ? kSlotsTmem : WB_GEMM_SLOTS(BN);
    // Ring 1: raw fp32 row tiles straight from TMA; freed by the transform warps, so it can run far ahead of
    // the MMAs - it is what keeps enough bytes in flight to cover the loaded HBM latency (~3.5 us).
    static constexpr int kRawStages = (224 * 1024 - kSlots * kBBytes) / kGemmABytes;
    static constexpr int kNumBars = 2 * kRawStages + 2 * kSlots + 4 + 2 * kGemmWQ;
    static constexpr size_t kSmemBytes =
        1024 + (size_t)kRawStages * kGemmABytes + (size_t)kSlots * kBBytes + kNumBars * 8 + 16 + 2 * BN * 4 + kGemmWQ * 8;
    static_assert(kSmemBytes <= 232448, "shared memory budget");
};

struct GemmParams {
    int64_t row_begin, row_end;   // this epoch's rows (row_begin is a multiple of 128)
    int nchunks;                  // ceil(ld / 32)
    int nq;                       // real queries
    int nqb;                      // query blocks of BN queries
    // ARGMAX mode (K4 add-time assignment, K6 k-means assignment): rows = points, queries = centroids;
    // each row keeps a running (max score, lowest index) over all query blocks - no candidate lists.
    int32_t* assign_out;          // [rows] argmax query index
    float* best_out;              // [rows] its score
    const float* bimg;            // [nqb][nchunks][2][8][BN][4] pre-split query images
    const float* thr;             // [nqb*BN] current k-th best score per query (+inf for padding)
    const float* margin;          // [nqb*BN] TERMS == 1 only: bound on |exact - one-term score| per query
    uint64_t* keys;               // [nq][kstride]: [0,k) current top-k, [k, k+cap) candidates
    int* cnt;                     // [nq] candidates appended so far
    int* overflow;                // set when a candidate list ran out of room
    int k, cap, kstride;
    unsigned int* work_counter;   // dynamic work dispenser of this launch (zero at launch); null: static interleave
    const uint32_t* allow;        // filtered search: bitmap over rows (= insertion positions); null: every row
};

// ---- tcgen05 / TMA PTX -----------------------------------------------------------------------
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
            smem_u32(dst)),
        "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar))
        : "memory");
}

__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}

// D[tmem] (+)= A[tmem] * B[smem desc]^T, tf32 inputs, fp32 accumulate
__device__ __forceinline__ void umma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                             uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n"
        "}\n" ::"r"(d_tmem),
        "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}

// K-major, no-swizzle shared-memory operand descriptor (cute::UMMA::SmemDescriptor):
// start>>4 [0,14) | LBO>>4 [16,30) | SBO>>4 [32,46) | version=1 [46,48) | layout_type=0 [61,64)
__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((smem_addr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | (1ull << 46);
}

// 64-bit descriptor from its two words.  Only the start-address field (low 14 bits of the low word) changes between
// MMAs, so the issuing thread adds byte offsets >> 4 to the low word with 32-bit adds and never builds carries.
__device__ __forceinline__ uint64_t desc_from_words(uint32_t lo, uint32_t hi) {
    uint64_t d;
    asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "r"(lo), "r"(hi));
    return d;
}

// cute::UMMA::InstrDescriptor: c=F32 [4,6) | a=TF32 [7,10) | b=TF32 [10,13) | K-major A,B | N>>3 [17,23) | M>>4 [24,29)
__host__ __device__ constexpr uint32_t umma_idesc_tf32(int M, int N) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

#define WB_R32(v) \
    v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7], v[8], v[9], v[10], v[11], v[12], v[13], v[14], v[15], v[16], \
        v[17], v[18], v[19], v[20], v[21], v[22], v[23], v[24], v[25], v[26], v[27], v[28], v[29], v[30], v[31]

__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, "
        "%15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
        "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
        "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]),
        "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]),
        "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
        : "memory");
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, "
        "%15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}

// ---- query pre-split: fp32 queries -> (hi, lo) images in the UMMA no-swizzle K-major layout ----
// image[qb][chunk][half][k16 = 0..7][n = 0..BN-1][4 floats]: a core matrix (8 queries x 16 B) is 128
// contiguous bytes, SBO = 128 B between 8-query groups, LBO = BN*16 B between 16-byte k columns.
// FOLD: image[qb][chunk][k16][half][n][4] - one operand of 2*BN rows (hi rows, then lo rows), LBO = 2*BN*16 B.
template <int BN, bool FOLD = false>
__global__ void split_queries_kernel(const float* q, int nq, int ld, int nchunks, int nqb, float* img) {
    constexpr int kGemmBN = BN;
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;  // one float4 per thread
    const int64_t total = (int64_t)nqb * nchunks * 8 * kGemmBN;
    if (i >= total) return;
    const int n = (int)(i % kGemmBN);
    const int k16 = (int)((i / kGemmBN) % 8);
    const int chunk = (int)((i / (kGemmBN * 8)) % nchunks);
    const int qb = (int)(i / ((int64_t)kGemmBN * 8 * nchunks));
    const int qi = qb * kGemmBN + n;
    const int col = chunk * kGemmBK + k16 * 4;
    float v[4] = {0.f, 0.f, 0.f, 0.f};
    if (qi < nq) {
#pragma unroll
        for (int e = 0; e < 4; ++e)
            if (col + e < ld) v[e] = q[(size_t)qi * ld + col + e];
    }
    float hi[4], lo[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        hi[e] = __uint_as_float(__float_as_uint(v[e]) & 0xFFFFE000u);
        lo[e] = v[e] - hi[e];
    }
    const size_t base = ((size_t)(qb * nchunks + chunk) * 2) * (8 * kGemmBN * 4);
    const size_t off = FOLD ? ((size_t)k16 * 2 * kGemmBN + n) * 4 : ((size_t)k16 * kGemmBN + n) * 4;
    const size_t lo_off = FOLD ? (size_t)kGemmBN * 4 : (size_t)8 * kGemmBN * 4;
    *reinterpret_cast<float4*>(img + base + off) = make_float4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<float4*>(img + base + lo_off + off) = make_float4(lo[0], lo[1], lo[2], lo[3]);
}

__global__ void init_gemm_state_kernel(float* thr, int nq, int nq_pad, int* cnt, uint64_t* keys, int k, int kstride,
                                       int* overflow) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < nq_pad) thr[i] = i < nq ? -INFINITY : INFINITY;
    if (i < nq) cnt[i] = 0;
    if (i == 0) *overflow = 0;
    if (i < (int64_t)nq * k) keys[(i / k) * kstride + (i % k)] = 0ull;
}

// ---- the kernel -----------------------------------------------------------------------------------
// TERMS = 3: scores are the 3xTF32 sums (exact to ~1e-6).  TERMS = 1 ("filter" epochs of a search): only hi x hi is
// issued - a third of the tensor work, no lo halves in TMEM - and a row becomes a candidate when its one-term score
// exceeds thr - margin, margin >= |exact - one-term| (2^-9 |x||q| by Cauchy-Schwarz on the two truncations, plus
// accumulation slack); compact_topk_kernel then re-scores the candidates in fp32, so the result is the exact top-k.
template <int BN, bool ARGMAX, int TERMS = 3>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_topk_kernel(const __grid_constant__ CUtensorMap tmap, const GemmParams p) {
    static_assert(TERMS == 3 || (TERMS == 1 && !ARGMAX), "one-term scores are only a filter");
    // one-term epochs use the plain (non-folded) image: hi and lo are apart, only the hi half is copied
    constexpr bool FOLD = kGemmFold<BN, ARGMAX> && TERMS == 3;
    using Cfg = GemmCfg<BN, FOLD>;
    constexpr int kDCols = Cfg::kDCols;
    constexpr int kRaw = Cfg::kRawStages;
    constexpr int kSlots = Cfg::kSlots;
    constexpr int kBBytes = Cfg::kBBytes;
    constexpr int kTmemAOff = Cfg::kTmemAOff;
    extern __shared__ __align__(1024) unsigned char smem_gemm[];
    // [raw row tiles 16 KB x kRaw | query images kBBytes x kSlots | barriers | thresholds].  SWIZZLE_128B needs
    // 1024-byte aligned tiles: align by hand (the launch reserves 1 KB of slack).
    unsigned char* raw = smem_gemm + ((1024u - (smem_u32(smem_gemm) & 1023u)) & 1023u);
    unsigned char* bimg_s = raw + (size_t)kRaw * kGemmABytes;
    uint64_t* raw_full = reinterpret_cast<uint64_t*>(bimg_s + (size_t)kSlots * kBBytes);
    uint64_t* raw_empty = raw_full + kRaw;
    uint64_t* a_full = raw_empty + kRaw;  // slot operands ready: A in TMEM (4 warp arrivals) + image bytes (1 + tx)
    uint64_t* slot_empty = a_full + kSlots;
    uint64_t* d_full = slot_empty + kSlots;
    uint64_t* d_empty = d_full + 2;
    uint64_t* wq_full = d_empty + 2;          // work queue: item published by producer A
    uint64_t* wq_empty = wq_full + kGemmWQ;   // ... and retired by the 4 epilogue warps (the last role to touch it)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(wq_empty + kGemmWQ);
    float* thr_s = reinterpret_cast<float*>(tmem_slot + 2);  // [2][BN]
    long long* wq = reinterpret_cast<long long*>(thr_s + 2 * BN);  // [kGemmWQ] work ids (-1: no more work)

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t ntiles = (p.row_end - p.row_begin + kGemmBM - 1) / kGemmBM;
    const int64_t nwork = ntiles * p.nqb;
    const bool dyn = !ARGMAX && p.work_counter != nullptr;
    // Work items (row tile, query block) of this CTA.  Search mode interleaves (tile, block) pairs over the CTAs
    // (neighbouring CTAs share a row tile in L2); ARGMAX mode gives a CTA whole tiles and walks all query blocks
    // of a tile back to back, so the per-row running maximum lives in the epilogue threads' registers.
    const int64_t my_tiles = ntiles > (int64_t)blockIdx.x ? (ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const int64_t my_work =
        ARGMAX ? my_tiles * p.nqb : (nwork > (int64_t)blockIdx.x ? (nwork - blockIdx.x + gridDim.x - 1) / gridDim.x : 0);
    auto work_at = [&](int64_t it, int64_t& tile, int& qb) {
        if (ARGMAX) {
            const int64_t t = it / p.nqb;
            tile = blockIdx.x + t * gridDim.x;
            qb = (int)(it - t * p.nqb);
        } else {
            const int64_t w = blockIdx.x + it * (int64_t)gridDim.x;
            tile = w / p.nqb;
            qb = (int)(w - tile * p.nqb);
        }
    };
    // Per-role cursor over the work items.  Static mode: the role's own counter.  Dynamic mode: the queue producer A
    // fills; `last` is the queue slot of the item just taken (the epilogue retires it).
    struct WorkCursor {
        int slot = 0, last = 0;
        uint32_t ph = 0;
        int64_t it = 0;
    };
    auto next_item = [&](WorkCursor& c, int64_t& tile, int& qb) -> bool {
        if (!dyn) {
            if (c.it >= my_work) return false;
            work_at(c.it++, tile, qb);
            return true;
        }
        mbar_wait(&wq_full[c.slot], c.ph);
        const long long w = *reinterpret_cast<volatile long long*>(&wq[c.slot]);
        c.last = c.slot;
        if (++c.slot == kGemmWQ) { c.slot = 0; c.ph ^= 1u; }
        if (w < 0) return false;
        tile = w / p.nqb;
        qb = (int)(w - tile * p.nqb);
        return true;
    };

    if (tid == 0) {
        for (int s = 0; s < kRaw; ++s) {
            mbar_init(&raw_full[s], 1);
            mbar_init(&raw_empty[s], 4);  // 4 transform warps
        }
        for (int s = 0; s < kSlots; ++s) {
            mbar_init(&a_full[s], 5);      // 4 transform warps + producer B's arrive.expect_tx
            mbar_init(&slot_empty[s], 1);  // tcgen05.commit
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&d_full[b], 1);
            mbar_init(&d_empty[b], 4);  // 4 epilogue warps
        }
        for (int i = 0; i < kGemmWQ; ++i) {
            mbar_init(&wq_full[i], 1);
            mbar_init(&wq_empty[i], 4);
        }
        fence_mbar_init();
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "n"(kTmemCols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // =============================== producer A: raw row tiles (ring 1) =========================
        {   // the whole warp runs the control flow (converged); one elected lane issues
            int s = 0;
            uint32_t ph = 0;
            auto draw = [&]() -> int64_t {  // next item from the global dispenser
                unsigned int v = 0;
                if (lane == 0) v = atomicAdd(p.work_counter, 1u);
                return (int64_t)__shfl_sync(0xffffffffu, v, 0);
            };
            int wslot = 0;
            uint32_t wph = 0;
            int64_t w = dyn ? draw() : 0;
            for (int64_t it = 0; dyn || it < my_work; ++it) {
                int64_t tile;
                int qb;
                if (dyn) {  // publish the item (or the end marker) to the other roles
                    mbar_wait(&wq_empty[wslot], wph ^ 1u);
                    if (elect_one_sync()) {
                        wq[wslot] = w < nwork ? (long long)w : -1ll;
                        mbar_arrive(&wq_full[wslot]);
                    }
                    __syncwarp();
                    if (++wslot == kGemmWQ) { wslot = 0; wph ^= 1u; }
                    if (w >= nwork) break;
                    tile = w / p.nqb;
                    qb = (int)(w - tile * p.nqb);
                    w = draw();  // one item ahead: the atomic is in flight while this item's loads are issued
                } else {
                    work_at(it, tile, qb);
                }
                const int row0 = (int)(p.row_begin + tile * kGemmBM);
                for (int c = 0; c < p.nchunks; ++c) {
                    mbar_wait(&raw_empty[s], ph ^ 1u);
                    if (elect_one_sync()) {
                        mbar_arrive_expect_tx(&raw_full[s], kGemmABytes);
                        tma_load_2d(raw + (size_t)s * kGemmABytes, &tmap, c * kGemmBK, row0, &raw_full[s]);
                    }
                    __syncwarp();
                    if (++s == kRaw) { s = 0; ph ^= 1u; }
                }
            }
        }
    } else if (warp == 3) {
        // =============================== producer B: query images (ring 2) ==========================
        {
            int s = 0;
            uint32_t ph = 0;
            WorkCursor wc;
            int64_t tile;
            int qb;
            while (next_item(wc, tile, qb)) {
                const float* bsrc = p.bimg + (size_t)qb * p.nchunks * (kBBytes / 4);
                for (int c = 0; c < p.nchunks; ++c) {
                    mbar_wait(&slot_empty[s], ph ^ 1u);
                    if (elect_one_sync()) {
                        // (non-folded images keep hi and lo apart: one-term epochs copy the hi half only)
                        constexpr uint32_t kCopy = (TERMS == 1 && !FOLD) ? kBBytes / 2 : kBBytes;
                        mbar_arrive_expect_tx(&a_full[s], kCopy);
                        bulk_g2s(bimg_s + (size_t)s * kBBytes, bsrc + (size_t)c * (kBBytes / 4), kCopy, &a_full[s]);
                    }
                    __syncwarp();
                    if (++s == kSlots) { s = 0; ph ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        // =============================== MMA issuer =============================================
        {   // converged warp; the elected lane issues the MMAs and the commits that track them
            constexpr uint32_t idesc = umma_idesc_tf32(kGemmBM, BN);
            constexpr uint32_t idesc_fold = umma_idesc_tf32(kGemmBM, 2 * BN);
            constexpr int kLbo = (FOLD ? 2 * BN : BN) * 16;  // bytes between 16-byte k columns of the image
            const uint64_t desc0 = umma_smem_desc(smem_u32(bimg_s), kLbo, 128);  // stage 0, k-step 0
            const uint32_t desc_lo0 = (uint32_t)desc0, desc_w1 = (uint32_t)(desc0 >> 32);
            int s = 0;
            uint32_t ph = 0;
            int buf = 0;
            uint32_t dph = 0;
            WorkCursor wc;
            int64_t tile_;
            int qb_;
            while (next_item(wc, tile_, qb_)) {
                mbar_wait(&d_empty[buf], dph ^ 1u);  // epilogue has drained this accumulator
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(buf * kDCols);
                for (int c = 0; c < p.nchunks; ++c) {
                    mbar_wait(&a_full[s], ph);  // A hi/lo written to TMEM and the query image landed
                    tc_fence_after();
                    if (elect_one_sync()) {
                        // The issuing thread is a serial instruction stream (~4-5 cycles per dependent uniform
                        // instruction): every instruction here is on the kernel's critical path at small BN
                        // (measured: 455 of 735 cycles per chunk, profiles/r01/gemm_experiments.md).
                        const uint32_t a_hi = tmem_base + (uint32_t)(kTmemAOff + s * 64);
                        const uint32_t a_lo = a_hi + 32;
                        const uint32_t dh0 = desc_lo0 + (uint32_t)s * (uint32_t)(kBBytes >> 4);
#pragma unroll
                        for (int j = 0; j < ((WB_GEMM_EXP & 4) ? 0 : kGemmBK / 8); ++j) {
                            // one k-step = 8 tf32 = two 16-byte k columns: LBO = kLbo, SBO = 128 B
                            const uint64_t dh = desc_from_words(dh0 + (uint32_t)((j * 2 * kLbo) >> 4), desc_w1);
                            if constexpr (TERMS == 1) {
                                umma_tf32_ts(d_tmem, a_hi + j * 8, dh, idesc, (c | j) != 0);  // hi.hi only (hi rows of the image)
                            } else if constexpr (FOLD) {
                                umma_tf32_ts(d_tmem, a_hi + j * 8, dh, idesc_fold, (c | j) != 0);  // [hi.hi | hi.lo]
                                umma_tf32_ts(d_tmem, a_lo + j * 8, dh, idesc, 1);                  // lo.hi -> first half
                            } else {
                                const uint64_t dl =
                                    desc_from_words(dh0 + (uint32_t)((kBBytes / 2 + j * 2 * kLbo) >> 4), desc_w1);
                                umma_tf32_ts(d_tmem, a_hi + j * 8, dh, idesc, (c | j) != 0);
                                umma_tf32_ts(d_tmem, a_hi + j * 8, dl, idesc, 1);
                                umma_tf32_ts(d_tmem, a_lo + j * 8, dh, idesc, 1);
                            }
                        }
                        umma_commit(&slot_empty[s]);  // slot (smem image + TMEM A) is free once these MMAs retire
                        if (c == p.nchunks - 1) umma_commit(&d_full[buf]);
                    }
                    __syncwarp();
                    if (++s == kSlots) { s = 0; ph ^= 1u; }
                }
                if (++buf == 2) { buf = 0; dph ^= 1u; }
            }
        }
    } else if ((warp >= 4 && warp < 8) || warp >= 12) {
        // =============================== transform: fp32 -> (hi, lo) in TMEM ======================
        // Two sets of four warps take alternate k-chunks, so the LDS -> split -> tcgen05.st -> wait::st
        // latency chain of one chunk overlaps the next chunk's.
        const int set = warp >= 12 ? 1 : 0;
        const int quarter = warp & 3;
        const int r = quarter * 32 + lane;  // row of the tile == TMEM lane
        // ring positions of the running chunk (advanced for every chunk, whichever set handles it)
        int sr = 0, ss = 0, par = 0;
        uint32_t phr = 0, phs = 0;
        auto next_chunk = [&]() {
            if (++sr == kRaw) { sr = 0; phr ^= 1u; }
            if (++ss == kSlots) { ss = 0; phs ^= 1u; }
            par ^= 1;
        };
        WorkCursor wc;
        int64_t tile_;
        int qb_;
        while (next_item(wc, tile_, qb_)) {
            for (int c = 0; c < p.nchunks; ++c, next_chunk()) {
                if (par != set) continue;
                mbar_wait(&raw_full[sr], phr);
                const unsigned char* a_raw = raw + (size_t)sr * kGemmABytes + (size_t)r * 128;
                uint32_t hi[32], lo[32];
#pragma unroll
                for (int ch = 0; ch < 8; ++ch) {
                    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                    if constexpr (!(WB_GEMM_EXP & 1))
                        v = *reinterpret_cast<const float4*>(a_raw + ((ch ^ (r & 7)) << 4));  // SWIZZLE_128B
                    const float x[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const uint32_t h = __float_as_uint(x[e]) & 0xFFFFE000u;
                        hi[ch * 4 + e] = h;
                        if constexpr (TERMS != 1) lo[ch * 4 + e] = __float_as_uint(x[e] - __uint_as_float(h));
                    }
                }
                // NOTE: the raw stage is handed back only AFTER the TMEM store below.  Releasing it here
                // ("the tile is in registers") was measured to race on B200: the next TMA load overwrote the
                // top rows of the stage before they had been read (profiles/r01/gemm_experiments.md).
                mbar_wait(&slot_empty[ss], phs ^ 1u);        // the MMAs that last read this TMEM slot have retired
                tc_fence_after();
                const uint32_t ta = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(kTmemAOff + ss * 64);
                if constexpr (!(WB_GEMM_EXP & 2)) {
                    tmem_st32(ta, hi);
                    if constexpr (TERMS != 1) tmem_st32(ta + 32, lo);
                    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) {
                    mbar_arrive(&a_full[ss]);
                    mbar_arrive(&raw_empty[sr]);
                }
            }
        }
    } else if (warp >= 8 && warp < 12) {
        // =============================== epilogue: threshold filter ================================
        const int quarter = warp & 3;
        const int etid = tid - 8 * 32;
        int buf = 0;
        uint32_t dph = 0;
        float best = -INFINITY;  // ARGMAX: running maximum of this thread's row over the query blocks
        int best_i = 0;
        WorkCursor wc;
        int64_t tile;
        int qb;
        while (next_item(wc, tile, qb)) {
            const int64_t row = p.row_begin + tile * kGemmBM + quarter * 32 + lane;
            const bool row_ok = row < p.row_end && row_allowed(p.allow, (uint32_t)row);
            if constexpr (!ARGMAX) {
                if (etid < BN) {
                    float t = p.thr[qb * BN + etid];
                    if constexpr (TERMS == 1) t -= p.margin[qb * BN + etid];  // -inf / +inf (padding) stay put
                    thr_s[buf * BN + etid] = t;
                }
                named_bar_sync(kBarEpilogue, 128);
            } else if (qb == 0) {
                best = -INFINITY;
                best_i = 0;
            }
            mbar_wait(&d_full[buf], dph);
            tc_fence_after();
            const uint32_t td = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(buf * kDCols);
            constexpr int kEpi = BN < 32 ? BN : 32;  // query columns handled per TMEM load
#pragma unroll 1
            for (int cb = 0; cb < BN / kEpi; ++cb) {
                uint32_t v[32];
                tmem_ld32(td + cb * 32, v);  // BN = 16 (always folded): both 16-column halves in one load
                if constexpr (FOLD && BN >= 32 && TERMS == 3) {
                    uint32_t w[32];
                    tmem_ld32(td + BN + cb * 32, w);
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) + __uint_as_float(w[j]));
                } else {
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                    if constexpr (FOLD && TERMS == 3) {
#pragma unroll
                        for (int j = 0; j < 16; ++j)
                            v[j] = __float_as_uint(__uint_as_float(v[j]) + __uint_as_float(v[16 + j]));
                    }
                }
                if constexpr (ARGMAX) {
                    const int q0 = qb * BN + cb * 32;
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const float sc = __uint_as_float(v[j]);
                        // columns are visited in ascending index order: strict '>' keeps the lowest index on ties;
                        // padded columns (index >= nq) hold zeros and must not win
                        if (q0 + j < p.nq && sc > best) {
                            best = sc;
                            best_i = q0 + j;
                        }
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < kEpi; ++j) {
                        const float sc = __uint_as_float(v[j]);
                        const bool pass = !(WB_GEMM_EXP & 4) && row_ok && sc > thr_s[buf * BN + cb * kEpi + j];
                        const unsigned m = __ballot_sync(0xffffffffu, pass);
                        if (m) {
                            const int qi = qb * BN + cb * kEpi + j;  // < nq: padded queries have thr = +inf
                            int base = 0;
                            if (lane == (__ffs(m) - 1)) base = atomicAdd(&p.cnt[qi], __popc(m));
                            base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
                            if (pass) {
                                const int slot = base + __popc(m & ((1u << lane) - 1));
                                if (slot < p.cap) p.keys[(size_t)qi * p.kstride + p.k + slot] = make_key(sc, (uint32_t)row);
                                else *p.overflow = 1;
                            }
                        }
                    }
                }
            }
            if constexpr (ARGMAX) {
                if (qb == p.nqb - 1 && row_ok) {
                    p.assign_out[row] = best_i;
                    if (p.best_out) p.best_out[row] = best;
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(&d_empty[buf]);
                if (dyn) mbar_arrive(&wq_empty[wc.last]);  // the last role is done with this item: its queue slot is free
            }
            if constexpr (!ARGMAX) named_bar_sync(kBarEpilogue, 128);  // thr_s[buf] may be rewritten two tiles later
            if (++buf == 2) { buf = 0; dph ^= 1u; }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(kTmemCols) : "memory");
    }
}

// =====================================================================================================
// 2-CTA variant (cta_group::2): a cluster of two CTAs on one TPC computes a 256-row x 128-query tile.
// Each CTA keeps ITS 128 rows (raw ring, transform, A operand in its TMEM, accumulator in its TMEM, epilogue)
// and only HALF of the query image (64 queries) in shared memory; the leader CTA issues one
// tcgen05.mma.cta_group::2 (M = 256) per term and both SMs' tensor cores execute it, each fetching the
// other half of B from its peer.  That halves the per-SM shared-memory traffic of the query operand
// (B reads 64 -> 32 B/cycle, image writes 32 -> 16 KB per chunk), which is what capped the 1-CTA kernel
// at ~72 % tensor-pipe activity (profiles/r01/gemm_experiments.md).
// Cross-CTA protocol: the peer's transform / epilogue warps arrive on the LEADER's a_full / d_empty barriers
// (mapa + mbarrier.arrive.shared::cluster), the peer's warp 1 forwards "my half image landed" to the leader's
// bp_full, and the leader's tcgen05.commit multicasts slot_empty / d_full to both CTAs.
constexpr int kG2ASlots = 4;   // A operand ring in TMEM (64 columns per slot)
constexpr int kG2BSlots = 8;   // half-image ring in shared memory: deeper, it has to hide the cross-CTA forward
template <int BN>              // BN = queries per block of the PAIR (32 / 64 / 128); each CTA holds BN / 2 of them
struct Gemm2Cfg {
    static constexpr int kHalf = BN / 2;
    static constexpr int kBBytes = 2 * kHalf * kGemmBK * 4;  // hi + lo image of this CTA's queries (16 KB at BN = 128)
    static constexpr int kRaw = (224 * 1024 - kG2BSlots * kBBytes) / kGemmABytes > 12
                                    ? 12 : (224 * 1024 - kG2BSlots * kBBytes) / kGemmABytes;
    static constexpr int kNumBars = 2 * kRaw + 3 * kG2BSlots + 2 * kG2ASlots + 4;
    static constexpr size_t kSmemBytes =
        1024 + (size_t)kRaw * kGemmABytes + (size_t)kG2BSlots * kBBytes + kNumBars * 8 + 16 + 2 * BN * 4;
};

__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the barrier at the same shared-memory offset in CTA `cta` of the cluster
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t* bar, uint32_t cta) {
    uint32_t ra;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(smem_u32(bar)), "r"(cta));
    // default semantics (as CUTLASS' ClusterBarrier::arrive): an explicit .release.cluster costs an ERRBAR/MEMBAR per
    // arrive, and what these arrivals publish (TMEM contents, async-proxy copies) is ordered by tcgen05 fences / the
    // transaction barrier, not by generic-proxy release semantics
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(ra) : "memory");
}
// Waits on barriers that receive remote arrivals / multicast commits use the ordinary CTA-scope wait: polling with
// .acquire.cluster makes every try_wait iteration invalidate L1 (CCTL.IVALL; 37 % of all stall samples, measured).
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) { mbar_wait(bar, parity); }
__device__ __forceinline__ void umma_commit_2cta(uint64_t* bar) {
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
            smem_u32(bar)),
        "h"((uint16_t)3)
        : "memory");
}
__device__ __forceinline__ void umma_tf32_ts_2cta(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                                  uint32_t accumulate) {
    const uint32_t z = 0;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::2.kind::tf32 [%0], [%1], %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n"
        "}\n" ::"r"(d_tmem),
        "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(z)
        : "memory");
}

template <int BN, bool ARGMAX>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kGemmThreads, 1)
gemm2_topk_kernel(const __grid_constant__ CUtensorMap tmap, const GemmParams p) {
    using Cfg2 = Gemm2Cfg<BN>;
    constexpr int kG2Half = Cfg2::kHalf;
    constexpr int kRaw = Cfg2::kRaw;
    constexpr int kASlots = kG2ASlots;
    constexpr int kBSlots = kG2BSlots;
    constexpr int kBBytes = Cfg2::kBBytes;
    constexpr int kTmemAOff = 2 * BN;
    extern __shared__ __align__(1024) unsigned char smem_gemm2[];
    unsigned char* raw = smem_gemm2 + ((1024u - (smem_u32(smem_gemm2) & 1023u)) & 1023u);
    unsigned char* bimg_s = raw + (size_t)kRaw * kGemmABytes;
    uint64_t* raw_full = reinterpret_cast<uint64_t*>(bimg_s + (size_t)kBSlots * kBBytes);
    uint64_t* raw_empty = raw_full + kRaw;
    uint64_t* b_full = raw_empty + kRaw;      // my half image landed (local)
    uint64_t* bp_full = b_full + kBSlots;     // leader only: the peer's half image landed
    uint64_t* b_empty = bp_full + kBSlots;    // both: the MMAs that read this image slot have retired (multicast commit)
    uint64_t* a_full = b_empty + kBSlots;     // leader only: A of BOTH CTAs is in TMEM (8 arrivals)
    uint64_t* a_empty = a_full + kASlots;     // both: the MMAs that read this TMEM slot have retired (multicast commit)
    uint64_t* d_full = a_empty + kASlots;     // both: accumulator ready (multicast commit)
    uint64_t* d_empty = d_full + 2;           // leader only: both epilogues drained the accumulator (8 arrivals)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(d_empty + 2);
    float* thr_s = reinterpret_cast<float*>(tmem_slot + 2);  // [2][BN]

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t crank = cluster_ctarank();
    const bool leader = crank == 0;
    const int64_t pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
    const int64_t ntiles = (p.row_end - p.row_begin + kGemmBM - 1) / kGemmBM;
    const int64_t ntp = (ntiles + 1) / 2;  // tile pairs
    const int64_t nwork = ntp * p.nqb;
    const int64_t my_tp = ntp > pair ? (ntp - pair + npairs - 1) / npairs : 0;
    const int64_t my_work = ARGMAX ? my_tp * p.nqb : (nwork > pair ? (nwork - pair + npairs - 1) / npairs : 0);
    auto work_at = [&](int64_t it, int64_t& tile, int& qb) {  // tile = THIS CTA's row tile
        int64_t tp;
        if (ARGMAX) {
            const int64_t t = it / p.nqb;
            tp = pair + t * npairs;
            qb = (int)(it - t * p.nqb);
        } else {
            const int64_t w = pair + it * npairs;
            tp = w / p.nqb;
            qb = (int)(w - tp * p.nqb);
        }
        tile = 2 * tp + crank;
    };

    if (tid == 0) {
        for (int s = 0; s < kRaw; ++s) {
            mbar_init(&raw_full[s], 1);
            mbar_init(&raw_empty[s], 4);
        }
        for (int s = 0; s < kBSlots; ++s) {
            mbar_init(&b_full[s], 1);
            mbar_init(&bp_full[s], 1);
            mbar_init(&b_empty[s], 1);
        }
        for (int s = 0; s < kASlots; ++s) {
            mbar_init(&a_full[s], 8);
            mbar_init(&a_empty[s], 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&d_full[b], 1);
            mbar_init(&d_empty[b], 8);
        }
        fence_mbar_init();
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                     "n"(kTmemCols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();  // both CTAs' barriers are initialised before any remote arrive
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // =============================== producer A: this CTA's raw row tiles =======================
        int s = 0;
        uint32_t ph = 0;
        for (int64_t it = 0; it < my_work; ++it) {
            int64_t tile;
            int qb;
            work_at(it, tile, qb);
            const int row0 = (int)(p.row_begin + tile * kGemmBM);  // may be past row_end: TMA zero-fills
            for (int c = 0; c < p.nchunks; ++c) {
                mbar_wait(&raw_empty[s], ph ^ 1u);
                if (elect_one_sync()) {
                    mbar_arrive_expect_tx(&raw_full[s], kGemmABytes);
                    tma_load_2d(raw + (size_t)s * kGemmABytes, &tmap, c * kGemmBK, row0, &raw_full[s]);
                }
                __syncwarp();
                if (++s == kRaw) { s = 0; ph ^= 1u; }
            }
        }
    } else if (warp == 3) {
        // =============================== producer B: this CTA's half of the query image =============
        int s = 0;
        uint32_t ph = 0;
        for (int64_t it = 0; it < my_work; ++it) {
            int64_t tile;
            int qb;
            work_at(it, tile, qb);
            const float* bsrc = p.bimg + (size_t)(2 * qb + (int)crank) * p.nchunks * (kBBytes / 4);  // images of BN/2 queries
            for (int c = 0; c < p.nchunks; ++c) {
                mbar_wait_cluster(&b_empty[s], ph ^ 1u);
                if (elect_one_sync()) {
                    mbar_arrive_expect_tx(&b_full[s], kBBytes);
                    bulk_g2s(bimg_s + (size_t)s * kBBytes, bsrc + (size_t)c * (kBBytes / 4), kBBytes, &b_full[s]);
                }
                __syncwarp();
                if (++s == kBSlots) { s = 0; ph ^= 1u; }
            }
        }
    } else if (warp == 1 && !leader) {
        // =============================== peer: tell the leader when my half image has landed =========
        int s = 0;
        uint32_t ph = 0;
        for (int64_t it = 0; it < my_work; ++it) {
            for (int c = 0; c < p.nchunks; ++c) {
                mbar_wait(&b_full[s], ph);
                if (elect_one_sync()) mbar_arrive_cluster(&bp_full[s], 0);
                __syncwarp();
                if (++s == kBSlots) { s = 0; ph ^= 1u; }
            }
        }
    } else if (warp == 1) {
        // =============================== leader: MMA issuer for the pair ===============================
        constexpr uint32_t idesc = umma_idesc_tf32(2 * kGemmBM, BN);
        const uint64_t desc_hi0 = umma_smem_desc(smem_u32(bimg_s), kG2Half * 16, 128);  // my half: LBO = (BN/2) * 16 B
        int s = 0, sa = 0;
        uint32_t ph = 0, pha = 0;
        int buf = 0;
        uint32_t dph = 0;
        for (int64_t it = 0; it < my_work; ++it) {
            mbar_wait_cluster(&d_empty[buf], dph ^ 1u);  // both epilogues have drained this accumulator
            tc_fence_after();
            const uint32_t d_tmem = tmem_base + (uint32_t)(buf * BN);
            for (int c = 0; c < p.nchunks; ++c) {
                mbar_wait(&b_full[s], ph);
                mbar_wait_cluster(&bp_full[s], ph);
                mbar_wait_cluster(&a_full[sa], pha);
                tc_fence_after();
                if (elect_one_sync()) {
                    const uint32_t a_hi = tmem_base + (uint32_t)(kTmemAOff + sa * 64);
                    const uint32_t a_lo = a_hi + 32;
                    const uint64_t dh0 = desc_hi0 + (uint64_t)(((uint32_t)s * kBBytes) >> 4);
                    const uint64_t dl0 = dh0 + (uint64_t)((kBBytes / 2) >> 4);
#pragma unroll
                    for (int j = 0; j < kGemmBK / 8; ++j) {
                        const uint64_t dh = dh0 + (uint64_t)((j * 2 * kG2Half * 16) >> 4);
                        const uint64_t dl = dl0 + (uint64_t)((j * 2 * kG2Half * 16) >> 4);
                        umma_tf32_ts_2cta(d_tmem, a_hi + j * 8, dh, idesc, (c | j) != 0);
                        umma_tf32_ts_2cta(d_tmem, a_hi + j * 8, dl, idesc, 1);
                        umma_tf32_ts_2cta(d_tmem, a_lo + j * 8, dh, idesc, 1);
                    }
                    umma_commit_2cta(&b_empty[s]);
                    umma_commit_2cta(&a_empty[sa]);
                    if (c == p.nchunks - 1) umma_commit_2cta(&d_full[buf]);
                }
                __syncwarp();
                if (++s == kBSlots) { s = 0; ph ^= 1u; }
                if (++sa == kASlots) { sa = 0; pha ^= 1u; }
            }
            if (++buf == 2) { buf = 0; dph ^= 1u; }
        }
    } else if ((warp >= 4 && warp < 8) || warp >= 12) {
        // =============================== transform: fp32 -> (hi, lo) in this CTA's TMEM ================
        const int set = warp >= 12 ? 1 : 0;
        const int quarter = warp & 3;
        const int r = quarter * 32 + lane;
        int64_t g = 0;
        for (int64_t it = 0; it < my_work; ++it) {
            for (int c = 0; c < p.nchunks; ++c, ++g) {
                if ((g & 1) != set) continue;
                const int sr = (int)(g % kRaw);
                const uint32_t phr = (uint32_t)((g / kRaw) & 1);
                const int ss = (int)(g % kASlots);
                const uint32_t phs = (uint32_t)((g / kASlots) & 1);
                mbar_wait(&raw_full[sr], phr);
                const unsigned char* a_raw = raw + (size_t)sr * kGemmABytes + (size_t)r * 128;
                uint32_t hi[32], lo[32];
#pragma unroll
                for (int ch = 0; ch < 8; ++ch) {
                    const float4 v = *reinterpret_cast<const float4*>(a_raw + ((ch ^ (r & 7)) << 4));
                    const float x[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const uint32_t h = __float_as_uint(x[e]) & 0xFFFFE000u;
                        hi[ch * 4 + e] = h;
                        lo[ch * 4 + e] = __float_as_uint(x[e] - __uint_as_float(h));
                    }
                }
                mbar_wait_cluster(&a_empty[ss], phs ^ 1u);
                tc_fence_after();
                const uint32_t ta = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(kTmemAOff + ss * 64);
                tmem_st32(ta, hi);
                tmem_st32(ta + 32, lo);
                asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                tc_fence_before();
                __syncwarp();
                if (lane == 0) {
                    mbar_arrive_cluster(&a_full[ss], 0);  // the leader counts 4 warps of each CTA
                    mbar_arrive(&raw_empty[sr]);
                }
            }
        }
    } else if (warp >= 8 && warp < 12) {
        // =============================== epilogue (this CTA's 128 rows) =================================
        const int quarter = warp & 3;
        const int etid = tid - 8 * 32;
        int buf = 0;
        uint32_t dph = 0;
        float best = -INFINITY;
        int best_i = 0;
        for (int64_t it = 0; it < my_work; ++it) {
            int64_t tile;
            int qb;
            work_at(it, tile, qb);
            const int64_t row = p.row_begin + tile * kGemmBM + quarter * 32 + lane;
            const bool row_ok = row < p.row_end && row_allowed(p.allow, (uint32_t)row);
            if constexpr (!ARGMAX) {
                if (etid < BN) thr_s[buf * BN + etid] = p.thr[qb * BN + etid];
                named_bar_sync(kBarEpilogue, 128);
            } else if (qb == 0) {
                best = -INFINITY;
                best_i = 0;
            }
            mbar_wait_cluster(&d_full[buf], dph);
            tc_fence_after();
            const uint32_t td = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(buf * BN);
#pragma unroll 1
            for (int cb = 0; cb < BN / 32; ++cb) {
                uint32_t v[32];
                tmem_ld32(td + cb * 32, v);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if constexpr (ARGMAX) {
                    const int q0 = qb * BN + cb * 32;
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const float sc = __uint_as_float(v[j]);
                        if (q0 + j < p.nq && sc > best) {
                            best = sc;
                            best_i = q0 + j;
                        }
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const float sc = __uint_as_float(v[j]);
                        const bool pass = row_ok && sc > thr_s[buf * BN + cb * 32 + j];
                        const unsigned m = __ballot_sync(0xffffffffu, pass);
                        if (m) {
                            const int qi = qb * BN + cb * 32 + j;
                            int base = 0;
                            if (lane == (__ffs(m) - 1)) base = atomicAdd(&p.cnt[qi], __popc(m));
                            base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
                            if (pass) {
                                const int slot = base + __popc(m & ((1u << lane) - 1));
                                if (slot < p.cap) p.keys[(size_t)qi * p.kstride + p.k + slot] = make_key(sc, (uint32_t)row);
                                else *p.overflow = 1;
                            }
                        }
                    }
                }
            }
            if constexpr (ARGMAX) {
                if (qb == p.nqb - 1 && row_ok) {
                    p.assign_out[row] = best_i;
                    if (p.best_out) p.best_out[row] = best;
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(&d_empty[buf], 0);
            if constexpr (!ARGMAX) named_bar_sync(kBarEpilogue, 128);
            if (++buf == 2) { buf = 0; dph ^= 1u; }
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();  // the peer's shared memory and TMEM stay alive until the leader's last MMA has retired
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(kTmemCols) : "memory");
    }
}

}  // namespace wb
