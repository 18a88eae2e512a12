// gemm_ss.cuh - K2 "filter" epochs for large batches: 256-query blocks on a CTA pair, BOTH operands read by the
// tensor core straight from shared memory (tcgen05.mma.cta_group::2.kind::tf32, SS form, M = 256, N = 256).
//
// Same contract as the one-term gemm_topk_kernel<BN, false, TERMS = 1> (gemm.cuh): one-term TF32 scores are only a filter, a row
// becomes a candidate when its score exceeds thr - margin and rescore_candidates_kernel / compact_topk_kernel
// (merge.cuh) re-score the candidates exactly in fp32, so the result is the exact top-k.  Replaces faiss
// exhaustive_inner_product_blas [faiss-upstream] reached from /root/reference/src/index/feature_search_index.py:113.
//
// Why a second kernel (round 2; profiles/r02/gemm_ss.md): kind::tf32 reads fp32 words and uses their top 19 bits,
// so the one-term operand needs NO transform at all:
//   * the raw fp32 row tile lands by 2-D TMA (SWIZZLE_128B) and IS the A operand (K-major SW128 descriptor);
//   * N = 256 queries per instruction: 16 KB rows + 16 KB image per chunk for 1 M MACs per SM - 1.5x fewer L2 bytes per
//     MAC than 128-query blocks, and half as many passes over the rows;
//   * no transform warps, no tcgen05.st, no A slots in tensor memory: TMEM holds two 256-column accumulators, so the
//     epilogue of one tile still overlaps the MMAs of the next.
// Measured on B200 (10M x 768, batch 1024): 47.7 -> 27.7 ms per search, bit-identical results; ncu: tensor pipe
// 97 % active at the power-capped clock (1.27 GHz), L2 -> SM 11.7 TB/s, DRAM 2.2 TB/s.
// Roles (12 warps): warp 0 producer (TMA rows + bulk copy of this CTA's half image, one barrier per stage),
// warp 1 MMA issuer (leader) / "my stage landed" forwarder (peer), warp 2 TMEM allocator, warps 4-11 epilogue
// (TMEM lane quarter = warp & 3, column half = (warp - 4) >> 2).
#pragma once
#include "gemm.cuh"

namespace wb {

// NH = queries per CTA (the pair's block is 2 * NH): 128 for batches above 128 queries and for the k-means assignment,
// 64 for a single block of 65..128 queries (one pass over the rows, HBM-bound: the TS kernel's transform + TMEM stores
// on top of N = 128 MMAs made that block tensor/TMEM-bound at the power-capped clock).
template <int NH>
struct F2Cfg {
    static constexpr int kBN = 2 * NH;
    static constexpr int kBBytes = NH * kGemmBK * 4;  // NH queries x 32 floats, no-swizzle core-matrix layout
    static constexpr int kStageBytes = kGemmABytes + kBBytes;
    static constexpr int kStages = NH >= 128 ? 6 : 8;
    static constexpr int kNumBars = 3 * kStages + 4;
    static constexpr size_t kSmemBytes = 1024 + (size_t)kStages * kStageBytes + kNumBars * 8 + 16 + 2 * kBN * 4;
    static_assert(kSmemBytes <= 232448, "shared memory budget");
    static_assert(2 * kBN <= kTmemCols, "two accumulators in tensor memory");
};
constexpr int kF2Half = 128;
constexpr int kF2BN = 2 * kF2Half;
constexpr int kF2BBytes = F2Cfg<128>::kBBytes;
constexpr int kF2StageBytes = F2Cfg<128>::kStageBytes;
constexpr int kF2Threads = 384;
constexpr int kF2EpiThreads = 256;
constexpr size_t kF2SmemBytes = F2Cfg<128>::kSmemBytes;

// Query image of the SS kernel: image[qb][half][chunk][k16 = 0..7][n = 0..NH-1][4 floats] - raw fp32 (the tensor core
// uses the tf32 part), K-major core matrices: 8 queries x 16 B are 128 contiguous bytes, SBO = 128 B between
// 8-query groups, LBO = NH * 16 B between 16-byte k columns.
template <int NH = 128>
__global__ void image_queries_f2_kernel(const float* q, int nq, int ld, int nchunks, int nqb, float* img) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;  // one float4 per thread
    const int64_t total = (int64_t)nqb * 2 * nchunks * 8 * NH;
    if (i >= total) return;
    const int n = (int)(i % NH);
    const int k16 = (int)((i / NH) % 8);
    const int chunk = (int)((i / (NH * 8)) % nchunks);
    const int half = (int)((i / ((int64_t)NH * 8 * nchunks)) % 2);
    const int qb = (int)(i / ((int64_t)NH * 8 * nchunks * 2));
    const int qi = qb * 2 * NH + half * NH + n;
    const int col = chunk * kGemmBK + k16 * 4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (qi < nq) {
        const float* src = q + (size_t)qi * ld + col;
        if (col + 3 < ld) v = *reinterpret_cast<const float4*>(src);  // ld is a multiple of 4
    }
    reinterpret_cast<float4*>(img)[i] = v;
}

__device__ __forceinline__ void umma_tf32_ss_2cta(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                                  uint32_t accumulate) {
    const uint32_t z = 0;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n"
        "}\n" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(z)
        : "memory");
}

// K-major SWIZZLE_128B operand (what a 2-D TMA load with CU_TENSOR_MAP_SWIZZLE_128B of 32-float rows produces):
// 8-row groups are 1024 B apart (SBO), LBO is unused (1), layout type 2, descriptor version 1.
__device__ __forceinline__ uint64_t umma_smem_desc_sw128(uint32_t smem_addr) {
    return (uint64_t)((smem_addr >> 4) & 0x3FFF) | (1ull << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) |
           (2ull << 61);
}

// ARGMAX (k-means TRAINING assignment, K6): rows = points, "queries" = centroids in 256-wide blocks; a pair walks
// all centroid blocks of its row tiles back to back and every row keeps a running (max, lowest index) in the
// epilogue registers - plain TF32 scores (SURVEY.md 8d allows it for training: "argmax only"), so two centroids
// whose scores differ by less than ~2e-3 |x||c| may swap.  Add-time assignment stays on the exact 3xTF32 kernel.
template <int NH = 128, bool ARGMAX = false, bool TIMING_ONLY = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kF2Threads, 1)
filter2_topk_kernel(const __grid_constant__ CUtensorMap tmap, const GemmParams p) {
    using Cfg = F2Cfg<NH>;
    constexpr int kStages = Cfg::kStages;
    constexpr int kStageBytes = Cfg::kStageBytes;
    constexpr int kBBytes = Cfg::kBBytes;
    constexpr int kBN = Cfg::kBN;
    extern __shared__ __align__(1024) unsigned char smem_f2[];
    unsigned char* stages = smem_f2 + ((1024u - (smem_u32(smem_f2) & 1023u)) & 1023u);  // same offset in both CTAs
    uint64_t* full = reinterpret_cast<uint64_t*>(stages + (size_t)kStages * kStageBytes);  // my rows + my half image landed
    uint64_t* peer_full = full + kStages;   // leader only: the peer's stage landed
    uint64_t* empty = peer_full + kStages;  // both: the MMAs that read this stage have retired (multicast commit)
    uint64_t* d_full = empty + kStages;     // both: accumulator ready (multicast commit)
    uint64_t* d_empty = d_full + 2;           // leader only: both epilogues drained the accumulator (16 warp arrivals)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(d_empty + 2);
    float* thr_s = reinterpret_cast<float*>(tmem_slot + 4);  // [2][2 * NH], 16-byte aligned

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t crank = cluster_ctarank();
    const bool leader = crank == 0;
    const int64_t pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
    const int64_t ntiles = (p.row_end - p.row_begin + kGemmBM - 1) / kGemmBM;
    const int64_t ntp = (ntiles + 1) / 2;  // tile pairs
    const int64_t nwork = ntp * p.nqb;
    const int64_t my_tp = ntp > pair ? (ntp - pair + npairs - 1) / npairs : 0;
    // A pair owns whole tile pairs and walks all query blocks of one before it moves on: the row tile is fetched from
    // DRAM once and re-read from L2 by the SAME pair a few microseconds later.  (Interleaving the blocks of a tile over
    // neighbouring pairs relied on those pairs staying in step; they drift, and ncu showed 1.9x the algorithmic DRAM
    // bytes.)  Small epochs keep the interleave, which balances better when there are few tile pairs per CTA pair.
    // ARGMAX needs the tile-major order anyway: the running maximum lives in the epilogue's registers.
    const bool tile_major = ARGMAX || ntp >= 8 * npairs;
    const int64_t my_work = tile_major ? my_tp * p.nqb : (nwork > pair ? (nwork - pair + npairs - 1) / npairs : 0);
    auto work_at = [&](int64_t it, int64_t& tile, int& qb) {  // tile = THIS CTA's row tile
        int64_t tp;
        if (tile_major) {
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
        for (int s = 0; s < kStages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&peer_full[s], 1);
            mbar_init(&empty[s], 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&d_full[b], 1);
            mbar_init(&d_empty[b], 16);
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
        // =============================== producer: rows (2-D TMA) + this CTA's half image ============
        int s = 0;
        uint32_t ph = 0;
        for (int64_t it = 0; it < my_work; ++it) {
            int64_t tile;
            int qb;
            work_at(it, tile, qb);
            const int row0 = (int)(p.row_begin + tile * kGemmBM);  // may be past row_end: TMA zero-fills
            const float* bsrc = p.bimg + (size_t)(2 * qb + (int)crank) * p.nchunks * (kBBytes / 4);
            for (int c = 0; c < p.nchunks; ++c) {
                mbar_wait(&empty[s], ph ^ 1u);
                if (elect_one_sync()) {
                    unsigned char* st = stages + (size_t)s * kStageBytes;
                    mbar_arrive_expect_tx(&full[s], kStageBytes);
                    tma_load_2d(st, &tmap, c * kGemmBK, row0, &full[s]);
                    bulk_g2s(st + kGemmABytes, bsrc + (size_t)c * (kBBytes / 4), kBBytes, &full[s]);
                }
                __syncwarp();
                if (++s == kStages) { s = 0; ph ^= 1u; }
            }
        }
    } else if (warp == 1 && !leader) {
        // =============================== peer: tell the leader when my stage has landed ==============
        int s = 0;
        uint32_t ph = 0;
        for (int64_t it = 0; it < my_work; ++it) {
            for (int c = 0; c < p.nchunks; ++c) {
                mbar_wait(&full[s], ph);
                if (elect_one_sync()) mbar_arrive_cluster(&peer_full[s], 0);
                __syncwarp();
                if (++s == kStages) { s = 0; ph ^= 1u; }
            }
        }
    } else if (warp == 1) {
        // =============================== leader: MMA issuer for the pair =============================
        constexpr uint32_t idesc = umma_idesc_tf32(2 * kGemmBM, kBN);
        const uint64_t adesc0 = umma_smem_desc_sw128(smem_u32(stages));
        const uint64_t bdesc0 = umma_smem_desc(smem_u32(stages + kGemmABytes), NH * 16, 128);
        const uint32_t a_lo0 = (uint32_t)adesc0, a_hi = (uint32_t)(adesc0 >> 32);
        const uint32_t b_lo0 = (uint32_t)bdesc0, b_hi = (uint32_t)(bdesc0 >> 32);
        int s = 0;
        uint32_t ph = 0;
        int buf = 0;
        uint32_t dph = 0;
        for (int64_t it = 0; it < my_work; ++it) {
            mbar_wait(&d_empty[buf], dph ^ 1u);  // both epilogues have drained this accumulator
            tc_fence_after();
            const uint32_t d_tmem = tmem_base + (uint32_t)(buf * kBN);
            for (int c = 0; c < p.nchunks; ++c) {
                mbar_wait(&full[s], ph);
                mbar_wait(&peer_full[s], ph);
                tc_fence_after();
                if (elect_one_sync()) {
                    const uint32_t so = (uint32_t)s * (uint32_t)(kStageBytes >> 4);
#pragma unroll
                    for (int j = 0; j < kGemmBK / 8; ++j) {
                        // one k-step = 8 tf32 = 32 B: inside the 128-byte swizzle atom for A, two 16-byte k columns for B
                        const uint64_t da = desc_from_words(a_lo0 + so + (uint32_t)(j * 2), a_hi);
                        const uint64_t db = desc_from_words(b_lo0 + so + (uint32_t)((j * 2 * NH * 16) >> 4), b_hi);
                        umma_tf32_ss_2cta(d_tmem, da, db, idesc, (c | j) != 0);
                    }
                    umma_commit_2cta(&empty[s]);
                    if (c == p.nchunks - 1) umma_commit_2cta(&d_full[buf]);
                }
                __syncwarp();
                if (++s == kStages) { s = 0; ph ^= 1u; }
            }
            if (++buf == 2) { buf = 0; dph ^= 1u; }
        }
    } else if (warp >= 4) {
        // =============================== epilogue (this CTA's 128 rows x 256 queries) ================
        const int quarter = warp & 3;
        const int chalf = (warp - 4) >> 2;  // which half (NH) of the block's 2 * NH query columns
        const int etid = tid - 4 * 32;      // 0..255
        int buf = 0;
        uint32_t dph = 0;
        float best = -INFINITY;  // ARGMAX: running maximum of this thread's row over its half of every centroid block
        int best_i = 0;
        for (int64_t it = 0; it < my_work; ++it) {
            int64_t tile;
            int qb;
            work_at(it, tile, qb);
            const int64_t row = p.row_begin + tile * kGemmBM + quarter * 32 + lane;
            const bool row_ok = row < p.row_end && row_allowed(p.allow, (uint32_t)row);
            if constexpr (!ARGMAX) {
                if (etid < kBN) thr_s[buf * kBN + etid] = p.thr[qb * kBN + etid] - p.margin[qb * kBN + etid];  // +inf for padding
                named_bar_sync(kBarEpilogue, kF2EpiThreads);
            } else if (qb == 0) {
                best = -INFINITY;
                best_i = 0;
            }
            mbar_wait(&d_full[buf], dph);
            tc_fence_after();
            const uint32_t td = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(buf * kBN + chalf * NH);
            const float* thr_w = thr_s + buf * kBN + chalf * NH;
#pragma unroll 1
            for (int cb = 0; cb < NH / 32; ++cb) {
                uint32_t v[32];
                tmem_ld32(td + cb * 32, v);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                if constexpr (TIMING_ONLY) continue;
                if constexpr (ARGMAX) {
                    const int c0 = qb * kBN + chalf * NH + cb * 32;
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const float sc = __uint_as_float(v[j]);
                        // ascending index order + strict '>' keeps the lowest index on ties; padded columns
                        // (index >= nq) hold zeros and must not win
                        if (c0 + j < p.nq && sc > best) {
                            best = sc;
                            best_i = c0 + j;
                        }
                    }
                    continue;
                }
                // almost nothing passes: one vote per 32 columns, the per-column path only when something did
                bool any = false;
#pragma unroll
                for (int j4 = 0; j4 < 8; ++j4) {
                    const float4 t = *reinterpret_cast<const float4*>(thr_w + cb * 32 + j4 * 4);
                    any |= __uint_as_float(v[j4 * 4 + 0]) > t.x;
                    any |= __uint_as_float(v[j4 * 4 + 1]) > t.y;
                    any |= __uint_as_float(v[j4 * 4 + 2]) > t.z;
                    any |= __uint_as_float(v[j4 * 4 + 3]) > t.w;
                }
                if (!__any_sync(0xffffffffu, any && row_ok)) continue;
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const float sc = __uint_as_float(v[j]);
                    const bool pass = row_ok && sc > thr_w[cb * 32 + j];
                    const unsigned m = __ballot_sync(0xffffffffu, pass);
                    if (m) {
                        const int qi = qb * kBN + chalf * NH + cb * 32 + j;  // < nq: padded queries have thr = +inf
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
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(&d_empty[buf], 0);
            if constexpr (!ARGMAX) {
                named_bar_sync(kBarEpilogue, kF2EpiThreads);  // thr_s[buf] may be rewritten two tiles later
            } else if (qb == p.nqb - 1) {
                // the two warps of a row quarter hold the maxima of the two column halves: combine through thr_s
                float* cb_s = thr_s;                                   // [128] best score of the upper half
                int* ci_s = reinterpret_cast<int*>(thr_s + kGemmBM);   // [128] its index
                if (chalf == 1) {
                    cb_s[quarter * 32 + lane] = best;
                    ci_s[quarter * 32 + lane] = best_i;
                }
                named_bar_sync(kBarEpilogue, kF2EpiThreads);
                if (chalf == 0 && row_ok) {
                    const float b1 = cb_s[quarter * 32 + lane];
                    const int i1 = ci_s[quarter * 32 + lane];
                    if (b1 > best || (b1 == best && i1 < best_i)) {
                        best = b1;
                        best_i = i1;
                    }
                    p.assign_out[row] = best_i;
                    if (p.best_out) p.best_out[row] = best;
                }
                named_bar_sync(kBarEpilogue, kF2EpiThreads);  // cb_s / ci_s are rewritten at the next tile
            }
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

// ---- TF32 tensor-pipe peak, measured with this library's own instruction shape ------------------------------------
// Every CTA pair issues `iters` x 4 back-to-back tcgen05.mma.cta_group::2.kind::tf32 (M = 256, N = 256, K = 8, both
// operands from shared memory) into two alternating
// accumulators and waits for the last commit.  No loads, no epilogue: this is the ceiling filter2_topk_kernel's
// MMA stream could reach, and the denominator bench.py reports batch-1024 throughput against.
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(128, 1) tf32_peak_kernel(int iters, int constant_operands) {
    extern __shared__ __align__(1024) unsigned char smem_pk[];
    unsigned char* st = smem_pk + ((1024u - (smem_u32(smem_pk) & 1023u)) & 1023u);
    __shared__ uint64_t done_bar;
    __shared__ uint32_t tmem_slot_pk;
    const int tid = threadIdx.x, warp = tid >> 5;
    const bool leader = cluster_ctarank() == 0;
    // pseudo-random operands in (-1, 1): the power a tensor pipe draws depends on how many operand bits toggle, and
    // under the 1 kW cap power sets the clock - constant operands sustained 1116 TFLOP/s at 1.84 GHz on the same GPU
    // that holds ~1.2-1.3 GHz on real data (profiles/r02/tf32_peak.md)
    for (int i = tid; i < kF2StageBytes / 4; i += blockDim.x) {
        uint32_t h = (uint32_t)i * 2654435761u + blockIdx.x * 40503u;
        h ^= h >> 15; h *= 2246822519u; h ^= h >> 13; h *= 3266489917u; h ^= h >> 16;
        reinterpret_cast<float*>(st)[i] = constant_operands ? 1.0f : (float)(int32_t)h * (1.0f / 2147483648.0f);
    }
    if (tid == 0) {
        mbar_init(&done_bar, 1);
        fence_mbar_init();
    }
    fence_proxy_async();
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot_pk)),
                     "n"(kTmemCols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = tmem_slot_pk;
    if (warp == 1 && leader) {
        constexpr uint32_t idesc = umma_idesc_tf32(2 * kGemmBM, kF2BN);
        const uint64_t adesc0 = umma_smem_desc_sw128(smem_u32(st));
        const uint64_t bdesc0 = umma_smem_desc(smem_u32(st + kGemmABytes), kF2Half * 16, 128);
        const uint32_t a_lo0 = (uint32_t)adesc0, a_hi = (uint32_t)(adesc0 >> 32);
        const uint32_t b_lo0 = (uint32_t)bdesc0, b_hi = (uint32_t)(bdesc0 >> 32);
        for (int it = 0; it < iters; ++it) {
            if (elect_one_sync()) {
                const uint32_t d_tmem = tmem_base + (uint32_t)((it & 1) * kF2BN);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const uint64_t da = desc_from_words(a_lo0 + (uint32_t)(j * 2), a_hi);
                    const uint64_t db = desc_from_words(b_lo0 + (uint32_t)((j * 2 * kF2Half * 16) >> 4), b_hi);
                    umma_tf32_ss_2cta(d_tmem, da, db, idesc, j != 0);
                }
                if (it == iters - 1) umma_commit_2cta(&done_bar);
            }
            __syncwarp();
        }
    }
    if (warp == 1) {
        mbar_wait(&done_bar, 0);  // the commit is multicast to both CTAs
        tc_fence_after();
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 2) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(kTmemCols) : "memory");
    }
}

}  // namespace wb
