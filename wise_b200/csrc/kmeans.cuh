// kmeans.cuh - K7 kmeans_update: deterministic per-list sums, mean, optional spherical renormalisation.
// Replaces faiss Clustering::train's compute_centroids + post_process_centroids
// [faiss-upstream], reached from index.train(), /root/reference/src/index/feature_search_index.py:75.
// (K6, the assignment, runs on the tensor cores: filter2_topk_kernel<ARGMAX> for training iterations,
// gemm2_topk_kernel<128, ARGMAX> (3xTF32) for add-time assignment; the grouping of the points by centroid is
// csr.cuh.)  HBM-bound: n*d*4 bytes read once, nlist*d*4 written.  No float atomics: each list is summed in
// insertion order with a fixed interleave, so training is bit-reproducible.
#pragma once
#include "common.cuh"

namespace wb {

// sums[c, 0:d] = sum over slots of list c of x[perm[slot], 0:d]; counts[c] = list size.
// One CTA per list; a thread owns 4 adjacent columns (one 128-bit load per row) when d, ldx and the alignment of x and
// sums allow it, rows are taken four at a time into four accumulators per column that are combined as
// (a0 + a1) + (a2 + a3): the order is static, so the sums do not depend on the schedule (and the scalar branch, which
// uses the same order, gives the same bits).
__global__ void __launch_bounds__(256) segment_sum_kernel(const float* x, int ldx, int d, const uint32_t* perm,
                                                          const int64_t* off, float* sums, int64_t* counts) {
    const int64_t c = blockIdx.x;
    const int64_t b = off[c], e = off[c + 1];
    if (threadIdx.x == 0) counts[c] = e - b;
    if ((((d | ldx) & 3) | (((uintptr_t)x | (uintptr_t)sums) & 15)) == 0) {
        const int d4 = d >> 2, ld4 = ldx >> 2;
        const float4* x4 = reinterpret_cast<const float4*>(x);
        for (int col = threadIdx.x; col < d4; col += blockDim.x) {
            float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0, a2 = a0, a3 = a0;
            int64_t s = b;
            for (; s + 4 <= e; s += 4) {
                const uint32_t r0 = perm[s], r1 = perm[s + 1], r2 = perm[s + 2], r3 = perm[s + 3];
                const float4 v0 = __ldg(x4 + (size_t)r0 * ld4 + col), v1 = __ldg(x4 + (size_t)r1 * ld4 + col);
                const float4 v2 = __ldg(x4 + (size_t)r2 * ld4 + col), v3 = __ldg(x4 + (size_t)r3 * ld4 + col);
                a0.x += v0.x; a0.y += v0.y; a0.z += v0.z; a0.w += v0.w;
                a1.x += v1.x; a1.y += v1.y; a1.z += v1.z; a1.w += v1.w;
                a2.x += v2.x; a2.y += v2.y; a2.z += v2.z; a2.w += v2.w;
                a3.x += v3.x; a3.y += v3.y; a3.z += v3.z; a3.w += v3.w;
            }
            for (; s < e; ++s) {
                const float4 v = __ldg(x4 + (size_t)perm[s] * ld4 + col);
                a0.x += v.x; a0.y += v.y; a0.z += v.z; a0.w += v.w;
            }
            float4 r;
            r.x = (a0.x + a1.x) + (a2.x + a3.x);
            r.y = (a0.y + a1.y) + (a2.y + a3.y);
            r.z = (a0.z + a1.z) + (a2.z + a3.z);
            r.w = (a0.w + a1.w) + (a2.w + a3.w);
            reinterpret_cast<float4*>(sums + c * d)[col] = r;
        }
        return;
    }
    for (int col = threadIdx.x; col < d; col += blockDim.x) {
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;  // fixed 4-way interleave: order is static
        int64_t s = b;
        for (; s + 4 <= e; s += 4) {
            a0 += x[(size_t)perm[s] * ldx + col];
            a1 += x[(size_t)perm[s + 1] * ldx + col];
            a2 += x[(size_t)perm[s + 2] * ldx + col];
            a3 += x[(size_t)perm[s + 3] * ldx + col];
        }
        for (; s < e; ++s) a0 += x[(size_t)perm[s] * ldx + col];
        sums[c * d + col] = (a0 + a1) + (a2 + a3);
    }
}

// centroid <- sums / count for non-empty lists (empty lists keep their centroid)
__global__ void centroid_mean_kernel(const float* sums, const int64_t* counts, float* cent, int ld, int d,
                                     int64_t nlist) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < nlist * d) {
        const int64_t c = i / d;
        const int col = (int)(i - c * d);
        const int64_t n = counts[c];
        if (n > 0) cent[c * ld + col] = sums[i] / (float)n;
    }
}

// split_clusters [faiss-upstream], device half: the host picks, for every empty list ci, the list cj it is split from
// (a sequential draw over the list sizes, see wb_kmeans_update_dev); this kernel applies the pairs IN ORDER: ci becomes a
// copy of cj, the two are pushed apart by the +-1/1024 alternating perturbation.  One thread per column walks all the
// pairs, so a pair whose cj was itself written by an earlier pair sees the updated row without any synchronisation.
__global__ void split_apply_kernel(float* cent, int ld, int d, const int32_t* pairs, int npairs) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= d) return;
    const float EPS = 1.0f / 1024.0f;
    const float fa = (j % 2 == 0) ? 1 + EPS : 1 - EPS;
    const float fb = (j % 2 == 0) ? 1 - EPS : 1 + EPS;
    for (int i = 0; i < npairs; ++i) {
        const size_t ci = (size_t)pairs[2 * i], cj = (size_t)pairs[2 * i + 1];
        const float b = cent[cj * ld + j];
        cent[ci * ld + j] = b * fa;
        cent[cj * ld + j] = b * fb;
    }
}

// spherical k-means: L2-normalise each centroid row (fvec_renorm_L2); zero rows stay zero
__global__ void __launch_bounds__(256) renorm_rows_kernel(float* cent, int ld, int d) {
    __shared__ float red[8];
    float* row = cent + (size_t)blockIdx.x * ld;
    float s = 0.f;
    for (int c = threadIdx.x; c < d; c += blockDim.x) s += row[c] * row[c];
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    float t = 0.f;
    for (int w = 0; w < 8; ++w) t += red[w];
    if (t > 0.f) {
        const float inv = 1.0f / sqrtf(t);
        for (int c = threadIdx.x; c < d; c += blockDim.x) row[c] *= inv;
    }
}

// out += sum(v[0:n]) in double (objective of one k-means iteration)
__global__ void __launch_bounds__(256) sum_f32_kernel(const float* v, int64_t n, double* out) {
    __shared__ double red[8];
    double s = 0.0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        s += (double)v[i];
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += red[w];
        atomicAdd(out, t);
    }
}

}  // namespace wb
