// hamming.cu -- 256-bit Hamming distance (ORBmatcher::DescriptorDistance, src/ORBmatcher.cc:1649-1665 ==
// DBoW2 FORB::distance, FORB.cpp:81-101) as hardware POPC, and the brute-force nearest / second-nearest search.
//
// sgs_hamming_bf: each thread owns one query descriptor in registers (two 128-bit loads); train descriptors are staged
// through shared memory in tiles read as warp-wide broadcasts.  The train set is split across blockIdx.y so that small
// query sets still fill the 148 SMs; partial (best, idx, second) triples are merged in train order, which preserves the
// reference's "first strictly smaller wins" tie-break.  The all-pairs sweep is POPC/ALU bound, not HBM bound (DESIGN.md).
#include <cuda_runtime.h>

#include <vector>

#include "host_call.h"
#include "sgs_common.h"

namespace sgs {

constexpr int kBfThreads = 128;
constexpr int kBfTile = 256;  // train descriptors per shared-memory tile (8 KB)

__device__ __forceinline__ int hamming256(const uint4& a0, const uint4& a1, const uint4& b0, const uint4& b1) {
    return __popc(a0.x ^ b0.x) + __popc(a0.y ^ b0.y) + __popc(a0.z ^ b0.z) + __popc(a0.w ^ b0.w) +
           __popc(a1.x ^ b1.x) + __popc(a1.y ^ b1.y) + __popc(a1.z ^ b1.z) + __popc(a1.w ^ b1.w);
}

__global__ void __launch_bounds__(kBfThreads) hamming_bf_kernel(const uint4* __restrict__ query, int nq, const uint4* __restrict__ train, int nt,
                                                                int chunk, int32_t* __restrict__ p_idx, int32_t* __restrict__ p_best,
                                                                int32_t* __restrict__ p_second) {
    __shared__ uint4 tile[kBfTile * 2];
    const int q = blockIdx.x * kBfThreads + threadIdx.x;
    const int t_begin = blockIdx.y * chunk;
    const int t_end = min(nt, t_begin + chunk);
    uint4 a0 = make_uint4(0, 0, 0, 0), a1 = a0;
    if (q < nq) { a0 = __ldg(&query[2 * q]); a1 = __ldg(&query[2 * q + 1]); }
    int best = 256, second = 256, idx = -1;
    for (int t0 = t_begin; t0 < t_end; t0 += kBfTile) {
        const int cnt = min(kBfTile, t_end - t0);
        __syncthreads();
        for (int i = threadIdx.x; i < cnt * 2; i += kBfThreads) tile[i] = __ldg(&train[2 * (int64_t)t0 + i]);
        __syncthreads();
#pragma unroll 4
        for (int j = 0; j < cnt; ++j) {
            const int d = hamming256(a0, a1, tile[2 * j], tile[2 * j + 1]);
            if (d < best) { second = best; best = d; idx = t0 + j; }
            else if (d < second) second = d;
        }
    }
    if (q < nq) {
        const int64_t o = (int64_t)blockIdx.y * nq + q;
        p_idx[o] = idx; p_best[o] = best; p_second[o] = second;
    }
}

__global__ void hamming_bf_merge_kernel(int nq, int nsplit, const int32_t* __restrict__ p_idx, const int32_t* __restrict__ p_best,
                                        const int32_t* __restrict__ p_second, int32_t* __restrict__ o_idx, int32_t* __restrict__ o_best,
                                        int32_t* __restrict__ o_second) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= nq) return;
    int best = 256, second = 256, idx = -1;
    for (int s = 0; s < nsplit; ++s) {  // ascending train order
        const int64_t o = (int64_t)s * nq + q;
        const int b = p_best[o], sc = p_second[o], ix = p_idx[o];
        if (b < best) { second = min(best, sc); best = b; idx = ix; }
        else second = min(second, b);
    }
    o_idx[q] = idx; o_best[q] = best; o_second[q] = second;
}

__global__ void hamming_pairs_kernel(const uint4* __restrict__ a, const uint4* __restrict__ b, int n, int32_t* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out[i] = hamming256(__ldg(&a[2 * i]), __ldg(&a[2 * i + 1]), __ldg(&b[2 * i]), __ldg(&b[2 * i + 1]));
}

// scratch: 3 * nsplit * nq int32.  Returns the split count through *nsplit_out when scratch == nullptr (sizing query).
int bf_plan_splits(int nq, int nt) {
    const int qblocks = (nq + kBfThreads - 1) / kBfThreads;
    int target = (2 * 148 + qblocks - 1) / qblocks;          // aim for >= 2 waves of blocks
    int max_split = (nt + kBfTile - 1) / kBfTile;            // at least one tile per split
    if (target > max_split) target = max_split;
    if (target < 1) target = 1;
    return target;
}

int hamming_bf_device(const uint8_t* d_q, int nq, const uint8_t* d_t, int nt, int32_t* d_idx, int32_t* d_best, int32_t* d_second,
                      int32_t* d_scratch, int nsplit, cudaStream_t st) {
    if (nq <= 0) return SGS_OK;
    const int qblocks = (nq + kBfThreads - 1) / kBfThreads;
    if (nt <= 0) nsplit = 1;
    int chunk = nt > 0 ? ((nt + nsplit - 1) / nsplit + kBfTile - 1) / kBfTile * kBfTile : kBfTile;
    if (nsplit == 1) {
        hamming_bf_kernel<<<dim3(qblocks, 1), kBfThreads, 0, st>>>((const uint4*)d_q, nq, (const uint4*)d_t, nt, chunk, d_idx, d_best, d_second);
    } else {
        int32_t* p_idx = d_scratch; int32_t* p_best = d_scratch + (int64_t)nsplit * nq; int32_t* p_second = d_scratch + 2 * (int64_t)nsplit * nq;
        hamming_bf_kernel<<<dim3(qblocks, nsplit), kBfThreads, 0, st>>>((const uint4*)d_q, nq, (const uint4*)d_t, nt, chunk, p_idx, p_best, p_second);
        hamming_bf_merge_kernel<<<(nq + 255) / 256, 256, 0, st>>>(nq, nsplit, p_idx, p_best, p_second, d_idx, d_best, d_second);
    }
    SGS_CUDA_TRY(cudaGetLastError());
    return SGS_OK;
}

}  // namespace sgs

using namespace sgs;

extern "C" {

SGS_API int sgs_hamming_pairs(const uint8_t* a, const uint8_t* b, int n, int32_t* dist, int device) {
    if (n < 0 || (n > 0 && (!a || !b || !dist))) { set_error("sgs_hamming_pairs: bad argument"); return SGS_ERR_INVALID; }
    if (n == 0) return SGS_OK;
    SGS_CUDA_TRY(cudaSetDevice(device));
    HostCall c("sgs_hamming_pairs");
    const uint4 *da, *db; int32_t* dd;
    c.in(&da, a, 2 * (size_t)n); c.in(&db, b, 2 * (size_t)n); c.out(&dd, dist, n);
    if (int rc = c.upload()) return rc;
    hamming_pairs_kernel<<<(n + 255) / 256, 256>>>(da, db, n, dd);
    SGS_CUDA_TRY(cudaGetLastError());
    return c.download();
}

SGS_API int sgs_hamming_bf_scratch_elems(int nq, int nt, int64_t* elems) {
    if (!elems) { set_error("sgs_hamming_bf_scratch_elems: NULL"); return SGS_ERR_INVALID; }
    const int ns = bf_plan_splits(nq, nt);
    *elems = ns > 1 ? 3 * (int64_t)ns * nq : 0;
    return SGS_OK;
}

SGS_API int sgs_hamming_bf_device(const uint8_t* d_query, int nq, const uint8_t* d_train, int nt, int32_t* d_best_idx, int32_t* d_best_dist,
                                  int32_t* d_second_dist, int32_t* d_scratch, void* stream) {
    if (nq < 0 || nt < 0) { set_error("sgs_hamming_bf_device: negative size"); return SGS_ERR_INVALID; }
    if (nq == 0) return SGS_OK;
    if (!d_query || !d_best_idx || !d_best_dist || !d_second_dist || (nt > 0 && !d_train)) { set_error("sgs_hamming_bf_device: NULL pointer"); return SGS_ERR_INVALID; }
    int ns = bf_plan_splits(nq, nt);
    if (ns > 1 && !d_scratch) ns = 1;  // no scratch: single pass over the train set per query block
    return hamming_bf_device(d_query, nq, d_train, nt, d_best_idx, d_best_dist, d_second_dist, d_scratch, ns, (cudaStream_t)stream);
}

SGS_API int sgs_hamming_bf(const uint8_t* query, int nq, const uint8_t* train, int nt, int32_t* best_idx, int32_t* best_dist,
                           int32_t* second_dist, int device) {
    if (nq < 0 || nt < 0) { set_error("sgs_hamming_bf: negative size"); return SGS_ERR_INVALID; }
    if (nq == 0) return SGS_OK;
    if (!query || !best_idx || !best_dist || !second_dist || (nt > 0 && !train)) { set_error("sgs_hamming_bf: NULL pointer"); return SGS_ERR_INVALID; }
    SGS_CUDA_TRY(cudaSetDevice(device));
    const int ns = bf_plan_splits(nq, nt);
    HostCall c("sgs_hamming_bf");
    const uint8_t *dq, *dt; int32_t *di, *dbst, *dsec, *dscr;
    c.in(&dq, query, 32 * (size_t)nq); c.in(&dt, train, 32 * (size_t)nt);
    c.out(&di, best_idx, nq); c.out(&dbst, best_dist, nq); c.out(&dsec, second_dist, nq); c.out(&dscr, nullptr, ns > 1 ? (size_t)3 * ns * nq : 0);
    if (int rc = c.upload()) return rc;
    if (int rc = hamming_bf_device(dq, nq, dt, nt, di, dbst, dsec, dscr, ns, 0)) return rc;
    return c.download();
}

}  // extern "C"

// MapPoint::ComputeDistinctiveDescriptors (src/MapPoint.cc:242-307) for a batch of map points: one warp per map point, lane i owns row i of
// the distance matrix (rows i and i + 32 when a point has more than 32 observations, at most 64), finds vDists[0.5 (n - 1)] of its row by
// counting ranks (distances are integers 0..256) and the warp keeps the first row with the smallest median.
namespace sgs {
__global__ void __launch_bounds__(256) distinctive_kernel(const uint8_t* __restrict__ desc, const int32_t* __restrict__ counts, int max_obs, int npoints,
                                                          int32_t* __restrict__ best_idx) {
    const int p = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (p >= npoints) return;
    const int n = min(counts[p], max_obs);
    const uint4* D = reinterpret_cast<const uint4*>(desc + (int64_t)p * max_obs * 32);
    const int k = (int)(0.5 * (double)(n - 1));
    unsigned best = 0xffffffffu;
    for (int i = lane; i < n; i += 32) {
        const uint4 a0 = __ldg(D + 2 * i), a1 = __ldg(D + 2 * i + 1);
        int dist[64];
        for (int j = 0; j < n; ++j) {
            const uint4 b0 = __ldg(D + 2 * j), b1 = __ldg(D + 2 * j + 1);
            dist[j] = __popc(a0.x ^ b0.x) + __popc(a0.y ^ b0.y) + __popc(a0.z ^ b0.z) + __popc(a0.w ^ b0.w) + __popc(a1.x ^ b1.x) + __popc(a1.y ^ b1.y) +
                      __popc(a1.z ^ b1.z) + __popc(a1.w ^ b1.w);
        }
        // k-th smallest: the value v with  #(dist < v) <= k < #(dist <= v)
        int median = 0;
        for (int j = 0; j < n; ++j) {
            int less = 0, leq = 0;
            for (int q = 0; q < n; ++q) { less += dist[q] < dist[j]; leq += dist[q] <= dist[j]; }
            if (less <= k && k < leq) { median = dist[j]; break; }
        }
        best = min(best, ((unsigned)median << 8) | (unsigned)i);
    }
    best = __reduce_min_sync(0xffffffffu, best);
    if (lane == 0) best_idx[p] = n > 0 ? (int)(best & 0xffu) : 0;
}
}  // namespace sgs

extern "C" {

SGS_API int sgs_distinctive_descriptor_batch_device(const uint8_t* d_desc, const int32_t* d_counts, int max_obs, int npoints, int32_t* d_best_idx, void* stream) {
    if (!d_desc || !d_counts || !d_best_idx || npoints < 1 || max_obs < 1) { sgs::set_error("sgs_distinctive_descriptor_batch_device: bad argument"); return SGS_ERR_INVALID; }
    if (max_obs > 64) { sgs::set_error("sgs_distinctive_descriptor_batch_device: at most 64 observations per map point"); return SGS_ERR_UNSUPPORTED; }
    sgs::distinctive_kernel<<<(npoints + 7) / 8, 256, 0, (cudaStream_t)stream>>>(d_desc, d_counts, max_obs, npoints, d_best_idx);
    SGS_CUDA_TRY(cudaGetLastError());
    return SGS_OK;
}

}  // extern "C"
