// dynreject.cu -- geometry half of Frame::RmDynamicPointWithSemanticAndGeometry (src/Frame.cc:430-612):
//   per keypoint: point-in-person-box test (isInDynamicRegion :629-652), epipolar distance in FP64
//   (CheckEpiLineDistToRmDynamicPoint :613-627) against 0.2 (inside a box) or 1.0, then the ORDERED compaction of
//   keypoints + descriptor rows that the erase loop (:563-597) amounts to, with the restore-all guard (:599-604).
// One block per frame; FP64 products and sums are individually rounded (the reference build has no FMA).
#include <cuda_runtime.h>

#include <vector>

#include "host_call.h"
#include "sgs_common.h"

namespace sgs {

constexpr int kDynThreads = 256;

__device__ __forceinline__ bool epi_keep(float x, float y, float px, float py, const double* F, bool in_box, double* dist_out) {
    const double xd = (double)x, yd = (double)y;
    const double a = __dadd_rn(__dadd_rn(__dmul_rn(xd, F[0]), __dmul_rn(yd, F[1])), F[2]);
    const double b = __dadd_rn(__dadd_rn(__dmul_rn(xd, F[3]), __dmul_rn(yd, F[4])), F[5]);
    const double c = __dadd_rn(__dadd_rn(__dmul_rn(xd, F[6]), __dmul_rn(yd, F[7])), F[8]);
    const double son = fabs(__dadd_rn(__dadd_rn(__dmul_rn(a, (double)px), __dmul_rn(b, (double)py)), c));
    const double mom = __dsqrt_rn(__dadd_rn(__dmul_rn(a, a), __dmul_rn(b, b)));
    const double dist = __ddiv_rn(son, mom);
    if (dist_out) *dist_out = dist;
    return dist < (in_box ? 0.2 : 1.0);   // NaN compares false -> removed, as in the reference
}

__device__ __forceinline__ bool in_any_box(float x, float y, const sgs_rect* boxes, int nboxes) {
    for (int b = 0; b < nboxes; ++b) {
        const sgs_rect r = boxes[b];
        if (x > r.x && x < __fadd_rn(r.x, r.w) && y > r.y && y < __fadd_rn(r.y, r.h)) return true;
    }
    return false;
}

// verdict-only kernel for the single-frame host API
__global__ void dynreject_flags_kernel(const float2* __restrict__ cur, const float2* __restrict__ prev, int n, const double* __restrict__ F, int have_F,
                                       const sgs_rect* __restrict__ boxes, int nboxes, int have_dyn, uint8_t* __restrict__ keep, double* __restrict__ dist) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float2 c = cur[i], p = prev[i];
    const bool inb = have_dyn && in_any_box(c.x, c.y, boxes, nboxes);
    double d = 0.0;
    bool ok = true;
    if (have_F) ok = epi_keep(c.x, c.y, p.x, p.y, F, inb, &d);
    keep[i] = ok ? 1 : 0;
    if (dist) dist[i] = d;
}

// fused batched kernel: verdicts + block-wide ordered compaction
__global__ void __launch_bounds__(kDynThreads) dynreject_batch_kernel(const sgs_keypoint* __restrict__ kps, const uint8_t* __restrict__ desc,
                                                                      const int32_t* __restrict__ counts, int cap, const float2* __restrict__ prev,
                                                                      const double* __restrict__ Fm, const sgs_rect* __restrict__ boxes,
                                                                      const int32_t* __restrict__ nboxes, int max_boxes,
                                                                      const uint8_t* __restrict__ have_dyn, int nfeatures,
                                                                      sgs_keypoint* __restrict__ kps_out, uint8_t* __restrict__ desc_out,
                                                                      int32_t* __restrict__ counts_out, uint8_t* __restrict__ keep_out) {
    extern __shared__ int32_t s_pos[];   // [cap] exclusive positions (or -1)
    __shared__ int s_warp[kDynThreads / 32];
    __shared__ int s_total, s_carry;
    __shared__ double sF[9];
    const int f = blockIdx.x;
    const int n = min(counts[f], cap);
    const int64_t base = (int64_t)f * cap;
    if (threadIdx.x < 9) sF[threadIdx.x] = Fm[9 * f + threadIdx.x];
    if (threadIdx.x == 0) { s_carry = 0; }
    __syncthreads();
    const bool have_F = !(sF[0] != sF[0]);   // NaN marks the empty matrix (quirk Q11: keep everything)
    const bool dyn = have_dyn[f] != 0;
    const int nb = dyn ? min(nboxes[f], max_boxes) : 0;
    const sgs_rect* bx = boxes + (int64_t)f * max_boxes;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i0 = 0; i0 < n; i0 += kDynThreads) {
        const int i = i0 + threadIdx.x;
        bool ok = false;
        if (i < n) {
            const sgs_keypoint k = kps[base + i];
            const float2 p = prev[base + i];
            const bool inb = dyn && in_any_box(k.x, k.y, bx, nb);
            ok = have_F ? epi_keep(k.x, k.y, p.x, p.y, sF, inb, nullptr) : true;
            if (keep_out) keep_out[base + i] = ok ? 1 : 0;
        }
        const unsigned m = __ballot_sync(0xffffffffu, ok);
        if (lane == 0) s_warp[warp] = __popc(m);
        __syncthreads();
        int off = s_carry;
        for (int w = 0; w < warp; ++w) off += s_warp[w];
        if (i < n) s_pos[i] = ok ? off + __popc(m & ((1u << lane) - 1)) : -1;
        __syncthreads();
        if (threadIdx.x == 0) { int t = 0; for (int w = 0; w < kDynThreads / 32; ++w) t += s_warp[w]; s_carry += t; }
        __syncthreads();
    }
    if (threadIdx.x == 0) s_total = s_carry;
    __syncthreads();
    const int total = s_total;
    const bool restore = dyn && ((double)total < (double)nfeatures * 0.1);     // Frame.cc:599
    const int n_out = restore ? n : total;
    if (threadIdx.x == 0) counts_out[f] = n_out;
    // move keypoints (7 words) and descriptor rows (8 words) with word-granular coalesced copies
    const uint32_t* kin = reinterpret_cast<const uint32_t*>(kps + base);
    uint32_t* kout = reinterpret_cast<uint32_t*>(kps_out + base);
    for (int t = threadIdx.x; t < n * 7; t += kDynThreads) {
        const int i = t / 7, wd = t - i * 7;
        const int dst = restore ? i : s_pos[i];
        if (dst >= 0) kout[dst * 7 + wd] = kin[t];
    }
    const uint32_t* din = reinterpret_cast<const uint32_t*>(desc + base * 32);
    uint32_t* dout = reinterpret_cast<uint32_t*>(desc_out + base * 32);
    for (int t = threadIdx.x; t < n * 8; t += kDynThreads) {
        const int i = t >> 3, wd = t & 7;
        const int dst = restore ? i : s_pos[i];
        if (dst >= 0) dout[dst * 8 + wd] = din[t];
    }
}

}  // namespace sgs

using namespace sgs;

extern "C" {

SGS_API int sgs_dynreject(const float* cur_xy, const float* prev_xy, int n, const double* F, const sgs_rect* boxes, int nboxes, int have_dyn,
                          int nfeatures, uint8_t* keep, double* dist, int* nkeep, int* restored, int device) {
    if (n < 0 || (n > 0 && (!cur_xy || !prev_xy || !keep)) || !nkeep) { set_error("sgs_dynreject: bad argument"); return SGS_ERR_INVALID; }
    if (nboxes < 0 || (nboxes > 0 && !boxes)) { set_error("sgs_dynreject: bad boxes"); return SGS_ERR_INVALID; }
    *nkeep = n;
    if (restored) *restored = 0;
    SGS_CUDA_TRY(cudaSetDevice(device));
    if (n > 0) {
        HostCall c("sgs_dynreject");
        const float2 *dc, *dp; const double* dF; const sgs_rect* db; uint8_t* dk; double* dd;
        // without F or boxes the kernel reads neither, but still gets a valid address: that of an empty slice
        c.in(&dc, cur_xy, n); c.in(&dp, prev_xy, n); c.in(&dF, F, F ? 9 : 0); c.in(&db, boxes, nboxes);
        c.out(&dk, keep, n); c.out(&dd, dist, n);
        if (int rc = c.upload()) return rc;
        dynreject_flags_kernel<<<(n + 255) / 256, 256>>>(dc, dp, n, dF, F ? 1 : 0, db, nboxes, have_dyn, dk, dd);
        SGS_CUDA_TRY(cudaGetLastError());
        if (int rc = c.download()) return rc;
    }
    int sum = 0;
    for (int i = 0; i < n; ++i) sum += keep[i];
    *nkeep = sum;
    if (restored) *restored = (have_dyn && (double)sum < (double)nfeatures * 0.1) ? 1 : 0;
    return SGS_OK;
}

SGS_API int sgs_dynreject_batch_device(const sgs_keypoint* d_kps, const uint8_t* d_desc, const int32_t* d_counts, int cap, int nframes,
                                       const float* d_prev_xy, const double* d_F, const sgs_rect* d_boxes, const int32_t* d_nboxes, int max_boxes,
                                       const uint8_t* d_have_dyn, int nfeatures, sgs_keypoint* d_kps_out, uint8_t* d_desc_out,
                                       int32_t* d_counts_out, uint8_t* d_keep, void* stream) {
    if (!d_kps || !d_desc || !d_counts || !d_prev_xy || !d_F || !d_nboxes || !d_have_dyn || !d_kps_out || !d_desc_out || !d_counts_out ||
        (max_boxes > 0 && !d_boxes) || cap < 1 || nframes < 1) { set_error("sgs_dynreject_batch_device: bad argument"); return SGS_ERR_INVALID; }
    const size_t smem = (size_t)cap * 4;
    if (smem > 160 * 1024) { set_error("sgs_dynreject_batch_device: cap too large"); return SGS_ERR_UNSUPPORTED; }
    SGS_CUDA_TRY(cudaFuncSetAttribute(dynreject_batch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dynreject_batch_kernel<<<nframes, kDynThreads, smem, (cudaStream_t)stream>>>(d_kps, d_desc, d_counts, cap, (const float2*)d_prev_xy, d_F, d_boxes, d_nboxes,
                                                                               max_boxes, d_have_dyn, nfeatures, d_kps_out, d_desc_out, d_counts_out, d_keep);
    SGS_CUDA_TRY(cudaGetLastError());
    return SGS_OK;
}

}  // extern "C"
