// frame_geom.cu -- two per-point pieces of the Frame class that sit between the extractor and the matchers:
//   Frame::ComputeStereoFromRGBD (src/Frame.cc:893-914): depth lookup at the (distorted) keypoint, uRight = xUn - bf / d;
//   Frame::isInFrustum (src/Frame.cc:296-352) + MapPoint::PredictScale (src/MapPoint.cc:400-418): the projection that fills
//   mbTrackInView / mTrackProjX / mTrackProjY / mTrackProjXR / mnTrackScaleLevel / mTrackViewCos for
//   ORBmatcher::SearchByProjection(Frame&, vector<MapPoint*>&, th) (src/ORBmatcher.cc:45-129).
// cv::Mat float arithmetic is reproduced as OpenCV evaluates it (pinned against cv2): a plain 3x3 * 3x1 gemm sums float products in
// float, transposed gemm / cv::norm / Mat::dot accumulate in double and round once; scalar float expressions are individually rounded (-fmad=false).  The only non-bit-exact piece is logf in PredictScale
// (device log vs glibc logf): the predicted level can differ when log(ratio)/log(scaleFactor) falls within an ulp of an integer.
#include <cuda_runtime.h>

#include "host_call.h"
#include "sgs_common.h"
#include "sgs_logf.h"

namespace sgs {

__global__ void __launch_bounds__(256) stereo_from_depth_kernel(const sgs_keypoint* __restrict__ kps, const sgs_keypoint* __restrict__ kps_un,
                                                                const int32_t* __restrict__ counts, int cap, const float* __restrict__ depth,
                                                                int64_t depth_fstride, int depth_pitch, float bf, float* __restrict__ u_right,
                                                                float* __restrict__ depth_out) {
    const int f = blockIdx.y, i = blockIdx.x * 256 + threadIdx.x;
    if (i >= cap) return;
    const int64_t o = (int64_t)f * cap + i;
    float ur = -1.f, dz = -1.f;
    if (i < min(counts[f], cap)) {
        const sgs_keypoint k = kps[o];
        const float d = __ldg(depth + (int64_t)f * depth_fstride + (int64_t)(int)k.y * depth_pitch + (int)k.x);
        if (d > 0) { dz = d; ur = __fsub_rn(kps_un ? kps_un[o].x : k.x, __fdiv_rn(bf, d)); }
    }
    u_right[o] = ur;
    if (depth_out) depth_out[o] = dz;
}

// cv::undistortPoints(pt, K, distCoef, R = I, P = K) for one point: calib3d cvUndistortPointsInternal -- double arithmetic, five fixed-point
// iterations (the default criteria), re-projection with K; every product and sum individually rounded (no FMA), the zero-coefficient terms of
// OpenCV's general expressions are kept so that the roundings are the same.  Bit-exact against cv2.undistortPoints.
__device__ __forceinline__ float2 undistort_point(float xf, float yf, double fx, double fy, double cx, double cy, double k0, double k1, double p1, double p2,
                                                  double k2) {
    const double ifx = 1. / fx, ify = 1. / fy;
    double x = xf, y = yf;
    const double u = x, v = y;
    x = (x - cx) * ifx; y = (y - cy) * ify;
    const double x0 = x, y0 = y;
    for (int j = 0; j < 5; ++j) {
        const double r2 = x * x + y * y;
        const double icdist = 1. / (1 + ((k2 * r2 + k1) * r2 + k0) * r2);       // numerator 1 + ((k7 r2 + k6) r2 + k5) r2 with k5..k7 = 0 is exactly 1
        if (icdist < 0) { x = (u - cx) * ifx; y = (v - cy) * ify; break; }
        const double deltaX = 2 * p1 * x * y + p2 * (r2 + 2 * x * x), deltaY = p1 * (r2 + 2 * y * y) + 2 * p2 * x * y;
        x = (x0 - deltaX) * icdist; y = (y0 - deltaY) * icdist;
    }
    return make_float2((float)(fx * x + cx), (float)(fy * y + cy));          // (xx * ww) with ww = 1/(0 x + 0 y + 1) = 1
}

__global__ void __launch_bounds__(256) undistort_kernel(const sgs_keypoint* __restrict__ kps, const float2* __restrict__ xy_in, const int32_t* __restrict__ counts,
                                                        int cap, float fx, float fy, float cx, float cy, float k0, float k1, float p1, float p2, float k2,
                                                        sgs_keypoint* __restrict__ kps_un, float2* __restrict__ xy_out) {
    const int f = blockIdx.y, i = blockIdx.x * 256 + threadIdx.x;
    const int n = counts ? min(counts[f], cap) : cap;
    if (i >= n) return;
    const int64_t o = (int64_t)f * cap + i;
    if (kps) {
        sgs_keypoint k = kps[o];
        const float2 r = k0 == 0.f ? make_float2(k.x, k.y) : undistort_point(k.x, k.y, fx, fy, cx, cy, k0, k1, p1, p2, k2);       // src/Frame.cc:656-660
        k.x = r.x; k.y = r.y;
        kps_un[o] = k;
    } else {
        const float2 q = xy_in[o];
        xy_out[o] = undistort_point(q.x, q.y, fx, fy, cx, cy, k0, k1, p1, p2, k2);
    }
}

__global__ void __launch_bounds__(256) frustum_kernel(const sgs_frustum_batch A, int nlevels, float log_sf) {
    const int f = blockIdx.y, i = blockIdx.x * 256 + threadIdx.x;
    const int n = min(A.mp_n[f], A.point_cap);
    if (i >= A.point_cap) return;
    const int64_t o = (int64_t)f * A.point_cap + i;
    uint8_t in = 0; float pu = 0.f, pv = 0.f, pxr = 0.f, vcos = 0.f; int lvl = 0;
    if (i < n) {
        const float* T = A.tcw + (int64_t)f * 16;
        const float R0 = T[0], R1 = T[1], R2 = T[2], R3 = T[4], R4 = T[5], R5 = T[6], R6 = T[8], R7 = T[9], R8 = T[10], t0 = T[3], t1 = T[7], t2 = T[11];
        // mOw = -Rcw^T tcw: transposed gemm = general path, double accumulator, one rounding
        const float Ox = (float)(((double)(-R0) * t0 + (double)(-R3) * t1) + (double)(-R6) * t2);
        const float Oy = (float)(((double)(-R1) * t0 + (double)(-R4) * t1) + (double)(-R7) * t2);
        const float Oz = (float)(((double)(-R2) * t0 + (double)(-R5) * t1) + (double)(-R8) * t2);
        const float X = A.mp_xyz[3 * o], Y = A.mp_xyz[3 * o + 1], Z = A.mp_xyz[3 * o + 2];
        // mRcw * P + mtcw: OpenCV's small-matrix gemm path (float products summed in float, then (float)((double)sum + (double)c))
        const float PcX = (float)((double)__fadd_rn(__fadd_rn(__fmul_rn(R0, X), __fmul_rn(R1, Y)), __fmul_rn(R2, Z)) + (double)t0);
        const float PcY = (float)((double)__fadd_rn(__fadd_rn(__fmul_rn(R3, X), __fmul_rn(R4, Y)), __fmul_rn(R5, Z)) + (double)t1);
        const float PcZ = (float)((double)__fadd_rn(__fadd_rn(__fmul_rn(R6, X), __fmul_rn(R7, Y)), __fmul_rn(R8, Z)) + (double)t2);
        bool ok = !(PcZ < 0.0f);
        const float invz = __fdiv_rn(1.0f, PcZ);
        const float u = __fadd_rn(__fmul_rn(__fmul_rn(A.cam.fx, PcX), invz), A.cam.cx), v = __fadd_rn(__fmul_rn(__fmul_rn(A.cam.fy, PcY), invz), A.cam.cy);
        ok = ok && !(u < A.cam.min_x || u > A.cam.max_x) && !(v < A.cam.min_y || v > A.cam.max_y);
        const float maxD = __fmul_rn(1.2f, A.mp_max_dist[o]), minD = __fmul_rn(0.8f, A.mp_min_dist[o]);
        const float Px = __fsub_rn(X, Ox), Py = __fsub_rn(Y, Oy), Pz = __fsub_rn(Z, Oz);
        const float dist = (float)sqrt(((double)Px * Px + (double)Py * Py) + (double)Pz * Pz);
        ok = ok && !(dist < minD || dist > maxD);
        const float nx = A.mp_normal[3 * o], ny = A.mp_normal[3 * o + 1], nz = A.mp_normal[3 * o + 2];
        const float vc = (float)((((double)Px * nx + (double)Py * ny) + (double)Pz * nz) / (double)dist);
        ok = ok && !(vc < A.viewing_cos_limit);
        if (ok) {
            const float ratio = __fdiv_rn(A.mp_max_dist[o], dist);
            int ns = (int)ceilf(__fdiv_rn(glibc_logf(ratio), log_sf));          // MapPoint.cc:402-418, libm logf restated (sgs_logf.h)
            ns = ns < 0 ? 0 : (ns >= nlevels ? nlevels - 1 : ns);
            in = 1; pu = u; pv = v; pxr = __fsub_rn(u, __fmul_rn(A.cam.bf, invz)); lvl = ns; vcos = vc;
        }
    }
    A.mp_inview[o] = in; A.proj_x[o] = pu; A.proj_y[o] = pv; A.proj_xr[o] = pxr; A.level[o] = lvl; A.view_cos[o] = vcos;
}

}  // namespace sgs

using namespace sgs;

extern "C" {

SGS_API int sgs_stereo_from_depth_batch_device(const sgs_keypoint* d_kps, const sgs_keypoint* d_kps_un, const int32_t* d_counts, int cap, int nframes,
                                               const float* d_depth, size_t depth_frame_stride, int depth_pitch, float bf, float* d_u_right,
                                               float* d_depth_out, void* stream) {
    if (!d_kps || !d_counts || !d_depth || !d_u_right || cap < 1 || nframes < 1 || depth_pitch < 1) {
        set_error("sgs_stereo_from_depth_batch_device: bad argument"); return SGS_ERR_INVALID;
    }
    dim3 grid((cap + 255) / 256, nframes);
    stereo_from_depth_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_kps, d_kps_un, d_counts, cap, d_depth, (int64_t)depth_frame_stride, depth_pitch, bf,
                                                                     d_u_right, d_depth_out);
    SGS_CUDA_TRY(cudaGetLastError());
    return SGS_OK;
}

SGS_API int sgs_undistort_batch_device(const sgs_keypoint* d_kps, const int32_t* d_counts, int cap, int nframes, float fx, float fy, float cx, float cy,
                                       const float* dist_coef5, sgs_keypoint* d_kps_un, void* stream) {
    if (!d_kps || !d_counts || !d_kps_un || !dist_coef5 || cap < 1 || nframes < 1) { set_error("sgs_undistort_batch_device: bad argument"); return SGS_ERR_INVALID; }
    dim3 grid((cap + 255) / 256, nframes);
    undistort_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_kps, nullptr, d_counts, cap, fx, fy, cx, cy, dist_coef5[0], dist_coef5[1], dist_coef5[2],
                                                             dist_coef5[3], dist_coef5[4], d_kps_un, nullptr);
    SGS_CUDA_TRY(cudaGetLastError());
    return SGS_OK;
}

SGS_API int sgs_undistort_points(const float* xy, int n, float fx, float fy, float cx, float cy, const float* dist_coef5, float* out_xy, int device) {
    if (n < 0 || !dist_coef5 || (n > 0 && (!xy || !out_xy))) { set_error("sgs_undistort_points: bad argument"); return SGS_ERR_INVALID; }
    if (n == 0) return SGS_OK;
    SGS_CUDA_TRY(cudaSetDevice(device));
    HostCall c("sgs_undistort_points");
    const float2* d_xy; float2* d_out;
    c.in(&d_xy, xy, n); c.out(&d_out, out_xy, n);
    if (int rc = c.upload()) return rc;
    undistort_kernel<<<dim3((n + 255) / 256, 1), 256>>>(nullptr, d_xy, nullptr, n, fx, fy, cx, cy, dist_coef5[0], dist_coef5[1], dist_coef5[2], dist_coef5[3],
                                                        dist_coef5[4], nullptr, d_out);
    return c.download();
}

// Frame::ComputeImageBounds (src/Frame.cc:686-714): mnMinX, mnMinY, mnMaxX, mnMaxY from the undistorted image corners
SGS_API int sgs_image_bounds(int width, int height, float fx, float fy, float cx, float cy, const float* dist_coef5, float* bounds4, int device) {
    if (!dist_coef5 || !bounds4) { set_error("sgs_image_bounds: NULL"); return SGS_ERR_INVALID; }
    if (dist_coef5[0] == 0.0f) { bounds4[0] = 0.f; bounds4[1] = 0.f; bounds4[2] = (float)width; bounds4[3] = (float)height; return SGS_OK; }
    const float c[8] = {0.f, 0.f, (float)width, 0.f, 0.f, (float)height, (float)width, (float)height};
    float u[8];
    const int rc = sgs_undistort_points(c, 4, fx, fy, cx, cy, dist_coef5, u, device);
    if (rc != SGS_OK) return rc;
    bounds4[0] = u[0] < u[4] ? u[0] : u[4]; bounds4[2] = u[2] > u[6] ? u[2] : u[6];
    bounds4[1] = u[1] < u[3] ? u[1] : u[3]; bounds4[3] = u[5] > u[7] ? u[5] : u[7];
    return SGS_OK;
}

SGS_API int sgs_frustum_batch_device(const sgs_frustum_batch* a, int nframes, void* stream) {
    if (!a || !a->tcw || !a->mp_xyz || !a->mp_normal || !a->mp_min_dist || !a->mp_max_dist || !a->mp_n || !a->mp_inview || !a->proj_x || !a->proj_y ||
        !a->proj_xr || !a->level || !a->view_cos || a->point_cap < 1 || nframes < 1) {
        set_error("sgs_frustum_batch_device: bad argument"); return SGS_ERR_INVALID;
    }
    if (a->cam.nlevels < 1 || a->cam.nlevels > 16 || !(a->cam.scale_factors[1] > 1.f) && a->cam.nlevels > 1) {
        set_error("sgs_frustum_batch_device: camera scale table missing"); return SGS_ERR_INVALID;
    }
    const float log_sf = logf(a->cam.nlevels > 1 ? a->cam.scale_factors[1] : 1.2f);      // mfLogScaleFactor = log(mfScaleFactor), src/Frame.cc:139
    dim3 grid((a->point_cap + 255) / 256, nframes);
    frustum_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(*a, a->cam.nlevels, log_sf);
    SGS_CUDA_TRY(cudaGetLastError());
    return SGS_OK;
}

// host-pointer variant for one frame (the reference calls isInFrustum per local-map point in Tracking::SearchLocalPoints, src/Tracking.cc:1262-1290)
SGS_API int sgs_frustum(const sgs_camera* cam, const float* tcw, int n, const float* xyz, const float* normal, const float* min_dist, const float* max_dist,
                        float viewing_cos_limit, uint8_t* inview, float* proj_x, float* proj_y, float* proj_xr, int32_t* level, float* view_cos, int device) {
    if (!cam || !tcw || n < 0 || (n > 0 && (!xyz || !normal || !min_dist || !max_dist || !inview || !proj_x || !proj_y || !proj_xr || !level || !view_cos))) {
        set_error("sgs_frustum: bad argument"); return SGS_ERR_INVALID;
    }
    if (n == 0) return SGS_OK;
    SGS_CUDA_TRY(cudaSetDevice(device));
    HostCall c("sgs_frustum");
    sgs_frustum_batch a;
    c.in(&a.tcw, tcw, 16); c.in(&a.mp_xyz, xyz, 3 * (size_t)n); c.in(&a.mp_normal, normal, 3 * (size_t)n); c.in(&a.mp_min_dist, min_dist, n);
    c.in(&a.mp_max_dist, max_dist, n); c.in(&a.mp_n, &n, 1);
    c.out(&a.mp_inview, inview, n); c.out(&a.proj_x, proj_x, n); c.out(&a.proj_y, proj_y, n); c.out(&a.proj_xr, proj_xr, n); c.out(&a.view_cos, view_cos, n);
    c.out(&a.level, level, n);
    a.cam = *cam; a.point_cap = n; a.viewing_cos_limit = viewing_cos_limit;
    if (int rc = c.upload()) return rc;
    if (int rc = sgs_frustum_batch_device(&a, 1, nullptr)) return rc;
    return c.download();
}

}  // extern "C"
