// fundamental.cu -- cv::findFundamentalMat(points1, points2, FM_RANSAC, 1.0, 0.99) as called by
// Frame::RmDynamicPointWithSemanticAndGeometry (src/Frame.cc:469-472), with the point selection in front of it (:454-468), for a
// batch of frames.  OpenCV's estimator (calib3d/fundam.cpp, ptsetreg.cpp) is a sequential loop (its result-defining rules are
// listed in DESIGN.md and pinned to cv2 by the parity tests).  Here the loop is re-cut for the GPU without changing its outcome:
//   * one block per frame; the frame's correspondences sit in shared memory;
//   * the sample indices of a ROUND of iterations are drawn ahead by one thread (the MWC generator and the redraw rules do not
//     depend on the models), one thread per iteration solves its 7-point problem, then the whole block counts the inliers of every
//     candidate model; a single thread finally replays the accept / update-niters decisions in iteration order, so the winner, the
//     adaptive stop and the tie-breaks are those of the sequential loop.  Iterations drawn past the stop are discarded.
//   * the 2-dimensional null space of the 7x9 system is the span OpenCV's JacobiSVD completion step produces: fixed pseudo-random
//     sign vectors projected off the row space.  The row space comes from a twice-applied modified Gram-Schmidt instead of the
//     Jacobi sweeps (same subspace, ~1e-15 relative difference in F).
// All arithmetic is FP64 with individually rounded products and sums (-fmad=false), errors are rounded to float before the
// threshold test like OpenCV's.  Fewer than 15 pairs take OpenCV's other branches in the same kernel: LMedS (8..14), plain 7-point (7), empty (< 7).
#include <cuda_runtime.h>

#include <cfloat>
#include <vector>

#include "host_call.h"
#include "sgs_common.h"

namespace sgs {

constexpr int kFmThreads = 256;
constexpr int kFmRound = 32;          // iterations per round (the first round draws kFmFirstRound)
constexpr int kFmFirstRound = 8;

struct FmRng {
    unsigned long long state;
    __device__ unsigned next() { state = (unsigned long long)(unsigned)state * 4164903690ULL + (unsigned)(state >> 32); return (unsigned)state; }
    __device__ int uniform(int a, int b) { return a == b ? a : (int)(next() % (unsigned)(b - a) + a); }
};

__device__ bool fm_collinear(const float2* m) {        // haveCollinearPoints: the 7th point against every pair of the first six
    const int i = 6;
    for (int j = 0; j < i; j++) {
        const double dx1 = (double)m[j].x - (double)m[i].x, dy1 = (double)m[j].y - (double)m[i].y;
        for (int k = 0; k < j; k++) {
            const double dx2 = (double)m[k].x - (double)m[i].x, dy2 = (double)m[k].y - (double)m[i].y;
            if (fabs(dx2 * dy1 - dy2 * dx1) <= (double)FLT_EPSILON * (fabs(dx1) + fabs(dy1) + fabs(dx2) + fabs(dy2))) return true;
        }
    }
    return false;
}

__device__ int fm_solve_cubic(const double* c, double* r) {      // cv::solveCubic
    double a0 = c[0], a1 = c[1], a2 = c[2], a3 = c[3];
    double x0 = 0, x1 = 0, x2 = 0;
    int n = 0;
    if (a0 == 0) {
        if (a1 == 0) {
            if (a2 == 0) n = a3 == 0 ? -1 : 0;
            else { x0 = -a3 / a2; n = 1; }
        } else {
            double d = a2 * a2 - 4 * a1 * a3;
            if (d >= 0) {
                d = sqrt(d);
                const double q1 = (-a2 + d) * 0.5, q2 = (a2 + d) * -0.5;
                if (fabs(q1) > fabs(q2)) { x0 = q1 / a1; x1 = a3 / q1; }
                else { x0 = q2 / a1; x1 = a3 / q2; }
                n = d > 0 ? 2 : 1;
            }
        }
    } else {
        a0 = 1. / a0; a1 *= a0; a2 *= a0; a3 *= a0;
        const double Q = (a1 * a1 - 3 * a2) * (1. / 9);
        const double R = (2 * a1 * a1 * a1 - 9 * a1 * a2 + 27 * a3) * (1. / 54);
        const double Qcubed = Q * Q * Q;
        double d = Qcubed - R * R;
        if (d > 0) {
            const double theta = acos(R / sqrt(Qcubed)), sqrtQ = sqrt(Q);
            const double t0 = -2 * sqrtQ, t1 = theta * (1. / 3), t2 = a1 * (1. / 3);
            x0 = t0 * cos(t1) - t2;
            x1 = t0 * cos(t1 + (2. * 3.14159265358979323846 / 3)) - t2;
            x2 = t0 * cos(t1 + (4. * 3.14159265358979323846 / 3)) - t2;
            n = 3;
        } else if (d == 0) {
            if (R >= 0) { x0 = -2 * pow(R, 1. / 3) - a1 / 3; x1 = pow(R, 1. / 3) - a1 / 3; }
            else { x0 = 2 * pow(-R, 1. / 3) - a1 / 3; x1 = -pow(-R, 1. / 3) - a1 / 3; }
            x2 = 0;
            n = x0 == x1 ? 1 : 2;
            x1 = x0 == x1 ? 0 : x1;
        } else {
            d = sqrt(-d);
            double e = pow(d + fabs(R), 1. / 3);
            if (R > 0) e = -e;
            x0 = (e + Q / e) - a1 * (1. / 3);
            n = 1;
        }
    }
    r[0] = x0; r[1] = x1; r[2] = x2;
    return n;
}

// run7Point on the sample (m1[i], m2[i]), i < 7.  Writes up to three row-major 3x3 models, returns their number.
__device__ int fm_run7point(const float2* m1, const float2* m2, double* Fout) {
    double c1x = 0, c1y = 0, c2x = 0, c2y = 0;
    for (int i = 0; i < 7; i++) { c1x += m1[i].x; c1y += m1[i].y; c2x += m2[i].x; c2y += m2[i].y; }
    const double t = 1. / 7;
    c1x *= t; c1y *= t; c2x *= t; c2y *= t;
    double s1 = 0, s2 = 0;
    for (int i = 0; i < 7; i++) {
        s1 += sqrt((m1[i].x - c1x) * (m1[i].x - c1x) + (m1[i].y - c1y) * (m1[i].y - c1y));
        s2 += sqrt((m2[i].x - c2x) * (m2[i].x - c2x) + (m2[i].y - c2y) * (m2[i].y - c2y));
    }
    s1 *= t; s2 *= t;
    if (s1 < (double)FLT_EPSILON || s2 < (double)FLT_EPSILON) return 0;
    s1 = sqrt(2.) / s1; s2 = sqrt(2.) / s2;
    double q[9][9];                 // rows 0..6: the system, orthonormalised in place; rows 7, 8: the null-space basis
    for (int i = 0; i < 7; i++) {
        const double x0 = (m1[i].x - c1x) * s1, y0 = (m1[i].y - c1y) * s1, x1 = (m2[i].x - c2x) * s2, y1 = (m2[i].y - c2y) * s2;
        double* r = q[i];
        r[0] = x1 * x0; r[1] = x1 * y0; r[2] = x1; r[3] = y1 * x0; r[4] = y1 * y0; r[5] = y1; r[6] = x0; r[7] = y0; r[8] = 1;
    }
    // orthonormal basis of the row space: modified Gram-Schmidt, every row orthogonalised twice
    for (int i = 0; i < 7; i++) {
        for (int pass = 0; pass < 2; pass++)
            for (int j = 0; j < i; j++) {
                double d = 0;
                for (int k = 0; k < 9; k++) d += q[i][k] * q[j][k];
                for (int k = 0; k < 9; k++) q[i][k] -= d * q[j][k];
            }
        double nn = 0;
        for (int k = 0; k < 9; k++) nn += q[i][k] * q[i][k];
        nn = nn > 0 ? 1. / sqrt(nn) : 0.;
        for (int k = 0; k < 9; k++) q[i][k] *= nn;
    }
    // JacobiSVD's completion of the two missing right singular vectors: RNG(0x12345678) sign vectors of magnitude 1/9, projected
    // off every previous row (two sweeps, rescaled to unit L1 norm after each projection), then normalised
    FmRng gen; gen.state = 0x12345678ULL;
    const double eps100 = DBL_EPSILON * 10 * 100;
    for (int i = 7; i < 9; i++) {
        for (int k = 0; k < 9; k++) q[i][k] = (gen.next() & 256) != 0 ? 1. / 9 : -(1. / 9);
        for (int pass = 0; pass < 2; pass++)
            for (int j = 0; j < i; j++) {
                double d = 0;
                for (int k = 0; k < 9; k++) d += q[i][k] * q[j][k];
                double asum = 0;
                for (int k = 0; k < 9; k++) { const double v = q[i][k] - d * q[j][k]; q[i][k] = v; asum += fabs(v); }
                asum = asum > eps100 ? 1 / asum : 0;
                for (int k = 0; k < 9; k++) q[i][k] *= asum;
            }
        double nn = 0;
        for (int k = 0; k < 9; k++) nn += q[i][k] * q[i][k];
        nn = sqrt(nn);
        const double s = nn > DBL_MIN ? 1 / nn : 0.;
        for (int k = 0; k < 9; k++) q[i][k] *= s;
    }
    double* f1 = q[7]; double* f2 = q[8];
    for (int i = 0; i < 9; i++) f1[i] -= f2[i];
    double c[4], r[3];
    double t0 = f2[4] * f2[8] - f2[5] * f2[7], t1 = f2[3] * f2[8] - f2[5] * f2[6], t2 = f2[3] * f2[7] - f2[4] * f2[6];
    c[3] = f2[0] * t0 - f2[1] * t1 + f2[2] * t2;
    c[2] = f1[0] * t0 - f1[1] * t1 + f1[2] * t2 - f1[3] * (f2[1] * f2[8] - f2[2] * f2[7]) + f1[4] * (f2[0] * f2[8] - f2[2] * f2[6]) -
           f1[5] * (f2[0] * f2[7] - f2[1] * f2[6]) + f1[6] * (f2[1] * f2[5] - f2[2] * f2[4]) - f1[7] * (f2[0] * f2[5] - f2[2] * f2[3]) +
           f1[8] * (f2[0] * f2[4] - f2[1] * f2[3]);
    t0 = f1[4] * f1[8] - f1[5] * f1[7]; t1 = f1[3] * f1[8] - f1[5] * f1[6]; t2 = f1[3] * f1[7] - f1[4] * f1[6];
    c[0] = f1[0] * t0 - f1[1] * t1 + f1[2] * t2;
    c[1] = f2[0] * t0 - f2[1] * t1 + f2[2] * t2 - f2[3] * (f1[1] * f1[8] - f1[2] * f1[7]) + f2[4] * (f1[0] * f1[8] - f1[2] * f1[6]) -
           f2[5] * (f1[0] * f1[7] - f1[1] * f1[6]) + f2[6] * (f1[1] * f1[5] - f1[2] * f1[4]) - f2[7] * (f1[0] * f1[5] - f1[2] * f1[3]) +
           f2[8] * (f1[0] * f1[4] - f1[1] * f1[3]);
    const int n = fm_solve_cubic(c, r);
    if (n < 1 || n > 3) return 0;
    for (int k = 0; k < n; k++) {
        double lambda = r[k], mu = 1.;
        const double s = f1[8] * r[k] + f2[8];
        double f0[9];
        if (fabs(s) > DBL_EPSILON) { mu = 1. / s; lambda *= mu; f0[8] = 1.; } else f0[8] = 0.;
        for (int i = 0; i < 8; i++) f0[i] = f1[i] * lambda + f2[i] * mu;
        // T2^T f0 T1,  T = [s 0 -s cx; 0 s -s cy; 0 0 1]; the general 3x3 products are kept so that zeros and ones round as they do on the CPU
        const double T1[9] = {s1, 0, -s1 * c1x, 0, s1, -s1 * c1y, 0, 0, 1}, T2[9] = {s2, 0, -s2 * c2x, 0, s2, -s2 * c2y, 0, 0, 1};
        double tmp[9], out[9];
        for (int i = 0; i < 3; i++)
            for (int j = 0; j < 3; j++) { double v = 0; for (int p = 0; p < 3; p++) v += T2[p * 3 + i] * f0[p * 3 + j]; tmp[i * 3 + j] = v; }
        for (int i = 0; i < 3; i++)
            for (int j = 0; j < 3; j++) { double v = 0; for (int p = 0; p < 3; p++) v += tmp[i * 3 + p] * T1[p * 3 + j]; out[i * 3 + j] = v; }
        if (fabs(out[8]) > DBL_EPSILON) { const double sc = 1. / out[8]; for (int i = 0; i < 9; i++) out[i] *= sc; }
        for (int i = 0; i < 9; i++) Fout[9 * k + i] = out[i];
    }
    return n;
}

__device__ __forceinline__ bool fm_inlier(const float4 p, const double* F, float t) {      // FMEstimatorCallback::computeError + findInliers
    const double x1 = p.x, y1 = p.y, x2 = p.z, y2 = p.w;
    double a = F[0] * x1 + F[1] * y1 + F[2], b = F[3] * x1 + F[4] * y1 + F[5], c = F[6] * x1 + F[7] * y1 + F[8];
    const double s2 = 1. / (a * a + b * b), d2 = x2 * a + y2 * b + c;
    a = F[0] * x2 + F[3] * y2 + F[6]; b = F[1] * x2 + F[4] * y2 + F[7]; c = F[2] * x2 + F[5] * y2 + F[8];
    const double s1 = 1. / (a * a + b * b), d1 = x1 * a + y1 * b + c;
    const float err = (float)fmax(d1 * d1 * s1, d2 * d2 * s2);
    return err <= t;
}
__device__ __forceinline__ float fm_error(const float4 p, const double* F) {                  // FMEstimatorCallback::computeError, one pair
    const double x1 = p.x, y1 = p.y, x2 = p.z, y2 = p.w;
    double a = F[0] * x1 + F[1] * y1 + F[2], b = F[3] * x1 + F[4] * y1 + F[5], c = F[6] * x1 + F[7] * y1 + F[8];
    const double s2 = 1. / (a * a + b * b), d2 = x2 * a + y2 * b + c;
    a = F[0] * x2 + F[3] * y2 + F[6]; b = F[1] * x2 + F[4] * y2 + F[7]; c = F[2] * x2 + F[5] * y2 + F[8];
    const double s1 = 1. / (a * a + b * b), d1 = x1 * a + y1 * b + c;
    return (float)fmax(d1 * d1 * s1, d2 * d2 * s2);
}

// RANSACPointSetRegistrator / LMeDSPointSetRegistrator::getSubset for `want` consecutive iterations (sequential RNG state: one thread).
// Returns the number of samples drawn; *ok = 0 when a draw failed (10000 attempts without a non-collinear sample): the estimator's loop ends there.
__device__ int fm_draw_samples(FmRng& rng, const float4* pts, int n, int want, int (*idx_out)[7], int* ok) {
    int got = 0;
    *ok = 1;
    for (; got < want; ++got) {
        bool found = false;
        for (int attempt = 0; attempt < 10000 && !found; ++attempt) {
            float2 a[7], b[7];
            int* idx = idx_out[got];
            for (int i = 0; i < 7; ++i) {
                int v;
                for (;;) {
                    v = rng.uniform(0, n);
                    bool dup = false;
                    for (int j = 0; j < i; ++j) dup |= idx[j] == v;
                    if (!dup) break;
                }
                idx[i] = v;
                const float4 p = pts[v];
                a[i] = make_float2(p.x, p.y); b[i] = make_float2(p.z, p.w);
            }
            found = !fm_collinear(a) && !fm_collinear(b);
        }
        if (!found) { *ok = 0; break; }
    }
    return got;
}

__device__ int fm_update_iters(double p, double ep, int max_iters) {     // RANSACUpdateNumIters, modelPoints = 7
    p = fmin(fmax(p, 0.), 1.); ep = fmin(fmax(ep, 0.), 1.);
    double num = fmax(1. - p, DBL_MIN), denom = 1. - pow(1. - ep, 7.);
    if (denom < DBL_MIN) return 0;
    num = log(num); denom = log(denom);
    return denom >= 0 || -num >= max_iters * (-denom) ? max_iters : (int)rint(num / denom);
}

// cur points come from keypoints (kps != nullptr) or a float2 array; prev from a float2 array.
// info[f] = {pairs used, inliers of the returned model, iterations run, status (0 ok, 1 fewer than 7 pairs, 2 no model, 3 no previous frame)}
// 7 pairs: the 7-point solver directly; 8..14 pairs: LMedS; 15 and more: RANSAC -- the three branches of cv::findFundamentalMat(FM_RANSAC).
__global__ void __launch_bounds__(kFmThreads) fm_ransac_kernel(const sgs_keypoint* __restrict__ kps, const float2* __restrict__ cur_xy,
                                                               const float2* __restrict__ prev_xy, const int32_t* __restrict__ counts, int cap,
                                                               const sgs_rect* __restrict__ prev_boxes, const int32_t* __restrict__ prev_nboxes,
                                                               const uint8_t* __restrict__ prev_have_dyn, int max_boxes,
                                                               const int32_t* __restrict__ prev_index, double thresh,
                                                               double confidence, int max_iters, double* __restrict__ F_out,
                                                               int32_t* __restrict__ info, uint8_t* __restrict__ mask_out) {
    extern __shared__ float4 s_pts[];                  // [cap] (x1, y1, x2, y2), the pairs handed to the estimator, in order
    __shared__ double s_models[kFmRound * 3][9];
    __shared__ int s_nmodels[kFmRound], s_good[kFmRound * 3], s_idx[kFmRound][7];
    __shared__ double s_best[9];
    __shared__ int s_warp[kFmThreads / 32];
    __shared__ int s_n, s_niters, s_done, s_round, s_maxgood, s_carry, s_drawn_ok;
    __shared__ unsigned long long s_rng;
    const int f = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n_all = counts ? min(counts[f], cap) : cap;
    const float2* prev = prev_xy + (int64_t)f * cap;
    auto cur_pt = [&](int i) -> float2 {
        if (kps) { const sgs_keypoint k = kps[(int64_t)f * cap + i]; return make_float2(k.x, k.y); }
        return cur_xy[(int64_t)f * cap + i];
    };
    // ---- selection (src/Frame.cc:454-472): ordered compaction of the pairs whose previous point is outside the previous boxes
    // prev_index (may be NULL): the batch row holding the previous frame's boxes; prev_index[f] == f marks a frame without a previous one
    const int fb = prev_index ? prev_index[f] : f;
    const bool no_prev = prev_index && fb == f;
    // The reference keeps "the previous frame had potential dynamic objects" at file scope and writes it only inside the rejection (src/Frame.cc:482-491), which
    // the first frame of a stream never runs (:154-162): the detections of a stream's first frame do not filter the pairs of its second frame (quirk Q13,
    // pinned by tests/test_frame_ref.py against the reference's own Frame.cc).  With prev_index the rows say which frames are first ones.
    const bool pre_dyn = prev_have_dyn && prev_have_dyn[fb] != 0 && !(prev_index && prev_index[fb] == fb);
    if (tid == 0) s_carry = 0;
    __syncthreads();
    if (pre_dyn && !no_prev) {
        const sgs_rect* boxes = prev_boxes + (int64_t)fb * max_boxes;
        const int nb = min(prev_nboxes[fb], max_boxes);
        for (int base = 0; base < n_all; base += kFmThreads) {
            const int i = base + tid;
            bool keep = false;
            float2 c = make_float2(0.f, 0.f), p = c;
            if (i < n_all) {
                p = prev[i]; c = cur_pt(i);
                keep = true;
                for (int b = 0; b < nb; ++b) {
                    const sgs_rect r = boxes[b];
                    if (p.x > r.x && p.x < __fadd_rn(r.x, r.w) && p.y > r.y && p.y < __fadd_rn(r.y, r.h)) { keep = false; break; }
                }
            }
            const unsigned bal = __ballot_sync(0xffffffffu, keep);
            if (lane == 0) s_warp[warp] = __popc(bal);
            __syncthreads();
            int off = s_carry;
            for (int w = 0; w < warp; ++w) off += s_warp[w];
            if (keep) s_pts[off + __popc(bal & ((1u << lane) - 1u))] = make_float4(c.x, c.y, p.x, p.y);
            __syncthreads();
            if (tid == 0) { int tot = 0; for (int w = 0; w < kFmThreads / 32; ++w) tot += s_warp[w]; s_carry += tot; }
            __syncthreads();
        }
    }
    int n = s_carry;
    if (!(pre_dyn && n > 20)) {
        __syncthreads();
        for (int i = tid; i < n_all; i += kFmThreads) { const float2 c = cur_pt(i), p = prev[i]; s_pts[i] = make_float4(c.x, c.y, p.x, p.y); }
        n = n_all;
    }
    __syncthreads();
    double* Fo = F_out + (int64_t)f * 9;
    int32_t* inf = info ? info + (int64_t)f * 4 : nullptr;
    if (thresh <= 0) thresh = 3;
    if (confidence < DBL_EPSILON || confidence > 1 - DBL_EPSILON) confidence = 0.99;
    const double kNaN = __longlong_as_double(0x7ff8000000000000LL);
    if (n < 7 || no_prev) {           // cv::findFundamentalMat returns an empty matrix below 7 pairs (fundam.cpp): "empty F" = NaN here
        if (tid < 9) Fo[tid] = kNaN;
        if (tid == 0 && inf) { inf[0] = n; inf[1] = 0; inf[2] = 0; inf[3] = no_prev ? 3 : 1; }
        if (mask_out) for (int i = tid; i < n_all; i += kFmThreads) mask_out[(int64_t)f * cap + i] = 0;
        return;
    }
    if (n == 7) {                     // exactly 7 pairs: the 7-point solver itself, up to three stacked solutions; the reference reads rows 0..2 = the first
        if (tid == 0) {
            float2 a[7], b[7];
            for (int i = 0; i < 7; ++i) { const float4 p = s_pts[i]; a[i] = make_float2(p.x, p.y); b[i] = make_float2(p.z, p.w); }
            double Fm[27];
            const int nm = fm_run7point(a, b, Fm);
            for (int i = 0; i < 9; ++i) Fo[i] = nm > 0 ? Fm[i] : kNaN;
            if (inf) { inf[0] = n; inf[1] = nm > 0 ? 7 : 0; inf[2] = 1; inf[3] = nm > 0 ? 0 : 2; }
        }
        if (mask_out) for (int i = tid; i < n_all; i += kFmThreads) mask_out[(int64_t)f * cap + i] = i < n ? 1 : 0;      // OpenCV sets the whole mask
        return;
    }
    if (n < 15) {
        // 8..14 pairs: cv::findFundamentalMat switches to LMeDSPointSetRegistrator(cb, 7, confidence) (fundam.cpp; ptsetreg.cpp): a FIXED number of
        // samples (outlier ratio 0.45, at most 1000), the model with the smallest median error (element n/2 of the sorted errors, strict '<'),
        // inliers within sigma = 2.5 * 1.4826 * (1 + 5 / (n - 7)) * sqrt(median) (at least 0.001); fewer than 7 inliers -> empty matrix.
        __shared__ float s_med[kFmRound * 3];
        __shared__ double s_minmed;
        __shared__ int s_lm_good;
        const int niters = max(fm_update_iters(confidence, 0.45, 1000), 3);
        if (tid == 0) { s_done = 0; s_rng = 0xffffffffffffffffULL; s_minmed = DBL_MAX; s_drawn_ok = 1; s_lm_good = 0; }
        __syncthreads();
        while (true) {
            if (tid == 0) {
                FmRng rng; rng.state = s_rng;
                int okd = 1;
                s_round = fm_draw_samples(rng, s_pts, n, min(kFmRound, niters - s_done), s_idx, &okd);
                if (!okd) s_drawn_ok = 0;
                s_rng = rng.state;
            }
            __syncthreads();
            const int round = s_round;
            if (tid < round) {
                float2 a[7], b[7];
                for (int i = 0; i < 7; ++i) { const float4 p = s_pts[s_idx[tid][i]]; a[i] = make_float2(p.x, p.y); b[i] = make_float2(p.z, p.w); }
                double Fm[27];
                const int nm = fm_run7point(a, b, Fm);
                s_nmodels[tid] = nm;
                for (int k = 0; k < nm; ++k) {
                    float e[14];
                    for (int i = 0; i < n; ++i) {                              // insertion sort of the n <= 14 errors
                        const float v = fm_error(s_pts[i], Fm + 9 * k);
                        int j = i;
                        for (; j > 0 && e[j - 1] > v; --j) e[j] = e[j - 1];
                        e[j] = v;
                    }
                    s_med[tid * 3 + k] = e[n / 2];
                    for (int i = 0; i < 9; ++i) s_models[tid * 3 + k][i] = Fm[9 * k + i];
                }
            }
            __syncthreads();
            if (tid == 0) {                                                    // sequential replay: strict improvement, iteration order, model order
                double mm = s_minmed;
                for (int it = 0; it < round; ++it)
                    for (int k = 0; k < s_nmodels[it]; ++k) {
                        const double med = (double)s_med[it * 3 + k];
                        if (med < mm) { mm = med; for (int i = 0; i < 9; ++i) s_best[i] = s_models[it * 3 + k][i]; }
                    }
                s_minmed = mm; s_done += round;
            }
            __syncthreads();
            if (s_done >= niters || !s_drawn_ok) break;
            __syncthreads();
        }
        bool ok = s_minmed < DBL_MAX;
        float tl = 0.f;
        if (ok) {
            double sigma = 2.5 * 1.4826 * (1 + 5. / (n - 7)) * sqrt(s_minmed);
            sigma = fmax(sigma, 0.001);
            tl = (float)(sigma * sigma);
            if (tid < n && fm_inlier(s_pts[tid], s_best, tl)) atomicAdd(&s_lm_good, 1);
        }
        __syncthreads();
        const int good = s_lm_good;
        ok = ok && good >= 7;
        if (tid < 9) Fo[tid] = ok ? s_best[tid] : kNaN;
        if (tid == 0 && inf) { inf[0] = n; inf[1] = good; inf[2] = s_done; inf[3] = ok ? 0 : 2; }
        if (mask_out) for (int i = tid; i < n_all; i += kFmThreads) mask_out[(int64_t)f * cap + i] = (ok && i < n && fm_inlier(s_pts[i], s_best, tl)) ? 1 : 0;
        return;
    }
    if (thresh <= 0) thresh = 3;
    if (confidence < DBL_EPSILON || confidence > 1 - DBL_EPSILON) confidence = 0.99;
    const float t = (float)(thresh * thresh);
    if (tid == 0) { s_n = n; s_niters = max(max_iters, 1); s_done = 0; s_maxgood = 0; s_rng = 0xffffffffffffffffULL; s_drawn_ok = 1; }
    __syncthreads();
    bool first = true;
    while (true) {
        // ---- draw the samples of this round (sequential state: one thread)
        if (tid == 0) {
            FmRng rng; rng.state = s_rng;
            const int want = min(first ? kFmFirstRound : kFmRound, s_niters - s_done);
            int okd = 1;
            const int got = fm_draw_samples(rng, s_pts, n, want, s_idx, &okd);      // a failed draw ends the loop (or fails it when it is the first iteration)
            if (!okd) s_drawn_ok = 0;
            s_round = got;
            s_rng = rng.state;
        }
        __syncthreads();
        const int round = s_round;
        // ---- one thread per iteration: the 7-point models
        if (tid < round) {
            float2 a[7], b[7];
            for (int i = 0; i < 7; ++i) { const float4 p = s_pts[s_idx[tid][i]]; a[i] = make_float2(p.x, p.y); b[i] = make_float2(p.z, p.w); }
            double Fm[27];
            const int nm = fm_run7point(a, b, Fm);
            s_nmodels[tid] = nm;
            for (int k = 0; k < nm; ++k)
                for (int i = 0; i < 9; ++i) s_models[tid * 3 + k][i] = Fm[9 * k + i];
        }
        if (tid < kFmRound * 3) s_good[tid] = 0;
        __syncthreads();
        // ---- inlier counts of every candidate model: the block sweeps the points once per model
        for (int it = 0; it < round; ++it) {
            const int nm = s_nmodels[it];
            for (int k = 0; k < nm; ++k) {
                const double* Fm = s_models[it * 3 + k];
                int cnt = 0;
                for (int i = tid; i < n; i += kFmThreads) cnt += fm_inlier(s_pts[i], Fm, t) ? 1 : 0;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
                if (lane == 0 && cnt) atomicAdd(&s_good[it * 3 + k], cnt);
            }
        }
        __syncthreads();
        // ---- replay the sequential accept / update decisions in iteration order
        if (tid == 0) {
            int done = s_done, niters = s_niters, maxgood = s_maxgood;
            for (int it = 0; it < round && done < niters; ++it, ++done) {
                for (int k = 0; k < s_nmodels[it]; ++k) {
                    const int good = s_good[it * 3 + k];
                    if (good > max(maxgood, 6)) {
                        for (int i = 0; i < 9; ++i) s_best[i] = s_models[it * 3 + k][i];
                        maxgood = good;
                        niters = fm_update_iters(confidence, (double)(n - good) / n, niters);
                    }
                }
            }
            s_done = done; s_niters = niters; s_maxgood = maxgood;
        }
        __syncthreads();
        first = false;
        if (s_done >= s_niters || !s_drawn_ok) break;
        __syncthreads();
    }
    const bool ok = s_maxgood > 0;
    if (tid < 9) Fo[tid] = ok ? s_best[tid] : __longlong_as_double(0x7ff8000000000000LL);
    if (tid == 0 && inf) { inf[0] = n; inf[1] = s_maxgood; inf[2] = s_done; inf[3] = ok ? 0 : 2; }
    if (mask_out) {         // mask of the returned model over the pairs used (positions >= n are cleared)
        for (int i = tid; i < n_all; i += kFmThreads)
            mask_out[(int64_t)f * cap + i] = (ok && i < n && fm_inlier(s_pts[i], s_best, t)) ? 1 : 0;
    }
}

int fm_launch(const sgs_keypoint* d_kps, const float2* d_cur, const float2* d_prev, const int32_t* d_counts, int cap, int nframes,
              const sgs_rect* d_boxes, const int32_t* d_nboxes, const uint8_t* d_have_dyn, int max_boxes, const int32_t* d_prev_index, double thresh,
              double confidence, int max_iters, double* d_F, int32_t* d_info, uint8_t* d_mask, cudaStream_t st) {
    const size_t smem = (size_t)cap * sizeof(float4);
    if (smem > 200 * 1024) { set_error("fundamental: %d pairs per frame do not fit shared memory", cap); return SGS_ERR_UNSUPPORTED; }
    if (smem > 40 * 1024)      // per device and cheap: set whenever the default 48 KB would not do
        SGS_CUDA_TRY(cudaFuncSetAttribute(fm_ransac_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    fm_ransac_kernel<<<nframes, kFmThreads, smem, st>>>(d_kps, d_cur, d_prev, d_counts, cap, d_boxes, d_nboxes, d_have_dyn, max_boxes, d_prev_index,
                                                        thresh, confidence, max_iters, d_F, d_info, d_mask);
    SGS_CUDA_TRY(cudaGetLastError());
    return SGS_OK;
}

}  // namespace sgs

using namespace sgs;

extern "C" {

SGS_API int sgs_fundamental_batch_device(const sgs_keypoint* d_kps, const float* d_prev_xy, const int32_t* d_counts, int cap, int nframes,
                                         const sgs_rect* d_prev_boxes, const int32_t* d_prev_nboxes, const uint8_t* d_prev_have_dyn, int max_boxes,
                                         const int32_t* d_prev_index, double ransac_thresh, double confidence, int max_iters, double* d_F, int32_t* d_info, void* stream) {
    if (!d_kps || !d_prev_xy || !d_counts || !d_F || cap < 1 || nframes < 1) { set_error("sgs_fundamental_batch_device: bad argument"); return SGS_ERR_INVALID; }
    if (d_prev_have_dyn && (!d_prev_boxes || !d_prev_nboxes || max_boxes < 1)) { set_error("sgs_fundamental_batch_device: boxes missing"); return SGS_ERR_INVALID; }
    return fm_launch(d_kps, nullptr, reinterpret_cast<const float2*>(d_prev_xy), d_counts, cap, nframes, d_prev_boxes, d_prev_nboxes, d_prev_have_dyn,
                     max_boxes, d_prev_index, ransac_thresh, confidence, max_iters, d_F, d_info, nullptr, (cudaStream_t)stream);
}

SGS_API int sgs_fundamental_ransac(const float* pts1_xy, const float* pts2_xy, int n, double ransac_thresh, double confidence, int max_iters,
                                   double* F, uint8_t* mask, int32_t* info, int device) {
    if (!pts1_xy || !pts2_xy || !F || n < 1) { set_error("sgs_fundamental_ransac: bad argument"); return SGS_ERR_INVALID; }
    SGS_CUDA_TRY(cudaSetDevice(device));
    HostCall c("sgs_fundamental_ransac");
    const float2 *d_a, *d_b; double* d_F; int32_t* d_info; uint8_t* d_mask;
    c.in(&d_a, pts1_xy, n); c.in(&d_b, pts2_xy, n); c.out(&d_F, F, 9); c.out(&d_mask, mask, n); c.out(&d_info, info, 4);
    if (int rc = c.upload()) return rc;
    if (int rc = fm_launch(nullptr, d_a, d_b, nullptr, n, 1, nullptr, nullptr, nullptr, 0, nullptr, ransac_thresh, confidence, max_iters, d_F, d_info, d_mask, nullptr))
        return rc;
    return c.download();
}

}  // extern "C"
