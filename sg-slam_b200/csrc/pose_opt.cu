// pose_opt.cu -- Optimizer::PoseOptimization(Frame*) (src/Optimizer.cc:239-451): the motion-only bundle adjustment run after every matcher call of
// the tracking thread (Tracking::TrackWithMotionModel :933, TrackReferenceKeyFrame :880, TrackLocalMap :1314), for a batch of frames.
// The reference drives g2o (Levenberg-Marquardt on one SE3 vertex with unary reprojection edges).  What decides the result is restated in FP64:
//   four rounds of ten LM iterations, each round restarting from the INITIAL pose with the edges that passed the previous round's chi-square test
//   (5.991 mono / 7.815 stereo, compared in float), Huber kernels for the first three rounds, g2o's lambda / rho / trial rules and its habit of
//   leaving the error vectors of a rejected trial in the edges (they are what the classification reads).  File:line references are in the
//   CPU restatement the parity tests use; the reference's own code could not be executed here (Eigen is absent), so this stage is checked against
//   that restatement and against first-order optimality, not against g2o output.
// One block per frame: the threads share the edges, the 6x6 normal equations are reduced across the block, one thread factorises and updates the
// pose.  Sums are reduced in a fixed tree order (deterministic), not in the edge order of g2o: poses agree to ~1e-12, not bit for bit.
#include <cuda_runtime.h>

#include <cfloat>

#include "host_call.h"
#include "sgs_common.h"

namespace sgs {

constexpr int kPoThreads = 128;

struct PoQuat { double x, y, z, w; };
struct PoSE3 { PoQuat r; double t[3]; };

__device__ PoQuat po_quat_from_matrix(const double* R) {      // Eigen::Quaterniond(Matrix3d)
    PoQuat q;
    double t = R[0] + R[4] + R[8];
    if (t > 0) {
        t = sqrt(t + 1.0);
        q.w = 0.5 * t; t = 0.5 / t;
        q.x = (R[7] - R[5]) * t; q.y = (R[2] - R[6]) * t; q.z = (R[3] - R[1]) * t;
    } else {
        int i = 0;
        if (R[4] > R[0]) i = 1;
        if (R[8] > R[3 * i + i]) i = 2;
        const int j = (i + 1) % 3, k = (j + 1) % 3;
        t = sqrt(R[3 * i + i] - R[3 * j + j] - R[3 * k + k] + 1.0);
        double c[3];
        c[i] = 0.5 * t; t = 0.5 / t;
        q.w = (R[3 * k + j] - R[3 * j + k]) * t;
        c[j] = (R[3 * j + i] + R[3 * i + j]) * t; c[k] = (R[3 * k + i] + R[3 * i + k]) * t;
        q.x = c[0]; q.y = c[1]; q.z = c[2];
    }
    return q;
}

__device__ void po_normalize(PoQuat& q) {
    if (q.w < 0) { q.x = -q.x; q.y = -q.y; q.z = -q.z; q.w = -q.w; }
    const double n = sqrt(q.x * q.x + q.y * q.y + q.z * q.z + q.w * q.w);
    q.x /= n; q.y /= n; q.z /= n; q.w /= n;
}

__device__ PoQuat po_mul(const PoQuat& a, const PoQuat& b) {
    PoQuat r;
    r.w = a.w * b.w - a.x * b.x - a.y * b.y - a.z * b.z;
    r.x = a.w * b.x + a.x * b.w + a.y * b.z - a.z * b.y;
    r.y = a.w * b.y + a.y * b.w + a.z * b.x - a.x * b.z;
    r.z = a.w * b.z + a.z * b.w + a.x * b.y - a.y * b.x;
    return r;
}

__device__ __forceinline__ void po_rotate(const PoQuat& q, const double* v, double* out) {      // Eigen _transformVector
    double uv0 = q.y * v[2] - q.z * v[1], uv1 = q.z * v[0] - q.x * v[2], uv2 = q.x * v[1] - q.y * v[0];
    uv0 += uv0; uv1 += uv1; uv2 += uv2;
    out[0] = v[0] + q.w * uv0 + (q.y * uv2 - q.z * uv1);
    out[1] = v[1] + q.w * uv1 + (q.z * uv0 - q.x * uv2);
    out[2] = v[2] + q.w * uv2 + (q.x * uv1 - q.y * uv0);
}

__device__ PoSE3 po_exp(const double* u) {                      // SE3Quat::exp
    const double om[3] = {u[0], u[1], u[2]}, up[3] = {u[3], u[4], u[5]};
    const double theta = sqrt(om[0] * om[0] + om[1] * om[1] + om[2] * om[2]);
    const double O[9] = {0, -om[2], om[1], om[2], 0, -om[0], -om[1], om[0], 0};
    double O2[9];
    for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) { double v = 0; for (int k = 0; k < 3; k++) v += O[3 * i + k] * O[3 * k + j]; O2[3 * i + j] = v; }
    double R[9], V[9];
    if (theta < 0.00001) {
        for (int i = 0; i < 9; i++) { R[i] = (i % 4 == 0 ? 1.0 : 0.0) + O[i] + O2[i]; V[i] = R[i]; }
    } else {
        const double a = sin(theta) / theta, b = (1 - cos(theta)) / (theta * theta), c = (theta - sin(theta)) / pow(theta, 3.0);
        for (int i = 0; i < 9; i++) { const double I = i % 4 == 0 ? 1.0 : 0.0; R[i] = I + a * O[i] + b * O2[i]; V[i] = I + b * O[i] + c * O2[i]; }
    }
    PoSE3 s;
    for (int i = 0; i < 3; i++) s.t[i] = V[3 * i] * up[0] + V[3 * i + 1] * up[1] + V[3 * i + 2] * up[2];
    s.r = po_quat_from_matrix(R); po_normalize(s.r);
    return s;
}

__device__ bool po_ldlt6(const double* Hin, const double* b, double* x) {
    double L[36], D[6], y[6];
    for (int i = 0; i < 36; i++) L[i] = 0;
    for (int j = 0; j < 6; j++) {
        double d = Hin[6 * j + j];
        for (int k = 0; k < j; k++) d -= L[6 * j + k] * L[6 * j + k] * D[k];
        if (!(d > 0)) return false;
        D[j] = d; L[6 * j + j] = 1;
        for (int i = j + 1; i < 6; i++) {
            double v = Hin[6 * i + j];
            for (int k = 0; k < j; k++) v -= L[6 * i + k] * L[6 * j + k] * D[k];
            L[6 * i + j] = v / d;
        }
    }
    for (int i = 0; i < 6; i++) { double v = b[i]; for (int k = 0; k < i; k++) v -= L[6 * i + k] * y[k]; y[i] = v; }
    for (int i = 0; i < 6; i++) y[i] /= D[i];
    for (int i = 5; i >= 0; i--) { double v = y[i]; for (int k = i + 1; k < 6; k++) v -= L[6 * k + i] * x[k]; x[i] = v; }
    return true;
}

struct PoArgs {
    float fx, fy, cx, cy, bf;
    const float* tcw_in; const sgs_keypoint* kps; const float* uright; const int32_t* n; int cap;
    const uint8_t* has_mp; const int32_t* mp_index; const float* points_xyz; int point_cap;
    const float* points2_xyz; int id_base2, point2_cap;      // optional second point array (local-map points of the chained call)
    float inv_sigma2[16];
    float* tcw_out; uint8_t* outlier; int32_t* ninliers;
    double* err;          // scratch [F][cap][3]: the error vector each edge carries between evaluations
    uint8_t* level;       // scratch [F][cap]: 1 = excluded from the next round (the edge's g2o level)
};

// sum of `v` over the block, result in every thread (fixed tree order: deterministic)
__device__ double po_block_sum(double v, double* s_red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
    __syncthreads();
    double t = 0;
#pragma unroll
    for (int w = 0; w < kPoThreads / 32; ++w) t += s_red[w];
    return t;
}

__global__ void __launch_bounds__(kPoThreads) pose_opt_kernel(const PoArgs A) {
    __shared__ PoSE3 s_est;
    __shared__ double s_red[kPoThreads / 32];
    __shared__ double s_sys[28];          // 21 upper-triangular entries of H, 6 of b, robust chi2
    __shared__ double s_x[6];
    __shared__ int s_ok2;
    const int f = blockIdx.x, tid = threadIdx.x;
    const int n = min(A.n[f], A.cap);
    const int64_t ko = (int64_t)f * A.cap;
    const double fx = A.fx, fy = A.fy, cx = A.cx, cy = A.cy, bf = A.bf;
    const float deltaMono = (float)sqrt(5.991), deltaStereo = (float)sqrt(7.815);

    auto has = [&](int i) -> bool { return A.mp_index ? A.mp_index[ko + i] >= 0 : A.has_mp[ko + i] != 0; };
    auto world = [&](int i, double* X) {
        const int id = A.mp_index ? A.mp_index[ko + i] : i;
        const float* p = (A.points2_xyz && id >= A.id_base2) ? A.points2_xyz + 3 * ((int64_t)f * A.point2_cap + (id - A.id_base2)) : A.points_xyz + 3 * ((int64_t)f * A.point_cap + id);
        X[0] = p[0]; X[1] = p[1]; X[2] = p[2];
    };
    // edge error at the current estimate (EdgeSE3ProjectXYZOnlyPose / EdgeStereoSE3ProjectXYZOnlyPose::computeError)
    auto edge_error = [&](int i, const PoSE3& est, double* e, double* pc) -> bool {
        double X[3]; world(i, X);
        po_rotate(est.r, X, pc);
        pc[0] += est.t[0]; pc[1] += est.t[1]; pc[2] += est.t[2];
        const sgs_keypoint k = A.kps[ko + i];
        const float ur = A.uright[ko + i];
        const bool stereo = !(ur < 0);
        if (!stereo) {
            e[0] = (double)k.x - (pc[0] / pc[2] * fx + cx); e[1] = (double)k.y - (pc[1] / pc[2] * fy + cy); e[2] = 0;
        } else {
            const float invz = (float)(1.0 / pc[2]);       // const float invz = 1.0f / trans_xyz[2]: double division, float result
            const double r0 = pc[0] * invz * fx + cx, r1 = pc[1] * invz * fy + cy, r2 = r0 - bf * invz;
            e[0] = (double)k.x - r0; e[1] = (double)k.y - r1; e[2] = (double)ur - r2;
        }
        return stereo;
    };

    int n_initial = 0;
    for (int i = tid; i < n; i += kPoThreads) {
        const bool h = has(i);
        n_initial += h ? 1 : 0;
        A.level[ko + i] = 0;
        if (h) A.outlier[ko + i] = 0;
    }
    n_initial = (int)po_block_sum((double)n_initial, s_red);
    if (tid < 16) A.tcw_out[16 * (int64_t)f + tid] = A.tcw_in[16 * (int64_t)f + tid];
    if (n_initial < 3) { if (tid == 0) A.ninliers[f] = 0; return; }

    int n_bad = 0;
    for (int it = 0; it < 4; ++it) {
        const bool robust = it < 3;
        if (tid == 0) {      // vSE3->setEstimate(Converter::toSE3Quat(pFrame->mTcw))
            const float* T = A.tcw_in + 16 * (int64_t)f;
            double R[9];
            for (int r = 0; r < 3; r++) { for (int c = 0; c < 3; c++) R[3 * r + c] = T[4 * r + c]; s_est.t[r] = T[4 * r + 3]; }
            s_est.r = po_quat_from_matrix(R); po_normalize(s_est.r);
        }
        __syncthreads();
        // evaluation at s_est: errors of the active edges (kept in A.err), robust chi2, optionally the normal equations
        auto evaluate = [&](bool with_system) {
            double acc[28];
#pragma unroll
            for (int q = 0; q < 28; ++q) acc[q] = 0;
            const PoSE3 est = s_est;
            for (int i = tid; i < n; i += kPoThreads) {
                if (!has(i) || A.level[ko + i]) continue;
                double e[3], pc[3];
                const bool stereo = edge_error(i, est, e, pc);
                double* E = A.err + 3 * (ko + i);
                E[0] = e[0]; E[1] = e[1]; E[2] = e[2];
                const double info = A.inv_sigma2[A.kps[ko + i].octave];
                const double c = (e[0] * e[0] + e[1] * e[1] + (stereo ? e[2] * e[2] : 0.0)) * info;
                const double delta = stereo ? deltaStereo : deltaMono, dsqr = delta * delta;
                double w = 1.0;
                if (robust) { if (c <= dsqr) acc[27] += c; else { const double sq = sqrt(c); acc[27] += 2 * sq * delta - dsqr; w = delta / sq; } }
                else acc[27] += c;
                if (with_system) {
                    const double x = pc[0], y = pc[1], invz = 1.0 / pc[2], invz_2 = invz * invz;
                    double J[3][6];
                    J[0][0] = x * y * invz_2 * fx; J[0][1] = -(1 + (x * x * invz_2)) * fx; J[0][2] = y * invz * fx; J[0][3] = -invz * fx; J[0][4] = 0; J[0][5] = x * invz_2 * fx;
                    J[1][0] = (1 + y * y * invz_2) * fy; J[1][1] = -x * y * invz_2 * fy; J[1][2] = -x * invz * fy; J[1][3] = 0; J[1][4] = -invz * fy; J[1][5] = y * invz_2 * fy;
                    J[2][0] = J[0][0] - bf * y * invz_2; J[2][1] = J[0][1] + bf * x * invz_2; J[2][2] = J[0][2]; J[2][3] = J[0][3]; J[2][4] = 0; J[2][5] = J[0][5] - bf * invz_2;
                    const int D = stereo ? 3 : 2;
                    int q = 0;
#pragma unroll
                    for (int r = 0; r < 6; ++r) {
                        double sb = 0;
                        for (int d = 0; d < D; ++d) sb += J[d][r] * info * e[d];
                        acc[21 + r] -= w * sb;
#pragma unroll
                        for (int cc = r; cc < 6; ++cc) { double h = 0; for (int d = 0; d < D; ++d) h += J[d][r] * (w * info) * J[d][cc]; acc[q++] += h; }
                    }
                }
            }
            for (int q = with_system ? 0 : 27; q < 28; ++q) {
                const double tot = po_block_sum(acc[q], s_red);
                if (tid == 0) s_sys[q] = tot;
            }
            __syncthreads();
        };
        // number of active edges (initializeOptimization(0)): nothing to optimise when there is none
        int n_active = 0;
        for (int i = tid; i < n; i += kPoThreads) n_active += (has(i) && !A.level[ko + i]) ? 1 : 0;
        n_active = (int)po_block_sum((double)n_active, s_red);
        if (n_active > 0) {
            double lambda = 0, ni = 2; int nbad_lm = 0;
            for (int i = 0; i < 10; ++i) {                       // SparseOptimizer::optimize(10)
                evaluate(true);
                double currentChi = s_sys[27];
                const double iniChi = currentChi;
                double H[36], b[6];
                { int q = 0; for (int r = 0; r < 6; ++r) for (int c = r; c < 6; ++c) { H[6 * r + c] = s_sys[q]; H[6 * c + r] = s_sys[q]; ++q; } }
                for (int r = 0; r < 6; ++r) b[r] = s_sys[21 + r];
                if (i == 0) { double md = 0; for (int j = 0; j < 6; ++j) md = fmax(fabs(H[6 * j + j]), md); lambda = 1e-5 * md; ni = 2; nbad_lm = 0; }
                double rho = 0; int qmax = 0;
                do {
                    const PoSE3 backup = s_est;
                    __syncthreads();
                    if (tid == 0) {
                        double Hl[36], x[6] = {0, 0, 0, 0, 0, 0};
                        for (int q = 0; q < 36; ++q) Hl[q] = H[q];
                        for (int j = 0; j < 6; ++j) Hl[6 * j + j] += lambda;
                        s_ok2 = po_ldlt6(Hl, b, x) ? 1 : 0;
                        for (int j = 0; j < 6; ++j) s_x[j] = x[j];
                        const PoSE3 ex = po_exp(x);             // setEstimate(SE3Quat::exp(update) * estimate())
                        PoSE3 r = ex;
                        double rt[3]; po_rotate(ex.r, s_est.t, rt);
                        for (int j = 0; j < 3; ++j) r.t[j] += rt[j];
                        r.r = po_mul(ex.r, s_est.r); po_normalize(r.r);
                        s_est = r;
                    }
                    __syncthreads();
                    evaluate(false);
                    double tempChi = s_sys[27];
                    if (!s_ok2) tempChi = DBL_MAX;
                    rho = currentChi - tempChi;
                    double scale = 0;
                    for (int j = 0; j < 6; ++j) scale += s_x[j] * (lambda * s_x[j] + b[j]);
                    scale += 1e-3;
                    rho /= scale;
                    if (rho > 0 && isfinite(tempChi)) {
                        double alpha = 1. - pow((2 * rho - 1), 3.0);
                        alpha = fmin(alpha, 2. / 3.);
                        lambda *= fmax(1. / 3., alpha); ni = 2; currentChi = tempChi;
                    } else {
                        lambda *= ni; ni *= 2;
                        __syncthreads();
                        if (tid == 0) s_est = backup;           // pop(): the edges keep the errors of the rejected trial
                        __syncthreads();
                    }
                    ++qmax;
                } while (rho < 0 && qmax < 10);
                if (qmax == 10 || rho == 0) break;
                if ((iniChi - currentChi) * 1e3 < iniChi) ++nbad_lm; else nbad_lm = 0;
                if (nbad_lm >= 3) break;
            }
        }
        __syncthreads();
        // re-classification (src/Optimizer.cc:364-425)
        int bad = 0;
        const PoSE3 est = s_est;
        for (int i = tid; i < n; i += kPoThreads) {
            if (!has(i)) continue;
            double* E = A.err + 3 * (ko + i);
            double e[3] = {E[0], E[1], E[2]}, pc[3];
            const float ur = A.uright[ko + i];
            const bool stereo = !(ur < 0);
            if (A.outlier[ko + i]) { edge_error(i, est, e, pc); E[0] = e[0]; E[1] = e[1]; E[2] = e[2]; }
            const double info = A.inv_sigma2[A.kps[ko + i].octave];
            const float chi2 = (float)((e[0] * e[0] + e[1] * e[1] + (stereo ? e[2] * e[2] : 0.0)) * info);
            if (chi2 > (stereo ? 7.815f : 5.991f)) { A.outlier[ko + i] = 1; A.level[ko + i] = 1; ++bad; }
            else { A.outlier[ko + i] = 0; A.level[ko + i] = 0; }
        }
        n_bad = (int)po_block_sum((double)bad, s_red);
        __syncthreads();
        if (n_initial < 10) break;
    }
    if (tid == 0) {
        const PoQuat q = s_est.r;
        const double tx = 2 * q.x, ty = 2 * q.y, tz = 2 * q.z;
        const double twx = tx * q.w, twy = ty * q.w, twz = tz * q.w, txx = tx * q.x, txy = ty * q.x, txz = tz * q.x, tyy = ty * q.y, tyz = tz * q.y, tzz = tz * q.z;
        const double R[9] = {1 - (tyy + tzz), txy - twz, txz + twy, txy + twz, 1 - (txx + tzz), tyz - twx, txz - twy, tyz + twx, 1 - (txx + tyy)};
        float* T = A.tcw_out + 16 * (int64_t)f;
        for (int r = 0; r < 3; r++) { for (int c = 0; c < 3; c++) T[4 * r + c] = (float)R[3 * r + c]; T[4 * r + 3] = (float)s_est.t[r]; }
        T[12] = T[13] = T[14] = 0.f; T[15] = 1.f;
        A.ninliers[f] = n_initial - n_bad;
    }
}

}  // namespace sgs

using namespace sgs;

extern "C" {

SGS_API int sgs_pose_optimization_batch_device(const sgs_poseopt_batch* a, int nframes, void* stream) {
    if (!a || !a->tcw_in || !a->kps || !a->uright || !a->n || !a->points_xyz || !a->tcw_out || !a->outlier || !a->ninliers || !a->scratch_err || !a->scratch_level ||
        (!a->has_mp && !a->mp_index) || a->cap < 1 || nframes < 1) { set_error("sgs_pose_optimization_batch_device: bad argument"); return SGS_ERR_INVALID; }
    PoArgs A;
    A.fx = a->cam.fx; A.fy = a->cam.fy; A.cx = a->cam.cx; A.cy = a->cam.cy; A.bf = a->cam.bf;
    A.tcw_in = a->tcw_in; A.kps = a->kps; A.uright = a->uright; A.n = a->n; A.cap = a->cap;
    A.has_mp = a->has_mp; A.mp_index = a->mp_index; A.points_xyz = a->points_xyz; A.point_cap = a->mp_index ? a->point_cap : a->cap;
    A.points2_xyz = a->mp_index ? a->points2_xyz : nullptr; A.id_base2 = a->id_base2; A.point2_cap = a->point2_cap;
    for (int l = 0; l < 16; ++l) A.inv_sigma2[l] = a->inv_level_sigma2[l];
    A.tcw_out = a->tcw_out; A.outlier = a->outlier; A.ninliers = a->ninliers; A.err = a->scratch_err; A.level = a->scratch_level;
    pose_opt_kernel<<<nframes, kPoThreads, 0, (cudaStream_t)stream>>>(A);
    SGS_CUDA_TRY(cudaGetLastError());
    return SGS_OK;
}

// host-pointer variant, one frame: has_mp [n], xyz [n][3] (GetWorldPos of mvpMapPoints[i]), kps = mvKeysUn, uright = mvuRight
SGS_API int sgs_pose_optimization(const sgs_camera* cam, const float* tcw_in, int n, const sgs_keypoint* kps_un, const float* uright, const uint8_t* has_mp,
                                  const float* xyz, const float* inv_level_sigma2, float* tcw_out, uint8_t* outlier, int* ninliers, int device) {
    if (!cam || !tcw_in || !tcw_out || !ninliers || !inv_level_sigma2 || n < 0 || (n > 0 && (!kps_un || !uright || !has_mp || !xyz || !outlier))) {
        set_error("sgs_pose_optimization: bad argument"); return SGS_ERR_INVALID;
    }
    for (int i = 0; i < 16; ++i) tcw_out[i] = tcw_in[i];
    *ninliers = 0;
    if (n == 0) return SGS_OK;
    SGS_CUDA_TRY(cudaSetDevice(device));
    HostCall c("sgs_pose_optimization");
    sgs_poseopt_batch b;
    c.in(&b.tcw_in, tcw_in, 16); c.in(&b.kps, kps_un, n); c.in(&b.uright, uright, n); c.in(&b.n, &n, 1); c.in(&b.has_mp, has_mp, n);
    c.in(&b.points_xyz, xyz, 3 * (size_t)n);
    c.out(&b.tcw_out, tcw_out, 16); c.out(&b.outlier, outlier, n, true); c.out(&b.ninliers, ninliers, 1);
    c.out(&b.scratch_err, nullptr, 3 * (size_t)n); c.out(&b.scratch_level, nullptr, n);
    b.cam = *cam; b.cap = n; b.mp_index = nullptr; b.point_cap = n;
    for (int l = 0; l < 16; ++l) b.inv_level_sigma2[l] = inv_level_sigma2[l];
    b.points2_xyz = nullptr; b.id_base2 = 0; b.point2_cap = 0;
    if (int rc = c.upload()) return rc;
    if (int rc = sgs_pose_optimization_batch_device(&b, 1, nullptr)) return rc;
    return c.download();
}

}  // extern "C"
