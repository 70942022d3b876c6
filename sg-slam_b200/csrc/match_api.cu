// match_api.cu -- C-ABI entry points of the projection matchers: the batched device API (sgs_matcher handle) and the
// single-frame host-pointer wrappers that flatten one Frame pair, run the same kernels with nframes = 1 and copy back.
#include <cuda_runtime.h>

#include <cstring>
#include <vector>

#include "host_call.h"
#include "match_dev.cuh"

using namespace sgs;

struct sgs_matcher {
    int device = 0, max_frames = 0, cur_cap = 0, point_cap = 0;
    PointPre* d_pre = nullptr;
    LocalPre* d_lpre = nullptr;
    int32_t* d_events = nullptr;
};

namespace {

int pow2_at_least(int v) { int p = 1; while (p < v) p <<= 1; return p; }

MatchCam to_cam(const sgs_camera& c) {
    MatchCam m;
    m.min_x = c.min_x; m.min_y = c.min_y; m.max_x = c.max_x; m.max_y = c.max_y;
    m.fx = c.fx; m.fy = c.fy; m.cx = c.cx; m.cy = c.cy; m.bf = c.bf; m.nlevels = c.nlevels;
    for (int i = 0; i < kMaxLevels; ++i) m.scale[i] = c.scale_factors[i];
    return m;
}

sgs_camera view_cam(const sgs_frame_view* v) {
    sgs_camera c;
    std::memset(&c, 0, sizeof c);
    c.min_x = v->min_x; c.min_y = v->min_y; c.max_x = v->max_x; c.max_y = v->max_y;
    c.fx = v->fx; c.fy = v->fy; c.cx = v->cx; c.cy = v->cy; c.bf = v->bf; c.nlevels = v->nlevels;
    for (int i = 0; i < v->nlevels && i < kMaxLevels; ++i) c.scale_factors[i] = v->scale_factors[i];
    return c;
}

int check_cur_cap(int cur_cap) {
    if (cur_cap > 8192) { set_error("sgs_matcher_create: cur_cap %d exceeds the 8192 keypoints per frame the shared-memory grid supports", cur_cap); return SGS_ERR_UNSUPPORTED; }
    return SGS_OK;
}

// the one-frame matcher of a host-pointer call: sgs_matcher_create(device, 1, cur_cap, point_cap), its scratch taken from the call's allocation
int stage_matcher(HostCall& c, int device, int cur_cap, int point_cap, sgs_matcher* m) {
    if (int rc = check_cur_cap(cur_cap)) return rc;
    SGS_CUDA_TRY(cudaSetDevice(device));
    m->device = device; m->max_frames = 1; m->cur_cap = cur_cap; m->point_cap = point_cap;
    c.out(&m->d_pre, nullptr, point_cap); c.out(&m->d_lpre, nullptr, point_cap); c.out(&m->d_events, nullptr, point_cap);
    return SGS_OK;
}

}  // namespace

extern "C" {

SGS_API int sgs_matcher_create(int device, int max_frames, int cur_cap, int point_cap, sgs_matcher** out) {
    if (!out || max_frames < 1 || cur_cap < 1 || point_cap < 1) { set_error("sgs_matcher_create: bad argument"); return SGS_ERR_INVALID; }
    if (int rc = check_cur_cap(cur_cap)) return rc;
    *out = nullptr;
    SGS_CUDA_TRY(cudaSetDevice(device));
    sgs_matcher* m = new sgs_matcher();
    m->device = device; m->max_frames = max_frames; m->cur_cap = cur_cap; m->point_cap = point_cap;
    const size_t np = (size_t)max_frames * point_cap;
    if (cudaMalloc(&m->d_pre, np * sizeof(PointPre)) != cudaSuccess || cudaMalloc(&m->d_lpre, np * sizeof(LocalPre)) != cudaSuccess ||
        cudaMalloc(&m->d_events, np * sizeof(int32_t)) != cudaSuccess) {
        set_error("sgs_matcher_create: cudaMalloc failed: %s", cudaGetErrorString(cudaGetLastError()));
        cudaFree(m->d_pre); cudaFree(m->d_lpre); cudaFree(m->d_events); delete m;
        return SGS_ERR_CUDA;
    }
    *out = m;
    return SGS_OK;
}

SGS_API void sgs_matcher_destroy(sgs_matcher* m) {
    if (!m) return;
    cudaSetDevice(m->device);
    cudaFree(m->d_pre); cudaFree(m->d_lpre); cudaFree(m->d_events);
    delete m;
}

SGS_API int sgs_match_project_lastframe_batch_device(sgs_matcher* m, const sgs_lastframe_batch* a, int nframes, void* stream) {
    if (!m || !a) { set_error("sgs_match_project_lastframe_batch_device: NULL"); return SGS_ERR_INVALID; }
    if (nframes < 1 || nframes > m->max_frames) { set_error("nframes outside [1,max_frames]"); return SGS_ERR_INVALID; }
    LastFrameArgs A;
    A.cam = to_cam(a->cam);
    A.cur_kps = a->cur_kps; A.cur_desc = a->cur_desc; A.cur_uright = a->cur_uright; A.cur_n = a->cur_n;
    A.cur_cap = m->cur_cap; A.cur_cap_pow2 = pow2_at_least(m->cur_cap);
    A.last_xyz = a->last_xyz; A.last_desc = a->last_desc; A.last_flags = a->last_flags; A.last_octave = a->last_octave;
    A.last_angle = a->last_angle; A.last_n = a->last_n; A.last_cap = m->point_cap;
    A.tcw_cur = a->tcw_cur; A.tcw_last = a->tcw_last; A.th = a->th; A.mono = a->mono; A.check_ori = a->check_orientation;
    A.cur_mp = a->cur_mp; A.cur_mp_obs_in = a->cur_mp_obs_in; A.nmatches = a->nmatches; A.ncand = (unsigned long long*)a->ncand;
    A.kf_mode = 0; A.orb_dist = 100; A.log_sf = 0.f; A.kf_min_dist = A.kf_max_dist = nullptr;      // TH_HIGH, src/ORBmatcher.cc:37
    A.frame_enable = a->frame_enable;
    A.pre = m->d_pre; A.events = m->d_events;
    return launch_match_lastframe(A, nframes, (cudaStream_t)stream);
}

SGS_API int sgs_fuse_search_batch_device(const sgs_fuse_batch* a, int nframes, void* stream) {
    if (!a || !a->kf_kps || !a->kf_desc || !a->kf_uright || !a->kf_n || !a->tcw || !a->ow || !a->mp_xyz || !a->mp_normal || !a->mp_min_dist || !a->mp_max_dist ||
        !a->mp_desc || !a->mp_valid || !a->mp_n || !a->best_idx || !a->best_dist || nframes < 1 || a->kf_cap < 1 || a->mp_cap < 1) {
        set_error("sgs_fuse_search_batch_device: bad argument"); return SGS_ERR_INVALID;
    }
    if (a->cam.nlevels < 2 || a->cam.nlevels > kMaxLevels || !(a->cam.scale_factors[1] > 1.f)) { set_error("sgs_fuse_search_batch_device: camera scale table missing"); return SGS_ERR_INVALID; }
    FuseArgs A;
    A.cam = to_cam(a->cam);
    A.kf_kps = a->kf_kps; A.kf_desc = a->kf_desc; A.kf_uright = a->kf_uright; A.kf_n = a->kf_n; A.kf_cap = a->kf_cap;
    A.tcw = a->tcw; A.ow = a->ow; A.mp_xyz = a->mp_xyz; A.mp_normal = a->mp_normal; A.mp_min_dist = a->mp_min_dist; A.mp_max_dist = a->mp_max_dist;
    A.mp_desc = a->mp_desc; A.mp_valid = a->mp_valid; A.mp_n = a->mp_n; A.mp_cap = a->mp_cap; A.th = a->th; A.log_sf = logf(a->cam.scale_factors[1]);
    for (int l = 0; l < kMaxLevels; ++l) A.inv_sigma2[l] = a->inv_level_sigma2[l];
    A.sim3_variant = a->sim3_variant; A.xform2 = a->xform2;
    if (a->sim3_variant < 0 || a->sim3_variant > 3 || (a->sim3_variant == 2 && !a->xform2) || (a->sim3_variant == 3 && !a->kf_matched)) {
        set_error("sgs_fuse_search_batch_device: bad variant"); return SGS_ERR_INVALID; }
    A.best_idx = a->best_idx; A.best_dist = a->best_dist;
    A.kf_matched = a->kf_matched; A.nmatches = a->nmatches;
    return launch_fuse_search(A, nframes, (cudaStream_t)stream);
}

SGS_API int sgs_match_project_keyframe_batch_device(sgs_matcher* m, const sgs_keyframe_batch* a, int nframes, void* stream) {
    if (!m || !a) { set_error("sgs_match_project_keyframe_batch_device: NULL"); return SGS_ERR_INVALID; }
    if (nframes < 1 || nframes > m->max_frames) { set_error("nframes outside [1,max_frames]"); return SGS_ERR_INVALID; }
    if (!a->cur_kps || !a->cur_desc || !a->cur_n || !a->kf_xyz || !a->kf_desc || !a->kf_valid || !a->kf_angle || !a->kf_min_dist || !a->kf_max_dist ||
        !a->kf_n || !a->tcw_cur || !a->cur_mp || !a->nmatches || !a->ncand || !a->cur_uright) { set_error("sgs_match_project_keyframe_batch_device: NULL array"); return SGS_ERR_INVALID; }
    if (a->cam.nlevels < 2 || !(a->cam.scale_factors[1] > 1.f)) { set_error("sgs_match_project_keyframe_batch_device: camera scale table missing"); return SGS_ERR_INVALID; }
    LastFrameArgs A;
    A.cam = to_cam(a->cam);
    A.cur_kps = a->cur_kps; A.cur_desc = a->cur_desc; A.cur_uright = a->cur_uright; A.cur_n = a->cur_n;
    A.cur_cap = m->cur_cap; A.cur_cap_pow2 = pow2_at_least(m->cur_cap);
    A.last_xyz = a->kf_xyz; A.last_desc = a->kf_desc; A.last_flags = a->kf_valid; A.last_octave = nullptr;
    A.last_angle = a->kf_angle; A.last_n = a->kf_n; A.last_cap = m->point_cap;
    A.tcw_cur = a->tcw_cur; A.tcw_last = nullptr; A.th = a->th; A.mono = 1; A.check_ori = a->check_orientation;
    A.cur_mp = a->cur_mp; A.cur_mp_obs_in = nullptr; A.nmatches = a->nmatches; A.ncand = (unsigned long long*)a->ncand;
    A.kf_mode = 1; A.orb_dist = a->orb_dist; A.log_sf = logf(a->cam.scale_factors[1]); A.kf_min_dist = a->kf_min_dist; A.kf_max_dist = a->kf_max_dist;
    A.frame_enable = nullptr;
    A.pre = m->d_pre; A.events = m->d_events;
    return launch_match_lastframe(A, nframes, (cudaStream_t)stream);
}

SGS_API int sgs_match_project_localmap_batch_device(sgs_matcher* m, const sgs_localmap_batch* a, int nframes, void* stream) {
    if (!m || !a) { set_error("sgs_match_project_localmap_batch_device: NULL"); return SGS_ERR_INVALID; }
    if (nframes < 1 || nframes > m->max_frames) { set_error("nframes outside [1,max_frames]"); return SGS_ERR_INVALID; }
    LocalMapArgs A;
    A.cam = to_cam(a->cam);
    A.cur_kps = a->cur_kps; A.cur_desc = a->cur_desc; A.cur_uright = a->cur_uright; A.cur_n = a->cur_n;
    A.cur_cap = m->cur_cap; A.cur_cap_pow2 = pow2_at_least(m->cur_cap);
    A.mp_inview = a->mp_inview; A.proj_x = a->proj_x; A.proj_y = a->proj_y; A.proj_xr = a->proj_xr; A.level = a->level;
    A.view_cos = a->view_cos; A.mp_desc = a->mp_desc; A.mp_obs = a->mp_obs; A.mp_n = a->mp_n; A.mp_cap = m->point_cap;
    A.th = a->th; A.nnratio = a->nnratio; A.id_base = a->id_base;
    A.f_mp = a->f_mp; A.f_mp_obs = a->f_mp_obs; A.nmatches = a->nmatches; A.ncand = (unsigned long long*)a->ncand;
    A.pre = m->d_lpre;
    return launch_match_localmap(A, nframes, (cudaStream_t)stream);
}

SGS_API int sgs_match_project_lastframe(const sgs_frame_view* cur, const float* tcw_cur, const float* tcw_last, int nlast,
                                        const uint8_t* last_has_mp, const float* last_xyz, const uint8_t* last_desc, const uint8_t* last_obs,
                                        const int32_t* last_octave, const float* last_angle, float th, int mono, int check_orientation,
                                        int32_t* cur_mp_inout, const uint8_t* cur_mp_obs_in, int* nmatches, int device) {
    if (!cur || !tcw_cur || !tcw_last || !nmatches || nlast < 0 || cur->n < 0) { set_error("sgs_match_project_lastframe: bad argument"); return SGS_ERR_INVALID; }
    *nmatches = 0;
    if (nlast == 0 || cur->n == 0) return SGS_OK;
    if (!last_has_mp || !last_xyz || !last_desc || !last_obs || !last_octave || !last_angle || !cur_mp_inout || !cur->keys_un || !cur->u_right || !cur->desc) {
        set_error("sgs_match_project_lastframe: NULL array"); return SGS_ERR_INVALID;
    }
    HostCall c("sgs_match_project_lastframe");
    sgs_matcher m;
    if (int rc = stage_matcher(c, device, cur->n, nlast, &m)) return rc;
    const int n = cur->n;
    std::vector<uint8_t> flags(nlast);
    for (int i = 0; i < nlast; ++i) flags[i] = (uint8_t)((last_has_mp[i] ? 1 : 0) | (last_obs[i] ? 2 : 0));
    sgs_lastframe_batch b;
    std::memset(&b, 0, sizeof b);
    b.cam = view_cam(cur);
    c.in(&b.cur_kps, cur->keys_un, n); c.in(&b.cur_desc, cur->desc, 32 * (size_t)n); c.in(&b.cur_uright, cur->u_right, n); c.in(&b.cur_n, &cur->n, 1);
    c.in(&b.last_xyz, last_xyz, 3 * (size_t)nlast); c.in(&b.last_desc, last_desc, 32 * (size_t)nlast); c.in(&b.last_flags, flags.data(), nlast);
    c.in(&b.last_octave, last_octave, nlast); c.in(&b.last_angle, last_angle, nlast); c.in(&b.last_n, &nlast, 1);
    c.in(&b.tcw_cur, tcw_cur, 16); c.in(&b.tcw_last, tcw_last, 16);
    c.inout(&b.cur_mp, cur_mp_inout, n);
    if (cur_mp_obs_in) c.in(&b.cur_mp_obs_in, cur_mp_obs_in, n);
    c.out(&b.nmatches, nmatches, 1); c.out(&b.ncand, nullptr, 1, true);
    b.th = th; b.mono = mono; b.check_orientation = check_orientation;
    if (int rc = c.upload()) return rc;
    if (int rc = sgs_match_project_lastframe_batch_device(&m, &b, 1, nullptr)) return rc;
    return c.download();
}

SGS_API int sgs_match_project_keyframe(const sgs_frame_view* cur, const float* tcw_cur, int nkf, const uint8_t* kf_valid, const float* kf_xyz,
                                       const uint8_t* kf_desc, const float* kf_angle, const float* kf_min_dist, const float* kf_max_dist, float th,
                                       int orb_dist, int check_orientation, int32_t* cur_mp_inout, int* nmatches, int device) {
    if (!cur || !tcw_cur || !nmatches || nkf < 0 || cur->n < 0) { set_error("sgs_match_project_keyframe: bad argument"); return SGS_ERR_INVALID; }
    *nmatches = 0;
    if (nkf == 0 || cur->n == 0) return SGS_OK;
    if (!kf_valid || !kf_xyz || !kf_desc || !kf_angle || !kf_min_dist || !kf_max_dist || !cur_mp_inout || !cur->keys_un || !cur->u_right || !cur->desc) {
        set_error("sgs_match_project_keyframe: NULL array"); return SGS_ERR_INVALID;
    }
    HostCall c("sgs_match_project_keyframe");
    sgs_matcher m;
    if (int rc = stage_matcher(c, device, cur->n, nkf, &m)) return rc;
    const int n = cur->n;
    std::vector<uint8_t> flags(nkf);
    for (int i = 0; i < nkf; ++i) flags[i] = kf_valid[i] ? 1 : 0;
    sgs_keyframe_batch b;
    std::memset(&b, 0, sizeof b);
    b.cam = view_cam(cur);
    c.in(&b.cur_kps, cur->keys_un, n); c.in(&b.cur_desc, cur->desc, 32 * (size_t)n); c.in(&b.cur_uright, cur->u_right, n); c.in(&b.cur_n, &cur->n, 1);
    c.in(&b.kf_valid, flags.data(), nkf); c.in(&b.kf_xyz, kf_xyz, 3 * (size_t)nkf); c.in(&b.kf_desc, kf_desc, 32 * (size_t)nkf);
    c.in(&b.kf_angle, kf_angle, nkf); c.in(&b.kf_min_dist, kf_min_dist, nkf); c.in(&b.kf_max_dist, kf_max_dist, nkf);
    c.in(&b.kf_n, &nkf, 1); c.in(&b.tcw_cur, tcw_cur, 16);
    c.inout(&b.cur_mp, cur_mp_inout, n); c.out(&b.nmatches, nmatches, 1); c.out(&b.ncand, nullptr, 1, true);
    b.th = th; b.orb_dist = orb_dist; b.check_orientation = check_orientation;
    if (int rc = c.upload()) return rc;
    if (int rc = sgs_match_project_keyframe_batch_device(&m, &b, 1, nullptr)) return rc;
    return c.download();
}

SGS_API int sgs_fuse_search(const sgs_frame_view* kf, const float* tcw, const float* ow, int nmp, const uint8_t* mp_valid, const float* mp_xyz,
                            const float* mp_normal, const float* mp_min_dist, const float* mp_max_dist, const uint8_t* mp_desc, float th,
                            const float* inv_level_sigma2, int sim3_variant, const float* xform2, int32_t* best_idx, int32_t* best_dist,
                            int32_t* kf_matched_inout, int* nmatches, int device) {
    if (!kf || !tcw || !ow || nmp < 0 || kf->n < 0 || !best_idx || !best_dist) { set_error("sgs_fuse_search: bad argument"); return SGS_ERR_INVALID; }
    if (nmatches) *nmatches = 0;
    for (int i = 0; i < nmp; ++i) { best_idx[i] = -1; best_dist[i] = 256; }
    if (nmp == 0 || kf->n == 0) return SGS_OK;
    if (!mp_valid || !mp_xyz || !mp_normal || !mp_min_dist || !mp_max_dist || !mp_desc || !kf->keys_un || !kf->u_right || !kf->desc ||
        (sim3_variant == 0 && !inv_level_sigma2) || (sim3_variant == 3 && !kf_matched_inout)) { set_error("sgs_fuse_search: NULL array"); return SGS_ERR_INVALID; }
    SGS_CUDA_TRY(cudaSetDevice(device));
    const int n = kf->n;
    HostCall c("sgs_fuse_search");
    sgs_fuse_batch b;
    std::memset(&b, 0, sizeof b);
    b.cam = view_cam(kf);
    c.in(&b.kf_kps, kf->keys_un, n); c.in(&b.kf_desc, kf->desc, 32 * (size_t)n); c.in(&b.kf_uright, kf->u_right, n); c.in(&b.kf_n, &kf->n, 1);
    c.in(&b.tcw, tcw, 16); c.in(&b.ow, ow, 3);
    c.in(&b.mp_xyz, mp_xyz, 3 * (size_t)nmp); c.in(&b.mp_normal, mp_normal, 3 * (size_t)nmp); c.in(&b.mp_min_dist, mp_min_dist, nmp);
    c.in(&b.mp_max_dist, mp_max_dist, nmp); c.in(&b.mp_desc, mp_desc, 32 * (size_t)nmp); c.in(&b.mp_valid, mp_valid, nmp); c.in(&b.mp_n, &nmp, 1);
    if (xform2) c.in(&b.xform2, xform2, 12);
    c.out(&b.best_idx, best_idx, nmp); c.out(&b.best_dist, best_dist, nmp);
    // vpMatched and the match count belong to variant 3 alone: only it reads and writes them, and only it copies them back
    if (sim3_variant == 3) c.inout(&b.kf_matched, kf_matched_inout, n);
    c.out(&b.nmatches, sim3_variant == 3 ? nmatches : nullptr, 1);
    b.kf_cap = n; b.mp_cap = nmp; b.th = th; b.sim3_variant = sim3_variant;
    for (int l = 0; l < 16; ++l) b.inv_level_sigma2[l] = inv_level_sigma2 && l < kf->nlevels ? inv_level_sigma2[l] : 0.f;
    if (int rc = c.upload()) return rc;
    if (int rc = sgs_fuse_search_batch_device(&b, 1, nullptr)) return rc;
    return c.download();
}

SGS_API int sgs_search_for_initialization_batch_device(const sgs_init_batch* a, int nframes, void* stream) {
    if (!a || !a->f1_kps || !a->f1_desc || !a->f1_n || !a->f2_kps || !a->f2_desc || !a->f2_n || !a->prev_xy || !a->match12 || nframes < 1 || a->f1_cap < 1 || a->f2_cap < 1 ||
        a->window_size < 0 || !(a->cam.max_x > a->cam.min_x) || !(a->cam.max_y > a->cam.min_y)) { set_error("sgs_search_for_initialization_batch_device: bad argument"); return SGS_ERR_INVALID; }
    InitArgs A;
    A.cam = to_cam(a->cam);
    A.f1_kps = a->f1_kps; A.f1_desc = a->f1_desc; A.f1_n = a->f1_n; A.f1_cap = a->f1_cap;
    A.f2_kps = a->f2_kps; A.f2_desc = a->f2_desc; A.f2_n = a->f2_n; A.f2_cap = a->f2_cap;
    A.prev_xy = a->prev_xy; A.window = a->window_size; A.nnratio = a->nnratio; A.check_ori = a->check_orientation; A.match12 = a->match12; A.nmatches = a->nmatches;
    return launch_search_init(A, nframes, (cudaStream_t)stream);
}

SGS_API int sgs_search_for_initialization(const sgs_frame_view* f1, const sgs_frame_view* f2, float* prev_xy, int window_size, float nnratio, int check_orientation,
                                          int32_t* match12, int* nmatches, int device) {
    if (!f1 || !f2 || !nmatches || f1->n < 0 || f2->n < 0) { set_error("sgs_search_for_initialization: bad argument"); return SGS_ERR_INVALID; }
    *nmatches = 0;
    if (f1->n > 0 && match12) for (int i = 0; i < f1->n; ++i) match12[i] = -1;
    if (f1->n == 0 || f2->n == 0) return SGS_OK;
    if (!prev_xy || !match12 || !f1->keys_un || !f1->desc || !f2->keys_un || !f2->desc) { set_error("sgs_search_for_initialization: NULL array"); return SGS_ERR_INVALID; }
    SGS_CUDA_TRY(cudaSetDevice(device));
    HostCall c("sgs_search_for_initialization");
    sgs_init_batch b;
    std::memset(&b, 0, sizeof b);
    b.cam = view_cam(f2);
    c.in(&b.f1_kps, f1->keys_un, f1->n); c.in(&b.f1_desc, f1->desc, 32 * (size_t)f1->n); c.in(&b.f1_n, &f1->n, 1);
    c.in(&b.f2_kps, f2->keys_un, f2->n); c.in(&b.f2_desc, f2->desc, 32 * (size_t)f2->n); c.in(&b.f2_n, &f2->n, 1);
    c.inout(&b.prev_xy, prev_xy, 2 * (size_t)f1->n); c.out(&b.match12, match12, f1->n); c.out(&b.nmatches, nmatches, 1);
    b.f1_cap = f1->n; b.f2_cap = f2->n; b.window_size = window_size; b.nnratio = nnratio; b.check_orientation = check_orientation;
    if (int rc = c.upload()) return rc;
    if (int rc = sgs_search_for_initialization_batch_device(&b, 1, nullptr)) return rc;
    return c.download();
}

SGS_API int sgs_match_bow_keyframes(int mode, int n1, const int32_t* node1, const double* weight1, const uint8_t* valid1, const uint8_t* desc1, const float* angle1,
                                    int n2, const int32_t* node2, const double* weight2, const uint8_t* valid2, const uint8_t* desc2, const float* angle2,
                                    float nnratio, int check_orientation, const uint8_t* stereo1, const uint8_t* stereo2, const float* xy1, const float* xy2,
                                    const int32_t* octave2, const float* F12, const float* epipole, const float* level_sigma2, const float* scale_factors, int nlevels,
                                    int only_stereo, int32_t* match12, int* nmatches, int device) {
    if (!nmatches || n1 < 0 || n2 < 0 || (mode != 1 && mode != 2)) { set_error("sgs_match_bow_keyframes: bad argument"); return SGS_ERR_INVALID; }
    *nmatches = 0;
    if (n1 > 0 && match12) for (int i = 0; i < n1; ++i) match12[i] = -1;
    if (n1 == 0 || n2 == 0) return SGS_OK;
    if (!node1 || !weight1 || !valid1 || !desc1 || !angle1 || !node2 || !weight2 || !valid2 || !desc2 || !angle2 || !match12) { set_error("sgs_match_bow_keyframes: NULL array"); return SGS_ERR_INVALID; }
    if (mode == 2 && (!stereo1 || !stereo2 || !xy1 || !xy2 || !octave2 || !F12 || !epipole || !level_sigma2 || !scale_factors || nlevels < 1 || nlevels > 16)) {
        set_error("sgs_match_bow_keyframes: triangulation mode needs stereo flags, positions, octaves, F12, the epipole and the level tables"); return SGS_ERR_INVALID; }
    SGS_CUDA_TRY(cudaSetDevice(device));
    HostCall c("sgs_match_bow_keyframes");
    sgs_bow_batch b;
    std::memset(&b, 0, sizeof b);
    c.in(&b.kf_node, node1, n1); c.in(&b.kf_weight, weight1, n1); c.in(&b.kf_valid, valid1, n1); c.in(&b.kf_desc, desc1, 32 * (size_t)n1); c.in(&b.kf_angle, angle1, n1);
    c.in(&b.f_node, node2, n2); c.in(&b.f_weight, weight2, n2); c.in(&b.f_valid, valid2, n2); c.in(&b.f_desc, desc2, 32 * (size_t)n2); c.in(&b.f_angle, angle2, n2);
    c.in(&b.kf_n, &n1, 1); c.in(&b.f_n, &n2, 1); c.out(&b.match_f, match12, n1); c.out(&b.nmatches, nmatches, 1);
    b.kf_cap = n1; b.f_cap = n2; b.keyframe_pair = mode; b.nnratio = nnratio; b.check_orientation = check_orientation;
    if (mode == 2) {
        c.in(&b.kf_stereo, stereo1, n1); c.in(&b.f_stereo, stereo2, n2); c.in(&b.kf_xy, xy1, 2 * (size_t)n1); c.in(&b.f_xy, xy2, 2 * (size_t)n2);
        c.in(&b.f_octave, octave2, n2); c.in(&b.F12, F12, 9); c.in(&b.epipole, epipole, 2);
        b.only_stereo = only_stereo;
        for (int l = 0; l < nlevels; ++l) { b.level_sigma2[l] = level_sigma2[l]; b.scale_factors[l] = scale_factors[l]; }
    }
    if (int rc = c.upload()) return rc;
    if (int rc = sgs_match_bow_batch_device(&b, 1, nullptr)) return rc;
    return c.download();
}

SGS_API int sgs_match_project_localmap(const sgs_frame_view* f, int nmp, const uint8_t* mp_inview, const float* proj_x, const float* proj_y,
                                       const float* proj_xr, const int32_t* level, const float* view_cos, const uint8_t* mp_desc,
                                       const uint8_t* mp_obs, float th, float nnratio, int32_t id_base, int32_t* f_mp_inout,
                                       uint8_t* f_mp_obs_inout, int* nmatches, int device) {
    if (!f || !nmatches || nmp < 0 || f->n < 0) { set_error("sgs_match_project_localmap: bad argument"); return SGS_ERR_INVALID; }
    *nmatches = 0;
    if (nmp == 0 || f->n == 0) return SGS_OK;
    if (!mp_inview || !proj_x || !proj_y || !proj_xr || !level || !view_cos || !mp_desc || !mp_obs || !f_mp_inout || !f_mp_obs_inout) {
        set_error("sgs_match_project_localmap: NULL array"); return SGS_ERR_INVALID;
    }
    HostCall c("sgs_match_project_localmap");
    sgs_matcher m;
    if (int rc = stage_matcher(c, device, f->n, nmp, &m)) return rc;
    const int n = f->n;
    sgs_localmap_batch b;
    std::memset(&b, 0, sizeof b);
    b.cam = view_cam(f);
    c.in(&b.cur_kps, f->keys_un, n); c.in(&b.cur_desc, f->desc, 32 * (size_t)n); c.in(&b.cur_uright, f->u_right, n); c.in(&b.cur_n, &f->n, 1);
    c.in(&b.mp_inview, mp_inview, nmp); c.in(&b.proj_x, proj_x, nmp); c.in(&b.proj_y, proj_y, nmp); c.in(&b.proj_xr, proj_xr, nmp); c.in(&b.level, level, nmp);
    c.in(&b.view_cos, view_cos, nmp); c.in(&b.mp_desc, mp_desc, 32 * (size_t)nmp); c.in(&b.mp_obs, mp_obs, nmp); c.in(&b.mp_n, &nmp, 1);
    c.inout(&b.f_mp, f_mp_inout, n); c.inout(&b.f_mp_obs, f_mp_obs_inout, n); c.out(&b.nmatches, nmatches, 1); c.out(&b.ncand, nullptr, 1, true);
    b.th = th; b.nnratio = nnratio; b.id_base = id_base;
    if (int rc = c.upload()) return rc;
    if (int rc = sgs_match_project_localmap_batch_device(&m, &b, 1, nullptr)) return rc;
    return c.download();
}

}  // extern "C"
