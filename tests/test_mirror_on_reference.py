"""The mirror headers RUN inside the reference's own tracking thread, without a device: src/Tracking.cc (TrackWithMotionModel, TrackLocalMap, SearchLocalPoints) is
compiled unmodified with include/sgslam/ORBmatcher.h in place of the reference's ORBmatcher and with Optimizer::PoseOptimization forwarded to
include/sgslam/Optimizer.h (tests/cpp/mirror_on_reference_pre.h), on the reference's real Frame / MapPoint classes; the three C-ABI entry points the mirror reaches
(sgs_match_project_lastframe, sgs_match_project_localmap, sgs_pose_optimization) are answered by the CPU oracle (tests/cpp/fake_sgs_backend.cpp) instead of the
CUDA library.  Result for result it must equal the all-reference build of the same code (oracle/_ref/libtracking_ref.so: the reference's ORBmatcher.cc and
Optimizer.cc + g2o): map point per keypoint after each half, outlier flags, mnMatchesInliers, both return values, poses.  Under test is the product's HEADER code --
flattening the object graph (NULL / outlier / bad / Observations() rules), the ids handed to the matchers, writing mvpMapPoints / mvbOutlier / the pose back -- on
the classes it will meet in the reference; the kernels behind the same entry points are tests/test_gpu_*.py.  Needs the reference tree (build container)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import oracle as O
from pysgs import binding as B
from pysgs import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = '/root/reference/src/sg-slam'
REFLIB = os.path.join(ROOT, 'oracle', '_ref', 'libtracking_ref.so')
pytestmark = pytest.mark.skipif(not (os.path.exists(os.path.join(REF, 'src', 'Tracking.cc')) and os.path.exists(REFLIB)), reason='reference tree / libtracking_ref.so absent')
W, H, TH = 640, 480, 15.0


@pytest.fixture(scope='module')
def mirror_lib(tmp_path_factory):
    out = str(tmp_path_factory.mktemp('mirror') / 'libtracking_mirror.so')
    o = os.path.join(ROOT, 'oracle'); src = os.path.join(REF, 'src'); dbow = os.path.join(REF, 'Thirdparty', 'DBoW2', 'DBoW2')
    cmd = ['g++', '-O1', '-std=c++11', '-fPIC', '-shared', '-fvisibility=hidden', '-w', '-ffp-contract=off', '-DSGS_WITH_OPENCV', '-I' + os.path.join(ROOT, 'include'),
           '-I' + os.path.join(o, 'tracking_shim'), '-I' + os.path.join(o, 'g2o_shim'), '-I' + os.path.join(o, 'frame_shim'), '-I' + os.path.join(o, 'orbmatcher_shim'),
           '-I' + REF, '-I' + os.path.join(REF, 'include'), '-I' + os.path.join(REF, 'Thirdparty', 'g2o'), '-include', os.path.join(ROOT, 'tests', 'cpp', 'mirror_on_reference_pre.h'),
           '-o', out, os.path.join(o, 'tracking_ref_driver.cpp'), os.path.join(ROOT, 'tests', 'cpp', 'fake_sgs_backend.cpp')] + \
          [os.path.join(src, f) for f in ('Tracking.cc', 'Frame.cc', 'MapPoint.cc', 'Converter.cc', 'ORBextractor.cc')] + \
          [os.path.join(dbow, 'BowVector.cpp'), os.path.join(dbow, 'FeatureVector.cpp'), '-Wl,-Bsymbolic', '-L' + o, '-l:liboracle.so', '-Wl,-rpath,' + o,
           '-L' + os.path.join(ROOT, 'sg-slam_b200', 'lib'), '-l:libsgs_cuda.so', '-Wl,-rpath,' + os.path.join(ROOT, 'sg-slam_b200', 'lib'), '-l:libstdc++.so.6', '-pthread']
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return out


@pytest.mark.parametrize('seed,mono_every', [(11, 0), (23, 7)])
def test_mirror_headers_inside_the_reference_tracking_thread(mirror_lib, seed, mono_every):
    import bench
    from test_tracking_ref import reference_chain
    nb, unique = 12, 6
    frames, boxes, unique = bench.make_frames(nb, seed, W, H, unique=unique)
    pidx = bench.prev_index(nb, unique)
    camd = dict(synth.TUM3)
    sf = synth.scale_factors(); cam = B.make_camera(W, H, camd, sf)
    NF = 1000; pc = NF + 64; cap = NF + 8 * 8 + 64; mcap = 1536
    kps = np.zeros((nb, cap), O.KP_DTYPE); desc = np.zeros((nb, cap, 32), np.uint8); cnt = np.zeros(nb, np.int32)
    for f in range(nb):
        k, d = O.extract(frames[f])[:2]
        cnt[f] = len(k); kps[f, :len(k)] = k; desc[f, :len(k)] = d
    ti = bench.make_track_inputs(kps, desc, cnt, boxes, cap, pc, pidx, W, H, camd)
    ti['lflags'][:, 9::23] |= 4
    if mono_every:
        ti['ur'][:, ::mono_every] = -1.0
    Tc = ti['T'].copy()
    c, s_ = np.cos(60.0 / camd['fx']), np.sin(60.0 / camd['fx'])
    R = np.eye(4, dtype=np.float32); R[0, 0] = c; R[0, 2] = s_; R[2, 0] = -s_; R[2, 2] = c
    Tc[3] = R.reshape(16); ti['ln'][3] = 300; ti['ln'][5] = 0
    rng = np.random.default_rng(seed)
    isig = np.zeros(16, np.float32); isig[:8] = 1.0 / (sf.astype(np.float32) ** 2)
    camv = np.array([camd['fx'], camd['fy'], camd['cx'], camd['cy'], camd['bf'], cam.min_x, cam.min_y, cam.max_x, cam.max_y], np.float32)
    nmatched = 0
    for f in range(nb):
        n = int(cnt[f]); m = int(ti['ln'][f])
        cur = O.FrameArrays(kps[f, :n], ti['ur'][f, :n], desc[f, :n], W, H, camd['fx'], camd['fy'], camd['cx'], camd['cy'], camd['bf'], sf)
        lm = bench.make_local_map(f, kps[f], desc[f], n, ti, mcap, camd, sf, rng, W, H)
        for j in np.nonzero(lm['lid'][:m] >= 0)[0]:
            l = lm['lid'][j]
            lm['xyz'][l] = ti['lxyz'][f, j]; lm['obs'][l] = (ti['lflags'][f, j] >> 1) & 1; lm['valid'][l] = 0 if ti['lflags'][f, j] & 4 else 1
        a = reference_chain(camv, sf, isig, cur, Tc[f], m, ti, f, lm, pc, lib=REFLIB)          # ORBmatcher.cc + Optimizer.cc + g2o
        b = reference_chain(camv, sf, isig, cur, Tc[f], m, ti, f, lm, pc, lib=mirror_lib)      # the mirror headers on the oracle-backed C ABI
        assert a['ok1'].value == b['ok1'].value and a['ok2'].value == b['ok2'].value and a['inl'].value == b['inl'].value, f
        assert np.array_equal(a['mp1'], b['mp1']) and np.array_equal(a['mp2'], b['mp2']) and np.array_equal(a['outl'], b['outl']), f
        assert np.abs(a['T1'] - b['T1']).max() <= 1e-6 and np.abs(a['T2'] - b['T2']).max() <= 1e-6, f
        nmatched += int((a['mp2'] >= 0).sum())
    assert nmatched > 500 * nb // 2


def _reference_keyframe(lib, camv, sf, isig, cur, cur_node, kf, Tl):
    L = C.CDLL(lib)
    n = cur.c.N; m = len(kf['xyz'])
    v = C.c_void_p
    P = lambda a: a.ctypes.data_as(v)
    a = lambda x, dt: np.ascontiguousarray(x, dt)
    xy = a(np.stack([cur.keysUn['x'], cur.keysUn['y']], 1), np.float32)
    keep = [xy, a(cur.keysUn['octave'], np.int32), a(cur.keysUn['angle'], np.float32), cur.uRight, cur.desc, a(cur_node, np.int32),
            a(kf['xyz'], np.float32), a(kf['desc'], np.uint8), a(kf['flags'], np.uint8), a(kf['angle'], np.float32), a(kf['node'], np.int32), a(Tl, np.float32)]
    out = dict(ok=C.c_int32(), T=np.zeros(16, np.float32), mp=np.zeros(n, np.int32), held=C.c_int32())
    L.ref_track_reference_keyframe(P(camv), P(a(sf, np.float32)), P(isig), 8, n, *[P(x) for x in keep[:6]], m, *[P(x) for x in keep[6:]],
                                   C.byref(out['ok']), P(out['T']), P(out['mp']), C.byref(out['held']))
    return out


@pytest.mark.parametrize('seed', [3, 8])
def test_mirror_search_by_bow_inside_track_reference_keyframe(mirror_lib, seed):
    """Tracking::TrackReferenceKeyFrame (src/Tracking.cc:796-838): SearchByBoW(reference key frame, frame) through the mirror + PoseOptimization + outlier discard,
    against the all-reference build.  The key frame is the previous frame of the stream with its depth-backed points; the vocabulary node of a feature is a coarse
    function of its position and octave (any partition works for the comparison; this one keeps true correspondences in the same node)."""
    import bench
    nb, unique = 8, 4
    frames, boxes, unique = bench.make_frames(nb, seed, W, H, unique=unique)
    pidx = bench.prev_index(nb, unique)
    camd = dict(synth.TUM3)
    sf = synth.scale_factors(); cam = B.make_camera(W, H, camd, sf)
    NF = 1000; pc = NF + 64; cap = NF + 8 * 8 + 64
    kps = np.zeros((nb, cap), O.KP_DTYPE); desc = np.zeros((nb, cap, 32), np.uint8); cnt = np.zeros(nb, np.int32)
    for f in range(nb):
        k, d = O.extract(frames[f])[:2]
        cnt[f] = len(k); kps[f, :len(k)] = k; desc[f, :len(k)] = d
    ti = bench.make_track_inputs(kps, desc, cnt, boxes, cap, pc, pidx, W, H, camd)
    ti['lflags'][:, 9::23] |= 4
    isig = np.zeros(16, np.float32); isig[:8] = 1.0 / (sf.astype(np.float32) ** 2)
    camv = np.array([camd['fx'], camd['fy'], camd['cx'], camd['cy'], camd['bf'], cam.min_x, cam.min_y, cam.max_x, cam.max_y], np.float32)
    node_of = lambda k: (k['octave'].astype(np.int64) * 64 + (k['y'] // 96).astype(np.int64) * 8 + (k['x'] // 96).astype(np.int64)).astype(np.int32)
    accepted = 0
    for f in range(nb):
        n = int(cnt[f]); g = int(pidx[f]); m = int(ti['ln'][f])
        cur = O.FrameArrays(kps[f, :n], ti['ur'][f, :n], desc[f, :n], W, H, camd['fx'], camd['fy'], camd['cx'], camd['cy'], camd['bf'], sf)
        cur_node = node_of(kps[f, :n]); cur_node[::13] = -1                      # some features are not listed in the FeatureVector
        kf = dict(xyz=ti['lxyz'][f, :m], desc=ti['ldesc'][f, :m], flags=ti['lflags'][f, :m].copy(), angle=ti['lang'][f, :m], node=node_of(kps[g, :m]))
        kf['flags'][::17] = 0                                                     # features of the key frame without a map point
        if f == 5:
            kf['flags'][:] = 0; kf['flags'][:10] = 3                             # too few points: nmatches < 15, the function returns before SetPose
        a = _reference_keyframe(REFLIB, camv, sf, isig, cur, cur_node, kf, ti['T'][f])
        b = _reference_keyframe(mirror_lib, camv, sf, isig, cur, cur_node, kf, ti['T'][f])
        assert a['ok'].value == b['ok'].value and a['held'].value == b['held'].value, (f, a['ok'].value, b['ok'].value, a['held'].value, b['held'].value)
        assert np.array_equal(a['mp'], b['mp']), (f, int((a['mp'] != b['mp']).sum()))
        assert np.abs(a['T'] - b['T']).max() <= 1e-6, f
        accepted += a['ok'].value
        if f == 5:
            assert a['ok'].value == 0
    assert accepted >= nb - 3
