"""The matchers of the tracking thread pinned against the REFERENCE'S OWN src/ORBmatcher.cc (oracle/_ref/liborbmatcher_ref.so: the file compiled unmodified
from the reference tree against stand-ins for cv::Mat / cv::KeyPoint and for the Frame / KeyFrame / MapPoint classes, recipe in oracle/Makefile):
`SearchByProjection(CurrentFrame, LastFrame, th, mono)` and `SearchByProjection(F, vpMapPoints, th)` run on the conflict-heavy random scenarios of the GPU
parity tests, and the oracle's restatement must return the same number of matches and the same map point for every keypoint.  This is what makes the
matcher control flow (window search, best / second-best with the ratio test, level gates, stereo gate, rotation histogram, claim rules) a pinned part of
the oracle rather than the builder's reading of it.  The cv::Mat arithmetic inside the stand-in follows the rules probed with cv2 (tests/golden/frustum.npz).
No device needed.  Skipped only when the library was never built (the reference tree is absent AND no prebuilt copy travelled)."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle as O
import refgolden as RG
import scenarios as S

LIB = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'oracle', '_ref', 'liborbmatcher_ref.so')


def _lib():
    L = RG.load(LIB, __name__)
    L.ref_search_by_projection_last.restype = C.c_int
    L.ref_search_by_projection_local.restype = C.c_int
    L.ref_descriptor_distance.restype = C.c_int
    return L


def _p(a):
    return RG.ptr(a) if a is not None else None


def _cam(s):
    c = s['cam']
    return np.array([c['fx'], c['fy'], c['cx'], c['cy'], c['bf'], 0, 0, s['w'], s['h']], np.float32)


def _frame(s):
    c = s['cam']
    return O.FrameArrays(s['kps'], s['uright'], s['desc'], s['w'], s['h'], c['fx'], c['fy'], c['cx'], c['cy'], c['bf'], s['sf'])


def ref_last(L, s, th, mono, check_ori, cur_mp=None, cur_obs=None):
    n = len(s['kps'])
    kps = np.ascontiguousarray(s['kps'], O.KP_DTYPE); ur = np.ascontiguousarray(s['uright'], np.float32); d = np.ascontiguousarray(s['desc'], np.uint8)
    sf = np.ascontiguousarray(s['sf'], np.float32); cam = _cam(s)
    Tc = np.ascontiguousarray(s['Tcw_cur'], np.float32).reshape(16); Tl = np.ascontiguousarray(s['Tcw_last'], np.float32).reshape(16)
    has = np.ascontiguousarray(s['last_has'], np.uint8); xyz = np.ascontiguousarray(s['last_xyz'], np.float32); ld = np.ascontiguousarray(s['last_desc'], np.uint8)
    lo = np.ascontiguousarray(s['last_obs'], np.uint8); loct = np.ascontiguousarray(s['last_oct'], np.int32); la = np.ascontiguousarray(s['last_angle'], np.float32)
    mp = np.full(n, -1, np.int32) if cur_mp is None else np.ascontiguousarray(cur_mp, np.int32).copy()
    ob = None if cur_obs is None else np.ascontiguousarray(cur_obs, np.uint8)
    nm = L.ref_search_by_projection_last(n, _p(kps), _p(ur), _p(d), _p(cam), len(sf), _p(sf), _p(Tc), _p(Tl), len(has), _p(has), _p(xyz), _p(ld), _p(lo), _p(loct), _p(la),
                                         C.c_float(th), int(mono), int(check_ori), _p(mp), _p(ob))
    return nm, mp


@pytest.mark.parametrize('seed', range(6))
@pytest.mark.parametrize('th', [15.0, 30.0])
def test_search_by_projection_last_equals_the_reference(seed, th):
    L = _lib()
    s = S.random_lastframe_scenario(seed, n_cur=1000 + 37 * seed, n_last=900 + 53 * seed, conflict=[0.0, 0.3, 0.6][seed % 3], mono=(seed == 5))
    fo = _frame(s)
    args = (s['Tcw_cur'], s['Tcw_last'], s['last_has'], s['last_xyz'], s['last_desc'], s['last_obs'], s['last_oct'], s['last_angle'], th)
    for check_ori in (True, False):
        nm_o, mp_o, _ = O.search_by_projection_last(fo, *args, mono=s['mono'], check_ori=check_ori)
        nm_r, mp_r = ref_last(L, s, th, s['mono'], check_ori)
        assert nm_r == nm_o, (seed, th, check_ori, nm_r, nm_o)
        assert np.array_equal(mp_r, mp_o)
        assert nm_o > 50


def test_search_by_projection_last_with_preexisting_matches():
    L = _lib()
    s = S.random_lastframe_scenario(7)
    fo = _frame(s)
    rng = np.random.RandomState(1)
    pre = np.full(len(s['kps']), -1, np.int32); m = rng.rand(len(pre)) < 0.3; pre[m] = 5
    pre_obs = (rng.rand(len(pre)) < 0.5).astype(np.uint8)
    args = (s['Tcw_cur'], s['Tcw_last'], s['last_has'], s['last_xyz'], s['last_desc'], s['last_obs'], s['last_oct'], s['last_angle'], 15.0)
    nm_o, mp_o, _ = O.search_by_projection_last(fo, *args, cur_mp=pre, cur_mp_obs=pre_obs)
    nm_r, mp_r = ref_last(L, s, 15.0, False, True, cur_mp=pre, cur_obs=pre_obs)
    assert nm_r == nm_o and np.array_equal(mp_r, mp_o)


@pytest.mark.parametrize('seed', range(5))
def test_search_by_projection_local_equals_the_reference(seed):
    L = _lib()
    s = S.random_localmap_scenario(seed, n_cur=1000, n_mp=2500 + 100 * seed, conflict=[0.2, 0.5][seed % 2])
    fo = _frame(s)
    n = len(s['kps'])
    kps = np.ascontiguousarray(s['kps'], O.KP_DTYPE); ur = np.ascontiguousarray(s['uright'], np.float32); d = np.ascontiguousarray(s['desc'], np.uint8)
    sf = np.ascontiguousarray(s['sf'], np.float32); cam = _cam(s)
    for th, ratio in ((3.0, 0.8), (1.0, 0.8), (5.0, 0.6)):
        a = (s['inview'], s['projx'], s['projy'], s['projxr'], s['level'], s['viewcos'], s['mp_desc'], s['mp_obs'], th, ratio, s['f_mp'], s['f_obs'])
        nm_o, mp_o, ob_o, _ = O.search_by_projection_local(fo, *a, id_base=7)
        mp = np.ascontiguousarray(s['f_mp'], np.int32).copy(); ob = np.ascontiguousarray(s['f_obs'], np.uint8).copy()
        arrs = [np.ascontiguousarray(s['inview'], np.uint8), np.ascontiguousarray(s['projx'], np.float32), np.ascontiguousarray(s['projy'], np.float32),
                np.ascontiguousarray(s['projxr'], np.float32), np.ascontiguousarray(s['level'], np.int32), np.ascontiguousarray(s['viewcos'], np.float32),
                np.ascontiguousarray(s['mp_desc'], np.uint8), np.ascontiguousarray(s['mp_obs'], np.uint8)]
        nm_r = L.ref_search_by_projection_local(n, _p(kps), _p(ur), _p(d), _p(cam), len(sf), _p(sf), len(arrs[0]), *[_p(x) for x in arrs], C.c_float(th), C.c_float(ratio), 7,
                                                _p(mp), _p(ob))
        assert nm_r == nm_o, (seed, th, nm_r, nm_o)
        assert np.array_equal(mp, mp_o) and np.array_equal(ob, ob_o)
        assert nm_o > 100


def test_descriptor_distance_equals_the_reference():
    L = _lib()
    rng = np.random.RandomState(3)
    a = rng.randint(0, 256, (200, 32)).astype(np.uint8); b = rng.randint(0, 256, (200, 32)).astype(np.uint8)
    for i in range(200):
        assert L.ref_descriptor_distance(_p(a[i]), _p(b[i])) == O.hamming(a[i], b[i])


@pytest.mark.parametrize('seed', range(4))
def test_relocalisation_search_equals_the_reference(seed):
    """SearchByProjection(Frame&, KeyFrame*, sAlreadyFound, th, ORBdist) (src/ORBmatcher.cc:1474-1601) incl. MapPoint::PredictScale through libm's logf."""
    L = _lib(); L.ref_search_by_projection_kf.restype = C.c_int
    s = S.keyframe_scenario(seed, n_cur=900 + 50 * seed, n_kf=800 + 70 * seed, conflict=[0.2, 0.5][seed % 2])
    fo = _frame(s)
    n = len(s['kps'])
    kps = np.ascontiguousarray(s['kps'], O.KP_DTYPE); ur = np.ascontiguousarray(s['uright'], np.float32); d = np.ascontiguousarray(s['desc'], np.uint8)
    sf = np.ascontiguousarray(s['sf'], np.float32); cam = _cam(s); Tc = np.ascontiguousarray(s['Tcw_cur'], np.float32).reshape(16)
    a = [np.ascontiguousarray(s['kf_valid'], np.uint8), np.ascontiguousarray(s['last_xyz'], np.float32), np.ascontiguousarray(s['last_desc'], np.uint8),
         np.ascontiguousarray(s['last_angle'], np.float32), np.ascontiguousarray(s['min_dist'], np.float32), np.ascontiguousarray(s['max_dist'], np.float32)]
    for th, orb_dist, ori in ((10.0, 100, True), (3.0, 64, True), (10.0, 100, False)):
        nm_o, mp_o, _ = O.search_by_projection_kf(fo, s['Tcw_cur'], *a, th, orb_dist, ori, cur_mp=s['cur_mp'])
        mp = np.ascontiguousarray(s['cur_mp'], np.int32).copy()
        nm_r = L.ref_search_by_projection_kf(n, _p(kps), _p(ur), _p(d), _p(cam), len(sf), _p(sf), _p(Tc), len(a[0]), *[_p(x) for x in a], C.c_float(th), orb_dist, int(ori), _p(mp))
        assert nm_r == nm_o, (seed, th, nm_r, nm_o)
        assert np.array_equal(mp, mp_o)
        assert nm_o > 30


@pytest.mark.parametrize('seed,window,ori', [(1, 100, True), (2, 100, False), (3, 40, True)])
def test_search_for_initialization_equals_the_reference(seed, window, ori):
    import test_match_init as TI
    L = _lib(); L.ref_search_for_initialization.restype = C.c_int
    s = TI.init_scenario(seed)
    nm_o, m_o, prev_o = O.search_for_initialization(s['f1'], s['f2'], s['prev'], window, 0.9, ori)
    c = s['cam']; cam = np.array([c['fx'], c['fy'], c['cx'], c['cy'], c['bf'], 0, 0, 640, 480], np.float32); sf = np.ascontiguousarray(s['sf'], np.float32)
    k1 = np.ascontiguousarray(s['k1'], O.KP_DTYPE); k2 = np.ascontiguousarray(s['k2'], O.KP_DTYPE)
    d1 = np.ascontiguousarray(s['d1'], np.uint8); d2 = np.ascontiguousarray(s['d2'], np.uint8)
    prev = np.ascontiguousarray(s['prev'], np.float32).copy(); m = np.zeros(len(k1), np.int32)
    nm_r = L.ref_search_for_initialization(len(k1), _p(k1), _p(d1), len(k2), _p(k2), _p(d2), _p(cam), len(sf), _p(sf), _p(prev), window, C.c_float(0.9), int(ori), _p(m))
    assert nm_r == nm_o and np.array_equal(m, m_o) and np.array_equal(prev, prev_o)
    assert nm_o > 40


@pytest.mark.parametrize('seed', range(3))
def test_search_by_bow_equals_the_reference(seed):
    """Both SearchByBoW forms (src/ORBmatcher.cc:159-290, :524-657) on feature vectors built like TemplatedVocabulary::transform builds them."""
    L = _lib(); L.ref_search_by_bow.restype = C.c_int; L.ref_search_by_bow_kfkf.restype = C.c_int
    voc = S.random_vocabulary(4 + seed, k=10, L=3)
    V = O.Vocabulary(voc['k'], voc['L'], voc['parent'], voc['desc'], voc['weight'])
    sc = S.bow_pair_scenario(2 + seed, voc, n_kf=900, n_f=1000)
    _, wk, nk = V.transform(sc['kf_desc'], 1); _, wf, nf = V.transform(sc['f_desc'], 1)
    nk = np.ascontiguousarray(nk, np.int32); nf = np.ascontiguousarray(nf, np.int32); wk = np.ascontiguousarray(wk, np.float64); wf = np.ascontiguousarray(wf, np.float64)
    kd = np.ascontiguousarray(sc['kf_desc'], np.uint8); fd = np.ascontiguousarray(sc['f_desc'], np.uint8)
    ka = np.ascontiguousarray(sc['kf_angle'], np.float32); fa = np.ascontiguousarray(sc['f_angle'], np.float32); kv = np.ascontiguousarray(sc['kf_valid'], np.uint8)
    for ori in (False, True):
        nm_o, m_o = O.search_by_bow(nk, wk, kv, kd, ka, nf, wf, fd, fa, 0.7, ori)
        m = np.zeros(len(nf), np.int32)
        nm_r = L.ref_search_by_bow(len(nk), _p(nk), _p(wk), _p(kv), _p(kd), _p(ka), len(nf), _p(nf), _p(wf), _p(fd), _p(fa), C.c_float(0.7), int(ori), _p(m))
        assert nm_r == nm_o and np.array_equal(m, m_o) and nm_o > 50
        fv = (np.random.RandomState(seed).rand(len(nf)) < 0.85).astype(np.uint8)
        nm_o, m_o = O.search_by_bow_kfkf(nk, wk, kv, kd, ka, nf, wf, fv, fd, fa, 0.8, ori)
        m1 = np.zeros(len(nk), np.int32)
        nm_r = L.ref_search_by_bow_kfkf(len(nk), _p(nk), _p(wk), _p(kv), _p(kd), _p(ka), len(nf), _p(nf), _p(wf), _p(fv), _p(fd), _p(fa), C.c_float(0.8), int(ori), _p(m1))
        assert nm_r == nm_o and np.array_equal(m1, m_o) and nm_o > 50


@pytest.mark.parametrize('only,ori', [(False, False), (True, False), (False, True)])
def test_search_for_triangulation_equals_the_reference(only, ori):
    """SearchForTriangulation + CheckDistEpipolarLine (src/ORBmatcher.cc:659-827, :140-157); the epipole is computed by the reference's own lines from the poses."""
    L = _lib(); L.ref_search_for_triangulation.restype = C.c_int
    f32 = np.float32
    voc = S.random_vocabulary(6, k=6, L=2)
    V = O.Vocabulary(voc['k'], voc['L'], voc['parent'], voc['desc'], voc['weight'])
    rs = np.random.RandomState(2)
    n1, n2 = 420, 460
    s = S.bow_pair_scenario(11, voc, n_kf=n1, n_f=n2, flips=25)
    d1b = np.unpackbits(s['kf_desc'], axis=1).astype(np.int16); d2b = np.unpackbits(s['f_desc'], axis=1).astype(np.int16)
    src = np.array([int(np.argmin(np.abs(d1b - d2b[j]).sum(1))) for j in range(n2)])
    xy1 = np.c_[rs.uniform(20, 620, n1), rs.uniform(20, 460, n1)].astype(f32)
    xy2 = np.c_[xy1[src, 0] + rs.uniform(-40, 40, n2), xy1[src, 1] + rs.normal(0, 1.5, n2)].astype(f32)
    sf = S.scale_factors().astype(f32); sigma2 = (sf * sf).astype(f32)
    _, w1, nd1 = V.transform(s['kf_desc'], 1); _, w2, nd2 = V.transform(s['f_desc'], 1)
    k1 = dict(node=nd1, weight=w1, free=(rs.rand(n1) < 0.8).astype(np.uint8), stereo=(rs.rand(n1) < 0.5).astype(np.uint8), desc=s['kf_desc'], xy=xy1, angle=s['kf_angle'])
    k2 = dict(node=nd2, weight=w2, free=(rs.rand(n2) < 0.8).astype(np.uint8), stereo=(rs.rand(n2) < 0.5).astype(np.uint8), desc=s['f_desc'], xy=xy2,
              octave=rs.randint(0, 8, n2).astype(np.int32), angle=s['f_angle'])
    F12 = np.array([[0, 0, 0], [0, 0, -1], [0, 1, 0]], f32)
    cam = np.array([535.4, 539.2, 320.1, 247.6, 40.0, 0, 0, 640, 480], f32)
    cw = np.array([0.31, -0.07, 2.5], f32)
    # the reference's lines :666-672 with KF2 at the identity: C2 = R2w*Cw + t2w = Cw (small-matrix gemm: exact here), invz = 1.0f / C2z, ex = fx*C2x*invz + cx
    invz = f32(1.0) / cw[2]
    ex = f32(f32(f32(cam[0] * cw[0]) * invz) + cam[2]); ey = f32(f32(f32(cam[1] * cw[1]) * invz) + cam[3])
    nm_o, m_o = O.search_for_triangulation(k1, k2, F12, float(ex), float(ey), sigma2, sf, only, ori)
    a = [np.ascontiguousarray(k1['node'], np.int32), np.ascontiguousarray(k1['weight'], np.float64), np.ascontiguousarray(k1['free'], np.uint8), np.ascontiguousarray(k1['stereo'], np.uint8),
         np.ascontiguousarray(k1['desc'], np.uint8), np.ascontiguousarray(k1['xy'], f32), np.ascontiguousarray(k1['angle'], f32)]
    b = [np.ascontiguousarray(k2['node'], np.int32), np.ascontiguousarray(k2['weight'], np.float64), np.ascontiguousarray(k2['free'], np.uint8), np.ascontiguousarray(k2['stereo'], np.uint8),
         np.ascontiguousarray(k2['desc'], np.uint8), np.ascontiguousarray(k2['xy'], f32), np.ascontiguousarray(k2['octave'], np.int32), np.ascontiguousarray(k2['angle'], f32)]
    m = np.zeros(n1, np.int32)
    nm_r = L.ref_search_for_triangulation(n1, *[_p(x) for x in a], n2, *[_p(x) for x in b], _p(F12.reshape(9).copy()), _p(cw), _p(cam), len(sf), _p(sigma2), _p(sf), int(only), int(ori), _p(m))
    assert nm_r == nm_o, (nm_r, nm_o)
    assert np.array_equal(m, m_o) and nm_o > 5


@pytest.mark.parametrize('seed,ncur,nmp,th', [(0, 900, 1200, 10), (1, 1000, 1500, 10), (2, 800, 900, 4)])
def test_search_by_projection_sim3_equals_the_reference(seed, ncur, nmp, th):
    """SearchByProjection(pKF, Scw, vpPoints, vpMatched, th) (src/ORBmatcher.cc:292-405): the order-dependent claims of the loop-closing search.  Scw has scale 1
    (RGB-D); the reference's own decomposition (row norm, division, -Rcw.t()*tcw) runs inside the call -- the test requires that the row norm rounds to 1.0f so
    that the Mat / scalar division (not pinned by the stand-in) is the identity."""
    import test_match_sim3 as TS
    L = _lib(); L.ref_search_by_projection_sim3.restype = C.c_int
    f32 = np.float32
    s, _, nrm, matched = TS.sim3_inputs(seed, ncur, nmp)
    T = np.ascontiguousarray(s['Tcw_cur'], f32)
    R = T[:3, :3]; t = T[:3, 3]
    assert f32(np.sqrt(np.dot(R[0].astype(np.float64), R[0].astype(np.float64)))) == f32(1.0)
    Ow = np.array([f32(-(float(R[0, r]) * float(t[0]) + float(R[1, r]) * float(t[1]) + float(R[2, r]) * float(t[2]))) for r in range(3)], f32)      # -Rcw.t()*tcw, double accumulator
    fo = _frame(s)
    nm_o, m_o = O.search_by_projection_sim3(fo, T, Ow, s['kf_valid'], s['last_xyz'], nrm, s['min_dist'], s['max_dist'], s['last_desc'], float(th), matched)
    kps = np.ascontiguousarray(s['kps'], O.KP_DTYPE); ur = np.ascontiguousarray(s['uright'], f32); d = np.ascontiguousarray(s['desc'], np.uint8)
    sf = np.ascontiguousarray(s['sf'], f32); cam = _cam(s)
    a = [np.ascontiguousarray(s['kf_valid'], np.uint8), np.ascontiguousarray(s['last_xyz'], f32), np.ascontiguousarray(nrm, f32), np.ascontiguousarray(s['min_dist'], f32),
         np.ascontiguousarray(s['max_dist'], f32), np.ascontiguousarray(s['last_desc'], np.uint8)]
    m = np.ascontiguousarray(matched, np.int32).copy()
    nm_r = L.ref_search_by_projection_sim3(len(kps), _p(kps), _p(ur), _p(d), _p(cam), len(sf), _p(sf), _p(T.reshape(16).copy()), len(a[0]), *[_p(x) for x in a], int(th), _p(m))
    assert nm_r == nm_o, (nm_r, nm_o)
    assert np.array_equal(m, m_o) and nm_o > 20


def _fuse_inputs(seed, ncur, nmp):
    s = S.keyframe_scenario(seed, n_cur=ncur, n_kf=nmp, conflict=0.3)
    rs = np.random.RandomState(seed + 7)
    T = np.ascontiguousarray(s['Tcw_cur'], np.float32)
    R = T[:3, :3]; t = T[:3, 3]
    Ow = np.array([np.float32(-(float(R[0, r]) * float(t[0]) + float(R[1, r]) * float(t[1]) + float(R[2, r]) * float(t[2]))) for r in range(3)], np.float32)
    to = s['last_xyz'].astype(np.float64) - Ow.astype(np.float64); d = np.linalg.norm(to, axis=1)
    nrm = to / np.maximum(d[:, None], 1e-9) + rs.normal(0, 0.6, (nmp, 3)); nrm = (nrm / np.linalg.norm(nrm, axis=1, keepdims=True)).astype(np.float32)
    return s, T, Ow, nrm, rs


@pytest.mark.parametrize('seed,ncur,nmp,th,sim3', [(1, 1000, 1000, 3.0, 0), (2, 1500, 3000, 3.0, 0), (3, 400, 2000, 5.0, 0), (4, 1000, 2000, 4.0, 1), (6, 900, 1500, 4.0, 1)])
def test_fuse_equals_the_reference(seed, ncur, nmp, th, sim3):
    """Both Fuse forms (src/ORBmatcher.cc:829-980, :982-1104): the feature every map point is fused onto, read back from the reference's side effects
    (AddObservation / Replace / vpReplacePoint), must be the oracle's best feature whenever its distance is <= TH_LOW, and nFused the number of those."""
    L = _lib(); L.ref_fuse.restype = C.c_int
    f32 = np.float32
    s, T, Ow, nrm, rs = _fuse_inputs(seed, ncur, nmp)
    sf = np.ascontiguousarray(s['sf'], f32); inv_s2 = (1.0 / (sf * sf)).astype(f32)
    if sim3:
        assert f32(np.sqrt(np.dot(T[0, :3].astype(np.float64), T[0, :3].astype(np.float64)))) == f32(1.0)       # Scw / scw is the identity (see the Sim3 projection test)
    fo = _frame(s)
    bi_o, bd_o = O.fuse_search(fo, T, Ow, s['kf_valid'], s['last_xyz'], nrm, s['min_dist'], s['max_dist'], s['last_desc'], th, inv_s2, sim3_variant=sim3)
    fused_o = (bi_o >= 0) & (bd_o <= 50)
    kps = np.ascontiguousarray(s['kps'], O.KP_DTYPE); ur = np.ascontiguousarray(s['uright'], f32); d = np.ascontiguousarray(s['desc'], np.uint8); cam = _cam(s)
    a = [np.ascontiguousarray(s['kf_valid'], np.uint8), np.ascontiguousarray(s['last_xyz'], f32), np.ascontiguousarray(nrm, f32), np.ascontiguousarray(s['min_dist'], f32),
         np.ascontiguousarray(s['max_dist'], f32), np.ascontiguousarray(s['last_desc'], np.uint8)]
    nobs = rs.randint(0, 5, nmp).astype(np.int32)
    kf_obs = np.where(rs.rand(ncur) < 0.3, rs.randint(0, 5, ncur), -1).astype(np.int32)       # some features of the key frame already hold a map point
    best = np.zeros(nmp, np.int32)
    nf = L.ref_fuse(len(kps), _p(kps), _p(ur), _p(d), _p(cam), len(sf), _p(sf), _p(T.reshape(16).copy()), _p(Ow), _p(T.reshape(16).copy()) if sim3 else None, nmp,
                    *[_p(x) for x in a], _p(nobs), _p(kf_obs), C.c_float(th), _p(inv_s2), _p(best))
    assert nf == int(fused_o.sum()), (nf, int(fused_o.sum()))
    assert np.array_equal(best >= 0, fused_o)
    assert np.array_equal(best[fused_o], bi_o[fused_o])
    assert nf > 10
