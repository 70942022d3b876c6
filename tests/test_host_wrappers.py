"""What the single-call host-pointer entry points do before their kernels run (no GPU needed): the code and text of a bad argument, the
status and host-side output initialisation of an empty input, the projection matchers' limit of 8192 keypoints per frame, and SGS_ERR_CUDA --
never a CPU fallback -- for a valid call on a machine without a device.  The GPU tests check what the kernels then compute.

Every wrapper has a helper below that takes the sizes, builds well-formed host arrays and returns (status, host outputs); ``bad=True``
replaces one required argument by an invalid one."""
import ctypes as C

import numpy as np
import pytest

from pysgs import binding as B

V, F32, F64 = C.c_void_p, C.c_float, C.c_double
TOO_MANY = 'sgs_matcher_create: cur_cap 9000 exceeds the 8192 keypoints per frame the shared-memory grid supports'


def _p(a):
    return a.ctypes.data_as(V)


def _has_device():
    n = C.c_int(-1)
    return B.lib().sgs_device_count(C.byref(n)) == B.SGS_OK and n.value > 0


def _error():
    return B.lib().sgs_last_error().decode()


def _frame(n):
    rng = np.random.default_rng(n)
    k = np.zeros(n, B.KP_DTYPE)
    k['x'], k['y'] = rng.uniform(0, 640, n), rng.uniform(0, 480, n)
    return B.HostFrame(k, np.full(n, -1, np.float32), rng.integers(0, 256, (n, 32), dtype=np.uint8), 640, 480, 500.0, 500.0, 320.0, 240.0, 40.0,
                       1.2 ** np.arange(8))


def _camera():
    return B.make_camera(640, 480, dict(fx=500.0, fy=500.0, cx=320.0, cy=240.0, bf=40.0), 1.2 ** np.arange(8))


def _desc(n):
    return np.random.default_rng(n + 1).integers(0, 256, (n, 32), dtype=np.uint8)


T = np.eye(4, dtype=np.float32)
INV_SIGMA2 = np.ones(16, np.float32)


def hamming_pairs(n, bad=False):
    a, b, dist = _desc(n), _desc(n), np.full(n, 7, np.int32)
    return B.lib().sgs_hamming_pairs(_p(a), _p(b), -1 if bad else n, _p(dist), 0), dist


def hamming_bf(nq, nt=5, bad=False):
    q, t = _desc(nq), _desc(nt)
    idx, best, second = (np.full(nq, 7, np.int32) for _ in range(3))
    return B.lib().sgs_hamming_bf(_p(q), -1 if bad else nq, _p(t), nt, _p(idx), _p(best), _p(second), 0), idx


def lastframe(n, nlast, bad=False):
    fr = _frame(n)
    has, obs, octave = np.ones(nlast, np.uint8), np.zeros(nlast, np.uint8), np.zeros(nlast, np.int32)
    xyz, angle, mp, nm = np.ones((nlast, 3), np.float32), np.zeros(nlast, np.float32), np.full(n, -1, np.int32), C.c_int(7)
    rc = B.lib().sgs_match_project_lastframe(None if bad else C.byref(fr.c), _p(T), _p(T), nlast, _p(has), _p(xyz), _p(_desc(nlast)), _p(obs), _p(octave),
                                             _p(angle), F32(15), 0, 1, _p(mp), None, C.byref(nm), 0)
    return rc, nm.value


def keyframe(n, nkf, bad=False):
    fr = _frame(n)
    valid, xyz, angle = np.ones(nkf, np.uint8), np.ones((nkf, 3), np.float32), np.zeros(nkf, np.float32)
    dmin, dmax, mp, nm = np.zeros(nkf, np.float32), np.full(nkf, 10, np.float32), np.full(n, -1, np.int32), C.c_int(7)
    rc = B.lib().sgs_match_project_keyframe(None if bad else C.byref(fr.c), _p(T), nkf, _p(valid), _p(xyz), _p(_desc(nkf)), _p(angle), _p(dmin), _p(dmax),
                                            F32(3), 100, 1, _p(mp), C.byref(nm), 0)
    return rc, nm.value


def localmap(n, nmp, bad=False):
    fr = _frame(n)
    inview, obs, level = np.ones(nmp, np.uint8), np.zeros(nmp, np.uint8), np.zeros(nmp, np.int32)
    px, py, pxr, vcos = (np.zeros(nmp, np.float32) for _ in range(4))
    mp, mpo, nm = np.full(n, -1, np.int32), np.zeros(n, np.uint8), C.c_int(7)
    rc = B.lib().sgs_match_project_localmap(None if bad else C.byref(fr.c), nmp, _p(inview), _p(px), _p(py), _p(pxr), _p(level), _p(vcos), _p(_desc(nmp)),
                                            _p(obs), F32(1), F32(0.8), 0, _p(mp), _p(mpo), C.byref(nm), 0)
    return rc, nm.value


def fuse(n, nmp, bad=False):
    fr = _frame(n)
    valid, xyz, normal = np.ones(nmp, np.uint8), np.ones((nmp, 3), np.float32), np.ones((nmp, 3), np.float32)
    dmin, dmax, ow = np.zeros(nmp, np.float32), np.full(nmp, 10, np.float32), np.zeros(3, np.float32)
    best_idx, best_dist, nm = np.full(nmp, 7, np.int32), np.full(nmp, 7, np.int32), C.c_int(7)
    rc = B.lib().sgs_fuse_search(None if bad else C.byref(fr.c), _p(T), _p(ow), nmp, _p(valid), _p(xyz), _p(normal), _p(dmin), _p(dmax), _p(_desc(nmp)), F32(3),
                                 _p(INV_SIGMA2), 0, None, _p(best_idx), _p(best_dist), None, C.byref(nm), 0)
    return rc, nm.value, best_idx, best_dist


def search_init(n1, n2, bad=False):
    f1, f2 = _frame(n1), _frame(n2)
    prev, match12, nm = np.zeros((n1, 2), np.float32), np.full(n1, 7, np.int32), C.c_int(7)
    rc = B.lib().sgs_search_for_initialization(None if bad else C.byref(f1.c), C.byref(f2.c), _p(prev), 100, F32(0.9), 1, _p(match12), C.byref(nm), 0)
    return rc, nm.value, match12


def _bow_side(n):
    return np.arange(n, dtype=np.int32), np.ones(n, np.float64), np.ones(n, np.uint8), _desc(n), np.zeros(n, np.float32)


def bow_keyframes(n1, n2, bad=False):
    s1, s2 = _bow_side(n1), _bow_side(n2)
    match12, nm = np.full(n1, 7, np.int32), C.c_int(7)
    rc = B.lib().sgs_match_bow_keyframes(0 if bad else 1, n1, *map(_p, s1), n2, *map(_p, s2), F32(0.75), 1, None, None, None, None, None, None, None, None,
                                         None, 0, 0, _p(match12), C.byref(nm), 0)
    return rc, nm.value, match12


def bow_transform(n):
    word, node, weight = np.zeros(n, np.int32), np.zeros(n, np.int32), np.zeros(n, np.float64)
    return B.lib().sgs_bow_transform(None, _p(_desc(n)), n, 4, _p(word), _p(weight), _p(node)), word


def match_bow(nkf, nf, bad=False):
    k, f = _bow_side(nkf), _bow_side(nf)
    match_f, nm = np.full(nf, 7, np.int32), C.c_int(7)
    rc = B.lib().sgs_match_bow(nkf, *map(_p, k), nf, _p(f[0]), _p(f[1]), _p(f[3]), _p(f[4]), F32(0.75), 1, _p(match_f), None if bad else C.byref(nm), 0)
    return rc, nm.value, match_f


def pose_opt(n, bad=False):
    cam, fr = _camera(), _frame(n)
    has, xyz, tcw_in = np.ones(n, np.uint8), np.ones((n, 3), np.float32), T + 0.5
    tcw_out, outlier, nin = np.zeros(16, np.float32), np.full(n, 7, np.uint8), C.c_int(7)
    rc = B.lib().sgs_pose_optimization(None if bad else C.byref(cam), _p(tcw_in), n, _p(fr.keysUn), _p(fr.uRight), _p(has), _p(xyz), _p(INV_SIGMA2),
                                       _p(tcw_out), _p(outlier), C.byref(nin), 0)
    return rc, nin.value, tcw_out, tcw_in


def undistort(n, bad=False):
    xy, out, k = np.ones((n, 2), np.float32), np.zeros((n, 2), np.float32), np.array([0.1, 0, 0, 0, 0], np.float32)
    return B.lib().sgs_undistort_points(_p(xy), -1 if bad else n, F32(500), F32(500), F32(320), F32(240), _p(k), _p(out), 0), out


def frustum(n, bad=False):
    cam = _camera()
    xyz, normal, dmin, dmax = np.ones((n, 3), np.float32), np.ones((n, 3), np.float32), np.zeros(n, np.float32), np.full(n, 10, np.float32)
    inview, level, px, py, pxr, vcos = np.zeros(n, np.uint8), np.zeros(n, np.int32), *(np.zeros(n, np.float32) for _ in range(4))
    rc = B.lib().sgs_frustum(None if bad else C.byref(cam), _p(T), n, _p(xyz), _p(normal), _p(dmin), _p(dmax), F32(0.5), _p(inview), _p(px), _p(py), _p(pxr),
                             _p(level), _p(vcos), 0)
    return rc, inview


def dynreject(n, bad=False):
    cur, prev, F = np.ones((n, 2), np.float32), np.ones((n, 2), np.float32), np.eye(3).reshape(9)
    keep, nkeep, restored = np.zeros(n, np.uint8), C.c_int(7), C.c_int(7)
    rc = B.lib().sgs_dynreject(_p(cur), _p(prev), -1 if bad else n, _p(F), None, 0, 1, 1000, _p(keep), None, C.byref(nkeep), C.byref(restored), 0)
    return rc, nkeep.value, restored.value


def fundamental(n, bad=False):
    a, b, F = np.ones((n, 2), np.float32), np.ones((n, 2), np.float32), np.zeros(9, np.float64)
    return B.lib().sgs_fundamental_ransac(None if bad else _p(a), _p(b), n, F64(1.0), F64(0.99), 1000, _p(F), None, None, 0), F


# (call with a bad argument, the message it leaves)
BAD = {
    'hamming_pairs': (lambda: hamming_pairs(4, bad=True), 'sgs_hamming_pairs: bad argument'),
    'hamming_bf': (lambda: hamming_bf(4, bad=True), 'sgs_hamming_bf: negative size'),
    'lastframe': (lambda: lastframe(4, 4, bad=True), 'sgs_match_project_lastframe: bad argument'),
    'keyframe': (lambda: keyframe(4, 4, bad=True), 'sgs_match_project_keyframe: bad argument'),
    'localmap': (lambda: localmap(4, 4, bad=True), 'sgs_match_project_localmap: bad argument'),
    'fuse': (lambda: fuse(4, 4, bad=True), 'sgs_fuse_search: bad argument'),
    'search_init': (lambda: search_init(4, 4, bad=True), 'sgs_search_for_initialization: bad argument'),
    'bow_keyframes': (lambda: bow_keyframes(4, 4, bad=True), 'sgs_match_bow_keyframes: bad argument'),
    'bow_transform': (lambda: bow_transform(4), 'sgs_bow_transform: bad argument'),
    'match_bow': (lambda: match_bow(4, 4, bad=True), 'sgs_match_bow: bad argument'),
    'pose_opt': (lambda: pose_opt(4, bad=True), 'sgs_pose_optimization: bad argument'),
    'undistort': (lambda: undistort(4, bad=True), 'sgs_undistort_points: bad argument'),
    'frustum': (lambda: frustum(4, bad=True), 'sgs_frustum: bad argument'),
    'dynreject': (lambda: dynreject(4, bad=True), 'sgs_dynreject: bad argument'),
    'fundamental': (lambda: fundamental(20, bad=True), 'sgs_fundamental_ransac: bad argument'),
}


@pytest.mark.parametrize('name', sorted(BAD))
def test_bad_argument(name):
    call, message = BAD[name]
    assert call()[0] == B.SGS_ERR_INVALID
    assert _error() == message


def test_empty_inputs_return_without_the_device():
    assert hamming_pairs(0)[0] == B.SGS_OK
    assert hamming_bf(0)[0] == B.SGS_OK
    for matcher in (lastframe, keyframe, localmap):
        assert matcher(4, 0) == (B.SGS_OK, 0) and matcher(0, 4) == (B.SGS_OK, 0)
    rc, nm, best_idx, best_dist = fuse(0, 3)
    assert rc == B.SGS_OK and nm == 0 and (best_idx == -1).all() and (best_dist == 256).all()
    for rc, nm, match in (search_init(3, 0), bow_keyframes(3, 0)):
        assert rc == B.SGS_OK and nm == 0 and (match == -1).all()
    rc, nm, match_f = match_bow(0, 3)
    assert rc == B.SGS_OK and nm == 0 and (match_f == -1).all()
    rc, nin, tcw_out, tcw_in = pose_opt(0)
    assert rc == B.SGS_OK and nin == 0 and np.array_equal(tcw_out, tcw_in.reshape(16))
    assert undistort(0)[0] == B.SGS_OK
    assert frustum(0)[0] == B.SGS_OK
    # fewer than one pair is a bad argument, not an empty success
    assert fundamental(0)[0] == B.SGS_ERR_INVALID and _error() == 'sgs_fundamental_ransac: bad argument'


def test_dynreject_selects_the_device_before_an_empty_input():
    rc, nkeep, restored = dynreject(0)
    assert rc == (B.SGS_OK if _has_device() else B.SGS_ERR_CUDA)
    assert nkeep == 0 and restored == 0


@pytest.mark.parametrize('matcher', [lastframe, keyframe, localmap], ids=lambda m: m.__name__)
def test_matcher_keypoint_limit(matcher):
    assert matcher(9000, 4) == (B.SGS_ERR_UNSUPPORTED, 0)
    assert _error() == TOO_MANY


VALID = {
    'hamming_pairs': lambda: hamming_pairs(4), 'hamming_bf': lambda: hamming_bf(4), 'lastframe': lambda: lastframe(100, 50),
    'keyframe': lambda: keyframe(100, 50), 'localmap': lambda: localmap(100, 50), 'fuse': lambda: fuse(100, 50), 'search_init': lambda: search_init(100, 100),
    'bow_keyframes': lambda: bow_keyframes(100, 100), 'match_bow': lambda: match_bow(100, 100), 'pose_opt': lambda: pose_opt(100),
    'undistort': lambda: undistort(100), 'frustum': lambda: frustum(100), 'dynreject': lambda: dynreject(100), 'fundamental': lambda: fundamental(100),
}


@pytest.mark.parametrize('name', sorted(VALID))
def test_valid_call_without_device_fails_loudly(name):
    if _has_device():
        pytest.skip('a CUDA device is present')
    assert VALID[name]()[0] == B.SGS_ERR_CUDA
