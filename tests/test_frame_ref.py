"""The dynamic-feature rejection and the Frame glue pinned against the REFERENCE'S OWN src/Frame.cc (oracle/_ref/libframe_ref.so: Frame.cc and ORBextractor.cc
compiled unmodified from the reference tree against the real include/Frame.h; cv::calcOpticalFlowPyrLK / findFundamentalMat / undistortPoints resolve to the
oracle's restatements, each pinned against the real cv2 primitive by tests/golden/*.npz).  A stream of RGB-D frames with planted detector results goes through
the reference's RGB-D constructor (src/Frame.cc:129-198) -- extraction, RmDynamicPointWithSemanticAndGeometry (:430-612: LK to the previous image, the
previous-frame box filter and its `> 20` rule, findFundamentalMat, the hand-over of the detector's results, the 0.2 / 1.0 epipolar thresholds, the erase loop,
the restore-all guard, the FILE-SCOPE previous-frame state), UndistortKeyPoints, ComputeStereoFromRGBD, ComputeImageBounds, AssignFeaturesToGrid -- and the
same stream through the chain composed from the oracle's functions (what oracle/chain.cpp and the GPU tests compose).  Everything the Frame ends up with must be
identical bit for bit; so must GetFeaturesInArea (:354-407) and isInFrustum (:296-352) of the resulting Frame.

What this pins is the control flow and state handling the reference itself wrote, including three behaviours that are easy to get wrong:
  * the detector's flags and boxes are taken only when it reported at least one NON-person object (mvObjects2D, src/Frame.cc:482-491); otherwise the Frame's own
    flag is never written (uninitialised member; read as false here: the Frame is built in zeroed memory -- quirk Q12) and the previous-frame flag is cleared;
  * the previous-frame state lives at file scope and is only updated inside the rejection, which the first frame of a stream never runs: detections of frame 0
    do not filter the pairs of frame 1;
  * the restore-all guard restores the keypoints only when the frame has person boxes (with none, a frame may keep a handful of keypoints).
No device needed."""
import ctypes as C
import os

import numpy as np

import oracle as O
import refgolden as RG
from pysgs import synth

LIB = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'oracle', '_ref', 'libframe_ref.so')

W, H, NF = 640, 480, 1000
CAM = synth.TUM3
NODIST = np.zeros(5, np.float32)
TUM1_DIST = np.array([0.262383, -0.953104, -0.005358, 0.002628, 1.163314], np.float32)


class Det:
    """What Detector2D holds when Tracking builds the Frame (src/Detector2D.cc:52-88)."""

    def __init__(self, nobjects=0, have_rm=False, have_map=False, rm_boxes=(), map_boxes=()):
        self.nobjects, self.have_rm, self.have_map = nobjects, have_rm, have_map
        self.rm_boxes = np.asarray(rm_boxes, np.float32).reshape(-1, 4); self.map_boxes = np.asarray(map_boxes, np.float32).reshape(-1, 4)


def _lib():
    L = RG.load(LIB, __name__)
    L.ref_frame_push.restype = C.c_int; L.ref_frame_features_in_area.restype = C.c_int; L.ref_frame_is_in_frustum.restype = C.c_int
    return L


def run_reference(frames, depth, dets, dist5=NODIST, cam=CAM):
    L = _lib()
    L.ref_set_monotone_allocator(1)          # quadtree ties by creation order (quirk Q1, tests/test_orbextractor_ref.py)
    L.ref_frame_reset(NF, C.c_float(1.2), 8, 20, 7)
    K4 = np.array([cam['fx'], cam['fy'], cam['cx'], cam['cy']], np.float32)
    d = np.ascontiguousarray(depth, np.float32)
    out = []
    cap = 4 * NF
    for img, det in zip(frames, dets):
        img = np.ascontiguousarray(img, np.uint8)
        k = np.zeros(cap, O.KP_DTYPE); ku = np.zeros(cap, O.KP_DTYPE); ds = np.zeros((cap, 32), np.uint8)
        ur = np.zeros(cap, np.float32); dz = np.zeros(cap, np.float32); flags = np.zeros(8, np.int32); bounds = np.zeros(6, np.float32)
        n = L.ref_frame_push(RG.ptr(img), W, H, RG.ptr(d), RG.ptr(K4), RG.ptr(np.ascontiguousarray(dist5, np.float32)),
                             C.c_float(cam['bf']), C.c_float(40.0), det.nobjects, int(det.have_rm), int(det.have_map),
                             RG.ptr(det.rm_boxes), len(det.rm_boxes), RG.ptr(det.map_boxes), len(det.map_boxes),
                             RG.ptr(k), RG.ptr(ku), RG.ptr(ds), RG.ptr(ur), RG.ptr(dz), cap,
                             RG.ptr(flags), RG.ptr(bounds))
        assert 0 <= n <= cap
        out.append(dict(n=n, keys=k[:n].copy(), keys_un=ku[:n].copy(), desc=ds[:flags[4]].copy(), u_right=ur[:n].copy(), depth=dz[:n].copy(),
                        have_rm=int(flags[0]), have_map=int(flags[1]), pre_have=int(flags[2]), pre_nboxes=int(flags[3]), bounds=bounds.copy()))
    L.ref_set_monotone_allocator(0)
    return out, L


def run_oracle(frames, depth, dets, dist5=NODIST, cam=CAM):
    """The same stream through the oracle's functions, with the reference's state machine written out."""
    pre_img, pre_have, pre_boxes = None, False, np.zeros((0, 4), np.float32)
    out = []
    for img, det in zip(frames, dets):
        k, d = O.extract(img)
        have_rm = have_map = False                                   # the Frame's flags: untouched (zero) unless the detector hands them over
        keys, desc = k, d
        info = {}
        if pre_img is not None:
            cur = np.stack([k['x'], k['y']], 1).astype(np.float32)
            prev = O.lk_track(img, pre_img, cur)
            s1, s2 = O.select_static_pairs(cur, prev, pre_boxes, pre_have)
            F, _, _ = O.find_fundamental_ransac(s1, s2)
            if det.nobjects > 0:                                     # src/Frame.cc:482-491
                have_rm, have_map = det.have_rm, det.have_map
                pre_have = have_rm
            else:
                pre_have = False
            if have_rm:
                pre_boxes = det.rm_boxes
            _, keep, dist, restored = O.dynreject(cur, prev, F, det.rm_boxes if have_rm else None, have_rm, NF)
            info = dict(removed=int((keep == 0).sum()), restored=restored, pairs=len(s1))
            if restored:
                keys, desc = k, d                                    # swap(mvKeys, mvKeys_Temp): the descriptors were never replaced
            else:
                keys, desc = k[keep != 0], d[keep != 0]
        pre_img = img
        if dist5[0] == 0:
            keys_un = keys.copy()
        else:
            keys_un = keys.copy()
            und = O.undistort_points(np.stack([keys['x'], keys['y']], 1), cam['fx'], cam['fy'], cam['cx'], cam['cy'], dist5)
            keys_un['x'] = und[:, 0]; keys_un['y'] = und[:, 1]
        ur, dz = O.stereo_from_rgbd(keys, depth, cam['bf'], keys_un)
        out.append(dict(n=len(keys), keys=keys, keys_un=keys_un, desc=desc, u_right=ur, depth=dz, have_rm=int(have_rm), have_map=int(have_map),
                        pre_have=int(pre_have), pre_nboxes=len(pre_boxes), **info))
    return out


def compare(ref, orc):
    assert len(ref) == len(orc)
    for t, (r, o) in enumerate(zip(ref, orc)):
        assert r['n'] == o['n'], (t, r['n'], o['n'], o)
        assert r['keys'].tobytes() == o['keys'].tobytes(), t
        assert r['keys_un'].tobytes() == o['keys_un'].tobytes(), t
        assert np.array_equal(r['desc'], o['desc']), t
        assert r['u_right'].tobytes() == o['u_right'].tobytes() and r['depth'].tobytes() == o['depth'].tobytes(), t
        for key in ('have_rm', 'have_map', 'pre_have', 'pre_nboxes'):
            assert r[key] == o[key], (t, key, r[key], o[key])


def stream(n=4, seed=3):
    frames, boxes = synth.stream_s2(n, W, H, seed=seed)
    return frames, boxes, synth.depth_s1(W, H)


def test_static_scene_without_detections():
    frames, _, depth = stream()
    dets = [Det() for _ in frames]
    ref, _ = run_reference(frames, depth, dets)
    orc = run_oracle(frames, depth, dets)
    compare(ref, orc)
    assert all(o['removed'] > 0 for o in orc[1:]), 'the moving person must lose keypoints to the 1.0 px epipolar test'
    assert ref[0]['n'] > 900 and all(r['n'] < ref[0]['n'] + 200 for r in ref)


def test_person_boxes_thresholds_and_previous_frame_filter():
    frames, boxes, depth = stream(5)
    dets = [Det(nobjects=2, have_rm=True, have_map=True, rm_boxes=[boxes[t]], map_boxes=[boxes[t]]) for t in range(5)]
    ref, _ = run_reference(frames, depth, dets)
    orc = run_oracle(frames, depth, dets)
    compare(ref, orc)
    # frame 0 never runs the rejection: its detections do not reach the file-scope state, so frame 1 selects all pairs; from frame 2 on the filter is active
    assert ref[0]['pre_have'] == 0 and ref[0]['have_rm'] == 0 and ref[1]['pre_have'] == 1
    assert orc[1]['pairs'] == len(O.extract(frames[1])[0]) and orc[2]['pairs'] < len(O.extract(frames[2])[0])
    # the 0.2 px threshold inside the box removes more than the 1.0 px threshold did without boxes
    plain = run_oracle(frames, depth, [Det() for _ in frames])
    assert sum(o['removed'] for o in orc[1:]) > sum(o['removed'] for o in plain[1:])


def test_flags_are_taken_only_with_a_non_person_object():
    frames, boxes, depth = stream(4)
    # persons reported (flags + boxes set) but mvObjects2D empty in frames 1 and 3: the Frame keeps its own (zero) flags and clears the previous-frame flag
    dets = [Det(nobjects=0 if t in (1, 3) else 1, have_rm=True, have_map=True, rm_boxes=[boxes[t]], map_boxes=[boxes[t]]) for t in range(4)]
    ref, _ = run_reference(frames, depth, dets)
    orc = run_oracle(frames, depth, dets)
    compare(ref, orc)
    assert [r['have_rm'] for r in ref] == [0, 0, 1, 0] and [r['pre_have'] for r in ref] == [0, 0, 1, 0]
    assert ref[3]['pre_nboxes'] == 1, 'the stale boxes stay behind the cleared flag'
    # flag false with objects present: thresholds stay at 1.0 and the boxes are not recorded
    dets = [Det(nobjects=3, have_rm=False, have_map=True, rm_boxes=[boxes[t]], map_boxes=[boxes[t]]) for t in range(3)]
    ref, _ = run_reference(frames[:3], depth, dets)
    compare(ref, run_oracle(frames[:3], depth, dets))
    assert [r['have_map'] for r in ref] == [0, 1, 1] and all(r['pre_nboxes'] == 0 for r in ref)


def test_restore_all_guard_needs_person_boxes():
    # a jump in the stream: LK loses the points, nearly every keypoint fails the epipolar test
    frames, boxes, depth = stream(40)
    sel = [0, 1, 39]
    fr = frames[sel]
    whole = [[0.0, 0.0, float(W), float(H)]]
    dets = [Det(), Det(), Det(nobjects=1, have_rm=True, rm_boxes=whole)]
    ref, _ = run_reference(fr, depth, dets)
    orc = run_oracle(fr, depth, dets)
    compare(ref, orc)
    assert orc[2]['restored'] and ref[2]['n'] == len(O.extract(fr[2])[0]), 'fewer than nFeatures / 10 survivors with person boxes: every keypoint comes back'
    dets = [Det(), Det(), Det()]
    ref, _ = run_reference(fr, depth, dets)
    orc = run_oracle(fr, depth, dets)
    compare(ref, orc)
    assert not orc[2]['restored'] and ref[2]['n'] < NF // 10, 'without person boxes the guard does not fire'


def test_distorted_camera_undistort_bounds_and_stereo():
    frames, boxes, depth = stream(3)
    dets = [Det(nobjects=1, have_rm=True, rm_boxes=[boxes[t]]) for t in range(3)]
    ref, _ = run_reference(frames, depth, dets, dist5=TUM1_DIST)
    orc = run_oracle(frames, depth, dets, dist5=TUM1_DIST)
    compare(ref, orc)
    assert not np.array_equal(ref[2]['keys_un']['x'], ref[2]['keys']['x'])
    corners = O.undistort_points(np.array([[0, 0], [W, 0], [0, H], [W, H]], np.float32), CAM['fx'], CAM['fy'], CAM['cx'], CAM['cy'], TUM1_DIST)   # src/Frame.cc:686-714
    want = np.array([min(corners[0, 0], corners[2, 0]), max(corners[1, 0], corners[3, 0]), min(corners[0, 1], corners[1, 1]), max(corners[2, 1], corners[3, 1])], np.float32)
    assert ref[0]['bounds'][:4].tobytes() == want.tobytes()
    assert ref[0]['bounds'][4] == np.float32(64) / np.float32(want[1] - want[0]) and ref[0]['bounds'][5] == np.float32(48) / np.float32(want[3] - want[2])


def test_grid_queries_and_frustum_of_the_reference_frame():
    frames, boxes, depth = stream(2)
    dets = [Det(), Det(nobjects=1, have_rm=True, rm_boxes=[boxes[1]])]
    ref, L = run_reference(frames, depth, dets)
    orc = run_oracle(frames, depth, dets)
    compare(ref, orc)
    o = orc[1]
    sf = O.orb_tables(O.params())['scale']
    fa = O.FrameArrays(o['keys_un'], o['u_right'], o['desc'], W, H, CAM['fx'], CAM['fy'], CAM['cx'], CAM['cy'], CAM['bf'], sf)
    rng = np.random.RandomState(5)
    buf = np.zeros(o['n'] + 1, np.int32)
    total = 0
    for q in range(400):
        x, y = rng.uniform(-30, W + 30), rng.uniform(-30, H + 30)
        r = float(rng.choice([4.0, 7.5, 15.0, 40.0, 90.0]))
        lo, hi = (-1, -1) if q % 3 == 0 else (int(rng.randint(0, 4)), int(rng.randint(3, 8)))
        n = L.ref_frame_features_in_area(C.c_float(x), C.c_float(y), C.c_float(r), lo, hi, RG.ptr(buf), len(buf))
        got = O.features_in_area(fa, np.float32(x), np.float32(y), np.float32(r), lo, hi)
        assert n == len(got) and np.array_equal(buf[:n], got), q
        total += n
    assert total > 2000
    # isInFrustum (incl. PredictScale through logf) for points around the camera
    npt = 3000
    xyz = np.stack([rng.uniform(-3, 3, npt), rng.uniform(-2, 2, npt), rng.uniform(-0.5, 6, npt)], 1).astype(np.float32)
    ang = 0.05
    T = np.eye(4, dtype=np.float32); T[:3, :3] = np.array([[np.cos(ang), 0, np.sin(ang)], [0, 1, 0], [-np.sin(ang), 0, np.cos(ang)]], np.float32); T[:3, 3] = (0.1, -0.05, 0.2)
    Ow = -T[:3, :3].T @ T[:3, 3]
    nrm = (xyz - Ow) / np.linalg.norm(xyz - Ow, axis=1, keepdims=True) + rng.normal(0, 0.6, (npt, 3))      # mean viewing direction: some within 60 degrees, some not
    nrm = (nrm / np.linalg.norm(nrm, axis=1, keepdims=True)).astype(np.float32)
    dist = np.linalg.norm(xyz - Ow, axis=1).astype(np.float32)
    mx = (dist * rng.uniform(0.6, 3.0, npt)).astype(np.float32); mn = (mx / np.float32(1.2 ** 7)).astype(np.float32)
    out = np.zeros((npt, 6), np.float32)
    cnt = L.ref_frame_is_in_frustum(RG.ptr(T), C.c_float(0.5), npt, RG.ptr(xyz), RG.ptr(nrm),
                                    RG.ptr(mn), RG.ptr(mx), RG.ptr(out))
    cam = (CAM['fx'], CAM['fy'], CAM['cx'], CAM['cy'], CAM['bf'], 0.0, 0.0, float(W), float(H))
    want = O.is_in_frustum(T, cam, 8, float(O.logf(np.float32(1.2))), xyz, nrm, mn, mx, 0.5)
    assert cnt == int(want['inview'].sum()) and 100 < cnt < npt - 100
    iv = want['inview'] != 0
    assert np.array_equal(out[:, 0] != 0, iv)
    for col, key in ((1, 'proj_x'), (2, 'proj_y'), (3, 'proj_xr'), (5, 'view_cos')):
        assert out[iv, col].tobytes() == want[key][iv].tobytes(), key
    assert np.array_equal(out[iv, 4].astype(np.int32), want['level'][iv])
