"""The pose chain -- what sgs_tracker_pose_chain_device computes after the front end: the rest of Tracking::TrackWithMotionModel (wide-window retry,
PoseOptimization, outlier discard) and Tracking::TrackLocalMap (UpdateLocalPoints, SearchLocalPoints with its seen / bad exclusions and isInFrustum,
SearchByProjection(F, local points, th), PoseOptimization, mnMatchesInliers) -- pinned against the REFERENCE'S OWN tracking front end
(oracle/_ref/libtracking_ref.so: src/Tracking.cc, Frame.cc, MapPoint.cc, ORBmatcher.cc, Optimizer.cc + vendored g2o, Converter.cc compiled unmodified from the
reference tree against the real Tracking.h / Frame.h / MapPoint.h; oracle/Makefile target ref_tracking).  The checker of the GPU chain is the composition of
oracle functions in tests/test_gpu_pose_chain.py (oracle_chain): here that same function runs on CPU-extracted frames and must give, for every frame, the same
map-point assignment per keypoint after each half, the same outlier flags, the same mnMatchesInliers, the same accept / reject decisions and the same poses as
the reference's code does on the object graph the arrays describe.  Where the reference bails out early (fewer than 20 matches even at 2 th: its caller would
relocalise) the device chain keeps going; those frames are compared up to that point.  No device needed."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle as O
import refgolden as RG
from pysgs import binding as B
from pysgs import synth

LIB = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'oracle', '_ref', 'libtracking_ref.so')
W, H, TH = 640, 480, 15.0


def _p(a):
    return RG.ptr(a)


def reference_chain(camv, sf, isig, cur, Tc, m, ti, f, lm, pc, lib=None):
    L = C.CDLL(lib) if lib else RG.load(LIB, __name__)
    n = cur.c.N
    xy = np.ascontiguousarray(np.stack([cur.keysUn['x'], cur.keysUn['y']], 1), np.float32)
    octv = np.ascontiguousarray(cur.keysUn['octave'], np.int32); ang = np.ascontiguousarray(cur.keysUn['angle'], np.float32)
    out = dict(ok1=C.c_int32(), T1=np.zeros(16, np.float32), mp1=np.zeros(n, np.int32), ok2=C.c_int32(), T2=np.zeros(16, np.float32), mp2=np.zeros(n, np.int32),
               outl=np.zeros(n, np.uint8), inl=C.c_int32())
    nl = lm['n']
    a = lambda x, dt: np.ascontiguousarray(x, dt)
    keep = [a(ti['lxyz'][f, :m], np.float32), a(ti['ldesc'][f, :m], np.uint8), a(ti['lflags'][f, :m], np.uint8), a(ti['loct'][f, :m], np.int32), a(ti['lang'][f, :m], np.float32),
            a(ti['T'][f], np.float32), a(lm['lid'][:max(m, 1)], np.int32)]
    lmk = [a(lm['xyz'][:nl], np.float32), a(lm['nrm'][:nl], np.float32), a(lm['mn'][:nl], np.float32), a(lm['mx'][:nl], np.float32), a(lm['dsc'][:nl], np.uint8),
           a(lm['valid'][:nl], np.uint8), a(lm['obs'][:nl], np.uint8)]
    L.ref_track_motion_and_local_map(_p(camv), _p(a(sf, np.float32)), _p(isig), 8, n, _p(xy), _p(octv), _p(ang), _p(cur.uRight), _p(cur.desc), _p(a(Tc, np.float32)),
                                     m, *[_p(x) for x in keep], nl, *[_p(x) for x in lmk], pc,
                                     C.byref(out['ok1']), _p(out['T1']), _p(out['mp1']), C.byref(out['ok2']), _p(out['T2']), _p(out['mp2']), _p(out['outl']), C.byref(out['inl']))
    return out


@pytest.mark.parametrize('seed,mono_every', [(11, 0), (23, 7)])
def test_pose_chain_composition_equals_the_reference_tracking_code(seed, mono_every):
    import bench
    from test_gpu_pose_chain import oracle_chain
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
    ti['lflags'][:, 9::23] |= 4                                         # some last-frame points are bad
    if mono_every:
        ti['ur'][:, ::mono_every] = -1.0                                # keypoints without depth: monocular observations in both searches and both optimisations
    assert np.array_equal(ti['T'], np.tile(np.eye(4, dtype=np.float32).reshape(1, 16), (nb, 1)))     # the driver's velocity trick needs identity last poses
    Tc = ti['T'].copy()

    def rot(axis, ang):
        c, s_ = np.cos(ang), np.sin(ang)
        R = np.eye(4, dtype=np.float32)
        if axis == 'y': R[0, 0] = c; R[0, 2] = s_; R[2, 0] = -s_; R[2, 2] = c
        else: R[1, 1] = c; R[1, 2] = -s_; R[2, 1] = s_; R[2, 2] = c
        return R.reshape(16)
    Tc[3] = rot('y', 60.0 / camd['fx']); Tc[7] = rot('x', -58.0 / camd['fy']); Tc[9] = rot('y', 6.0 / camd['fx'])
    ti['ln'][5] = 0; ti['ln'][3] = 300; ti['ln'][7] = 300
    ti['Tc'] = Tc
    rng = np.random.default_rng(seed)
    isig = np.zeros(16, np.float32); isig[:8] = 1.0 / (sf.astype(np.float32) ** 2)
    camv = np.array([camd['fx'], camd['fy'], camd['cx'], camd['cy'], camd['bf'], cam.min_x, cam.min_y, cam.max_x, cam.max_y], np.float32)
    full = bailed = added = retried = 0
    for f in range(nb):
        n = int(cnt[f]); m = int(ti['ln'][f])
        cur = O.FrameArrays(kps[f, :n], ti['ur'][f, :n], desc[f, :n], W, H, camd['fx'], camd['fy'], camd['cx'], camd['cy'], camd['bf'], sf)
        lm = bench.make_local_map(f, kps[f], desc[f], n, ti, mcap, camd, sf, rng, W, H)
        # one object per point in the reference: a local-map point that IS a last-frame point carries that point's flags and position
        for j in np.nonzero(lm['lid'][:m] >= 0)[0]:
            l = lm['lid'][j]
            lm['xyz'][l] = ti['lxyz'][f, j]; lm['obs'][l] = (ti['lflags'][f, j] >> 1) & 1; lm['valid'][l] = 0 if ti['lflags'][f, j] & 4 else 1
        fl = ti['lflags'][f, :m]
        nm0, mp0, _ = O.search_by_projection_last(cur, Tc[f].reshape(4, 4), ti['T'][f].reshape(4, 4), fl & 1, ti['lxyz'][f, :m], ti['ldesc'][f, :m], (fl >> 1) & 1,
                                                  ti['loct'][f, :m], ti['lang'][f, :m], TH)
        r = oracle_chain(f, cur, int(nm0), mp0.copy(), ti, lm, camv, camd, sf, isig, TH)
        g = reference_chain(camv, sf, isig, cur, Tc[f], m, ti, f, lm, pc)
        st = r['stats']
        retried += int(st[1])
        # the first half recomputed with the oracle's functions, to compare the assignments the reference holds when TrackWithMotionModel returns (the counter the
        # reference calls nmatches also counts assignments that overwrote a temporal point, so it is not the number of keypoints holding a point)
        mpA = mp0.copy()
        if nm0 < 20:
            _, mpA, _ = O.search_by_projection_last(cur, Tc[f].reshape(4, 4), ti['T'][f].reshape(4, 4), fl & 1, ti['lxyz'][f, :m], ti['ldesc'][f, :m], (fl >> 1) & 1,
                                                    ti['loct'][f, :m], ti['lang'][f, :m], 2 * TH)
        if st[2] < 20:                                                  # src/Tracking.cc:941-942: `if(nmatches<20) return false;` before PoseOptimization
            assert g['ok1'].value == 0 and np.array_equal(g['T1'].reshape(4, 4), Tc[f].reshape(4, 4)), f
            assert np.array_equal(g['mp1'], mpA), f
            bailed += 1
            continue
        xyzA = np.zeros((n, 3), np.float32); xyzA[mpA >= 0] = ti['lxyz'][f, mpA[mpA >= 0]]
        kxy = np.stack([cur.keysUn['x'], cur.keysUn['y']], 1)
        _, _, outA = O.pose_optimization(Tc[f].reshape(4, 4), (mpA >= 0).astype(np.uint8), xyzA, kxy, cur.keysUn['octave'], cur.uRight, isig, camd['fx'], camd['fy'], camd['cx'], camd['cy'], camd['bf'])
        mpA[(mpA >= 0) & (outA != 0)] = -1
        # after TrackWithMotionModel: the pose, the surviving assignments (bad points are still held: the reference drops them at the start of SearchLocalPoints),
        # the return value nmatchesMap >= 10
        assert np.abs(g['T1'].reshape(4, 4) - r['T1']).max() <= 1e-6, (f, np.abs(g['T1'].reshape(4, 4) - r['T1']).max())
        assert g['ok1'].value == int(st[4] >= 10), (f, st)
        assert np.array_equal(g['mp1'], mpA), (f, int((g['mp1'] != mpA).sum()))
        # after TrackLocalMap
        assert np.array_equal(g['mp2'], r['mp']), (f, int((g['mp2'] != r['mp']).sum()))
        assert np.array_equal(g['outl'], r['outlier']), f
        assert g['inl'].value == st[7], (f, g['inl'].value, st)
        assert g['ok2'].value == int(st[7] >= 30), (f, st)
        assert np.abs(g['T2'].reshape(4, 4) - r['T2']).max() <= 1e-6, f
        keep = (g['mp1'] >= 0) & ((fl[np.maximum(g['mp1'], 0)] & 6) == 2)
        assert np.array_equal(g['mp2'][keep], g['mp1'][keep])           # first-half matches with observations (and not bad) survive; temporal points may be replaced (src/ORBmatcher.cc:87-89)
        full += 1; added += int(st[6])
    assert full >= 9 and bailed >= 1 and retried >= 2 and added > 20 * full, (full, bailed, retried, added)
