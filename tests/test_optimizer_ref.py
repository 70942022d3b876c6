"""Optimizer::PoseOptimization pinned against the REFERENCE'S OWN src/Optimizer.cc, src/Converter.cc and vendored g2o (oracle/_ref/liboptimizer_ref.so: every
file compiled unmodified from the reference tree; see oracle/Makefile, target ref_optimizer).  The image has no Eigen, so the library is built against the Eigen
stand-in of oracle/g2o_shim/Eigen (eager evaluation of Eigen's published formulas): what is pinned is the control flow and arithmetic of Optimizer.cc and g2o --
graph set-up, Levenberg with its lambda schedule and rejected trials, the Huber kernel, the four rounds with their chi-square re-classification, the early exits --
not Eigen's instruction order.  The oracle's sgo_pose_optimization (oracle/pose_opt.cpp, the checker of the GPU's pose_opt_kernel) must return the same inlier
count and the same outlier flags; the pose (float32 on both sides) must agree within 1e-6 -- on every case below it is in fact identical.  No device needed."""
import ctypes as C
import os

import numpy as np

import oracle as O
import refgolden as RG
import scenarios as S

LIB = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'oracle', '_ref', 'liboptimizer_ref.so')
POSE_TOL = 1e-6


def ref_pose_optimization(s):
    L = RG.load(LIB, __name__); L.ref_pose_optimization.restype = C.c_int
    c = s['cam']; f32 = np.float32
    T = np.ascontiguousarray(s['T0'], f32).reshape(16)
    a = [np.ascontiguousarray(s['has'], np.uint8), np.ascontiguousarray(s['xyz'], f32), np.ascontiguousarray(s['xy'], f32), np.ascontiguousarray(s['octave'], np.int32),
         np.ascontiguousarray(s['uright'], f32)]
    isig = np.ascontiguousarray(s['inv_s2'], f32)
    n = len(a[0]); out = np.zeros(16, f32); outl = np.zeros(n, np.uint8)
    r = L.ref_pose_optimization(RG.ptr(T), n, *[RG.ptr(x) for x in a], RG.ptr(isig), len(isig), C.c_float(c['fx']), C.c_float(c['fy']),
                                C.c_float(c['cx']), C.c_float(c['cy']), C.c_float(c['bf']), RG.ptr(out), RG.ptr(outl))
    return r, out.reshape(4, 4), outl


def oracle_pose_optimization(s):
    c = s['cam']
    return O.pose_optimization(s['T0'], s['has'], s['xyz'], s['xy'], s['octave'], s['uright'], s['inv_s2'], c['fx'], c['fy'], c['cx'], c['cy'], c['bf'])


def _same(s, tag):
    rn, rT, ro = ref_pose_optimization(s)
    on, oT, oo = oracle_pose_optimization(s)
    assert rn == on, (tag, rn, on)
    assert np.array_equal(ro, oo), (tag, int((ro != oo).sum()))
    assert np.abs(rT.astype(np.float64) - oT.astype(np.float64)).max() <= POSE_TOL, (tag, np.abs(rT - oT).max())
    return rn, bool(np.array_equal(rT, oT))


def test_tracking_like_frames():
    identical = 0
    for seed in range(1, 25):
        n, same = _same(S.pose_scenario(seed), ('plain', seed))
        assert n > 300
        identical += same
    assert identical >= 20                                  # in practice all of them: both sides round the same double pose to float32


def test_hard_frames_rejected_trials_many_outliers_and_noise():
    for seed in range(30, 42):
        _same(S.pose_scenario(seed, outlier_frac=0.45, noise=1.5, pose_err=(0.08, 0.3)), ('hard', seed))
    for seed in range(42, 48):                              # a start far from the optimum: Levenberg rejects trials and raises lambda
        _same(S.pose_scenario(seed, n=300, outlier_frac=0.3, noise=1.0, pose_err=(0.25, 0.8)), ('far', seed))


def test_monocular_only_and_stereo_only():
    for seed in (50, 51, 52):
        _same(S.pose_scenario(seed, mono_frac=1.0), ('mono', seed))
        _same(S.pose_scenario(seed, mono_frac=0.0), ('stereo', seed))


def test_early_exits():
    s = S.pose_scenario(5, outlier_frac=0.0, noise=0.2)
    for k in (0, 1, 2):                                     # fewer than three correspondences: pose untouched, 0 returned (src/Optimizer.cc:338-339)
        s2 = dict(s); s2['has'] = np.zeros_like(s['has']); s2['has'][:k] = 1
        n, same = _same(s2, ('few', k))
        assert n == 0 and same
    for k in (3, 4, 6, 9, 10, 11, 14):                      # fewer than ten edges: a single round (:427-428); ten and more: four
        s3 = dict(s); s3['has'] = np.zeros_like(s['has']); s3['has'][:k] = 1
        _same(s3, ('edges', k))
    s4 = S.pose_scenario(7, n=12, outlier_frac=0.5, noise=2.0)           # tiny graphs with outliers
    s4['has'][:] = 1
    _same(s4, ('tiny', 7))


def test_points_behind_the_camera_and_exact_start():
    s = S.pose_scenario(9)
    s['xyz'][:40] *= -1                                     # negative depth: huge residuals, flagged in the first round
    _same(s, ('behind', 9))
    s = S.pose_scenario(11, outlier_frac=0.0, noise=0.0, pose_err=(0.0, 0.0))   # already at the optimum: tiny gradient, Levenberg's stop rules
    _same(s, ('exact', 11))
