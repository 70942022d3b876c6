"""What Detector2D::detect does with ncnn's DetectionOutput rows (src/Detector2D.cc:52-88: the two thresholds, clamping to the 300 x 300 network frame, scaling to
the image, the person split, the two 'have dynamic object' flags) pinned against the REFERENCE'S OWN src/Detector2D.cc, compiled unmodified against stand-ins
(oracle/_ref/libdetector2d_ref.so; ncnn's extract() hands back planted rows -- the network itself is NOT part of this pin).  The oracle's postprocess() must
produce the same objects, boxes and flags bit for bit, including the float-vs-double comparison `prob > 0.2`.  No device needed."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'oracle'))
import detector_oracle as DO  # noqa: E402
import refgolden as RG  # noqa: E402

LIB = os.path.join(ROOT, 'oracle', '_ref', 'libdetector2d_ref.so')


def ref_post(rows, w, h, det_thr, dyn_thr):
    L = RG.load(LIB, __name__)
    rows = np.ascontiguousarray(rows, np.float32).reshape(-1, 6)
    cap = max(1, len(rows))
    tv = np.zeros((cap, 6), np.float32); ob = np.zeros((cap, 6), np.float32); dm = np.zeros((cap, 4), np.float32); dr = np.zeros((cap, 4), np.float32)
    n = [C.c_int() for _ in range(6)]
    p = RG.ptr
    L.ref_detector2d_postprocess(len(rows), p(rows), w, h, C.c_float(det_thr), C.c_float(dyn_thr), cap, p(tv), C.byref(n[0]), p(ob), C.byref(n[1]), p(dm), C.byref(n[2]),
                                 p(dr), C.byref(n[3]), C.byref(n[4]), C.byref(n[5]))
    return tv[:n[0].value], ob[:n[1].value], dm[:n[2].value], dr[:n[3].value], bool(n[4].value), bool(n[5].value)


@pytest.mark.parametrize('seed', range(6))
def test_postprocess_equals_the_reference(seed):
    rs = np.random.RandomState(seed)
    n = 100
    rows = np.zeros((n, 6), np.float32)
    rows[:, 0] = rs.choice([15, 15, 9, 7, 20, 1], n)
    rows[:, 1] = rs.uniform(0, 1, n)
    rows[:10, 1] = np.float32(0.2)                           # person rows exactly at the float 0.2: the reference compares against the DOUBLE literal 0.2
    rows[:10, 0] = 15
    rows[10:14, 1] = [0.5, 0.1, 0.01, 0.9]                   # rows sitting on thresholds
    c = rs.uniform(-0.2, 1.2, (n, 4)).astype(np.float32)     # corners beyond the frame get clamped
    rows[:, 2] = np.minimum(c[:, 0], c[:, 2]); rows[:, 4] = np.maximum(c[:, 0], c[:, 2]); rows[:, 3] = np.minimum(c[:, 1], c[:, 3]); rows[:, 5] = np.maximum(c[:, 1], c[:, 3])
    for (w, h) in ((640, 480), (1280, 720)):
        for det_thr, dyn_thr in ((0.5, 0.1), (0.9, 0.01), (0.2, 0.2)):
            tv, ob, dm, dr, hm, hr = ref_post(rows, w, h, det_thr, dyn_thr)
            objs, dyn_map, dyn_rm = DO.postprocess(rows, w, h, det_thr, dyn_thr)
            assert np.array_equal(objs, tv)                                           # every accepted row, persons included, in detection order
            assert np.array_equal(objs[objs[:, 0] != 15], ob)                         # mvObjects2D: the non-person objects
            assert np.array_equal(dyn_map, dm) and np.array_equal(dyn_rm, dr)
            assert hm == (len(dyn_map) > 0) and hr == (len(dyn_rm) > 0)
            assert len(tv) > 10


def test_no_rows():
    tv, ob, dm, dr, hm, hr = ref_post(np.zeros((0, 6), np.float32), 640, 480, 0.5, 0.1)
    assert len(tv) == len(ob) == len(dm) == len(dr) == 0 and not hm and not hr
