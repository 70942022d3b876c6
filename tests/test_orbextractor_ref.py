"""The extractor pinned against the REFERENCE'S OWN src/ORBextractor.cc (oracle/_ref/liborbextractor_ref.so: the file compiled unmodified from the reference
tree; the OpenCV algorithms it calls -- cv::resize, cv::FAST, cv::GaussianBlur, cv::fastAtan2 -- resolve to the oracle's restatements, each pinned bit for bit
against the real cv2 primitive by tests/test_oracle_golden.py).  What this pins is everything the reference itself wrote: the constructor's tables, the pyramid
loop, the per-cell FAST calls with the threshold fallback, DistributeOctTree / DivideNode on std::list, IC_Angle, the rotated BRIEF sampling, the scaling of the
keypoints in the call operator.  The oracle must return the same keypoints (every field, bit for bit) and the same descriptors.

One defined quirk is involved: DistributeOctTree sorts (size, ExtractorNode*) pairs (src/ORBextractor.cc:684), so nodes of equal size are ordered by their
ADDRESS.  With glibc's malloc -- freed list nodes are reused last-in-first-out -- that order depends on the history of the heap and the reference's output is not
a function of its input (test_address_order_is_the_only_difference shows a handful of keypoints per frame moving).  The oracle and the GPU fix the tie-break as
creation sequence (quirk Q1); the reference is run on an allocator whose addresses grow with creation order, which makes the two comparable.  No device needed."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle as O
import refgolden as RG
from pysgs import synth

LIB = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'oracle', '_ref', 'liborbextractor_ref.so')


def ref_extract(img, nfeatures=1000, scale=1.2, nlevels=8, ini=20, mn=7, monotone=True):
    L = RG.load(LIB, __name__); L.ref_orb_extract.restype = C.c_int
    L.ref_set_monotone_allocator(1 if monotone else 0)
    img = np.ascontiguousarray(img, np.uint8)
    cap = 4 * nfeatures + 4096
    k = np.zeros(cap, O.KP_DTYPE); d = np.zeros((cap, 32), np.uint8)
    n = L.ref_orb_extract(RG.ptr(img), img.shape[1], img.shape[0], img.strides[0], nfeatures, C.c_float(scale), nlevels, ini, mn, RG.ptr(k), RG.ptr(d), cap)
    L.ref_set_monotone_allocator(0)
    assert 0 <= n <= cap
    return k[:n], d[:n]


def same(img, **kw):
    p = O.params(kw.get('nfeatures', 1000), kw.get('scale', 1.2), kw.get('nlevels', 8), kw.get('ini', 20), kw.get('mn', 7))
    ko, do = O.extract(img, p)
    kr, dr = ref_extract(img, **kw)
    assert len(kr) == len(ko), (len(kr), len(ko))
    assert kr.tobytes() == ko.tobytes()
    assert np.array_equal(dr, do)
    return len(ko)


def test_s2_stream_frames():
    frames, _ = synth.stream_s2(6, 640, 480, seed=3)
    assert sum(same(frames[f]) for f in range(6)) > 5000


@pytest.mark.parametrize('w,h,nf', [(640, 480, 1000), (1280, 720, 2000), (321, 243, 500), (752, 480, 1200)])
def test_other_geometries(w, h, nf):
    img = synth.frame_s1(w, h, seed=5)
    assert same(img, nfeatures=nf) > nf // 3


def test_other_parameters():
    img = synth.frame_s1(640, 480, seed=9)
    assert same(img, nfeatures=700, scale=1.3, nlevels=6) > 300
    assert same(img, nfeatures=1500, ini=12, mn=5) > 700


def test_degenerate_images():
    rng = np.random.RandomState(1)
    assert same(rng.randint(0, 256, (480, 640)).astype(np.uint8)) > 900                          # noise: far more candidates than features, deep quadtree
    assert same(np.full((480, 640), 127, np.uint8)) == 0                                        # constant: nothing anywhere, every cell takes the fallback
    cb = ((np.add.outer(np.arange(480) // 16, np.arange(640) // 16) & 1) * 255).astype(np.uint8)
    same(cb)                                                                                    # checkerboard: many exactly tied responses


def test_address_order_is_the_only_difference():
    """With glibc's allocator the reference's quadtree breaks size ties by heap address: the candidates are the same, a few kept keypoints differ."""
    frames, _ = synth.stream_s2(3, 640, 480, seed=3)
    moved = 0
    for f in range(3):
        ko, _ = O.extract(frames[f])
        kr, _ = ref_extract(frames[f], monotone=False)
        a = set(zip(ko['x'].tolist(), ko['y'].tolist(), ko['octave'].tolist())); b = set(zip(kr['x'].tolist(), kr['y'].tolist(), kr['octave'].tolist()))
        moved += len(a ^ b)
        assert len(a & b) >= 0.97 * len(a)
    print('keypoints differing between address order and creation order over 3 frames: %d' % moved)
