"""MapPoint::ComputeDistinctiveDescriptors, PredictScale (both overloads) and the 0.8 / 1.2 invariance getters pinned against the REFERENCE'S OWN src/MapPoint.cc
(oracle/_ref/libmappoint_ref.so: the file compiled unmodified from the reference tree against the real include/MapPoint.h; stand-ins only for KeyFrame / Frame /
Map / ORBmatcher).  The oracle's sgo_distinctive_descriptor (the checker of the GPU's distinctive_kernel) must pick the same descriptor -- including ties between
equal medians, which the reference resolves by the iteration order of its std::map<KeyFrame*, size_t>, i.e. by key-frame ADDRESS (ascending here) -- and the
predicted pyramid level of the oracle's isInFrustum (glibc logf restated) must equal the reference's for every distance ratio.  No device needed."""
import ctypes as C
import os

import numpy as np

import oracle as O
import refgolden as RG

LIB = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'oracle', '_ref', 'libmappoint_ref.so')


def ref_distinctive(desc, bad=None):
    L = RG.load(LIB, __name__); L.ref_mp_distinctive.restype = C.c_int
    d = np.ascontiguousarray(desc, np.uint8); out = np.zeros(32, np.uint8)
    b = None if bad is None else np.ascontiguousarray(bad, np.uint8)
    ok = L.ref_mp_distinctive(RG.ptr(d), RG.ptr(b) if b is not None else None, len(d), RG.ptr(out))
    return out if ok else None


def test_distinctive_descriptor_incl_ties_and_bad_key_frames():
    rng = np.random.RandomState(3)
    ties = 0
    for trial in range(300):
        n = int(rng.choice([1, 2, 3, 4, 5, 8, 13, 17, 40, 64]))
        base = rng.randint(0, 256, (max(1, n // 3), 32)).astype(np.uint8)
        d = base[rng.randint(0, len(base), n)].copy()                  # clusters of near-duplicates: many equal medians
        flips = rng.randint(0, 256, (n, 3))
        for i in range(n):
            for fbit in flips[i][:rng.randint(0, 4)]:
                d[i, fbit >> 3] ^= 1 << (fbit & 7)
        bad = (rng.uniform(size=n) < 0.2).astype(np.uint8) if trial % 3 == 0 else None
        got = ref_distinctive(d, bad)
        keep = d if bad is None else d[bad == 0]
        if len(keep) == 0:
            assert got is None
            continue
        idx = O.distinctive_descriptor(keep)
        assert got is not None and np.array_equal(got, keep[idx]), (trial, n)
        # count the trials in which a different tie-break would have shown: another descriptor with the same median but other bytes
        dm = np.array([[O.hamming(a, b) for b in keep] for a in keep])
        med = np.sort(dm, axis=1)[:, int(0.5 * (len(keep) - 1))]
        ties += int(any(med[j] == med[idx] and not np.array_equal(keep[j], keep[idx]) for j in range(len(keep))))
    assert ties > 20


def test_predict_scale_and_invariance_getters():
    L = RG.load(LIB, __name__)
    rng = np.random.RandomState(5)
    nlevels = 8
    log_sf = float(O.logf(np.float32(1.2)))
    T = np.eye(4, dtype=np.float32)
    cam = (500.0, 500.0, 320.0, 240.0, 40.0, 0.0, 0.0, 640.0, 480.0)
    total = 0
    for mx in (0.7, 1.0, 3.3, 12.5, 40.0):
        mx = np.float32(mx); mn = np.float32(mx / 1e4)
        # ratios around every level boundary (1.2^k, k = -1..9), exact boundaries in float, and random ones; d <= 1.2 mx keeps the point inside the invariance range
        k = np.arange(-1, 10)
        edges = (mx / np.float32(1.2) ** k.astype(np.float32)).astype(np.float32)
        d = np.concatenate([edges, np.nextafter(edges, np.float32(0)), np.nextafter(edges, np.float32(1e9)),
                            (mx / rng.uniform(0.84, 6.0, 4000)).astype(np.float32)]).astype(np.float32)
        d = d[(d <= np.float32(1.2) * mx) & (d >= np.float32(0.8) * mn)]
        lk = np.zeros(len(d), np.int32); lf = np.zeros(len(d), np.int32); inv = np.zeros(2, np.float32)
        L.ref_mp_predict_scale(C.c_float(mn), C.c_float(mx), RG.ptr(d), len(d), nlevels, C.c_float(log_sf), RG.ptr(lk), RG.ptr(lf), RG.ptr(inv))
        assert np.array_equal(lk, lf)
        assert inv[0] == np.float32(0.8) * mn and inv[1] == np.float32(1.2) * mx
        xyz = np.zeros((len(d), 3), np.float32); xyz[:, 2] = d
        nrm = np.zeros((len(d), 3), np.float32); nrm[:, 2] = 1
        out = O.is_in_frustum(T, cam, nlevels, log_sf, xyz, nrm, np.full(len(d), mn, np.float32), np.full(len(d), mx, np.float32), 0.5)
        assert out['inview'].all()
        assert np.array_equal(out['level'], lf), (float(mx), np.nonzero(out['level'] != lf)[0][:5])
        assert set(np.unique(lf)) == set(range(nlevels))
        total += len(d)
    assert total > 15000
