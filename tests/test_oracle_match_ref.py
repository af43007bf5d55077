"""CPU: the matcher oracles (oracle/search.cc, bow.cc, linesearch.cc, planematch.cc) pinned against THE REFERENCE'S OWN matchers: src/ORBmatcher.cc,
src/LSDmatcher.cpp and src/PlaneMatcher.cpp compile unmodified from /root/reference together with the object graph they walk (src/Frame.cc, KeyFrame.cc,
MapPoint.cc, MapLine.cpp, MapPlane.cc, Map.cc ...) into oracle/_ref/libmatch_ref.so; oracle/ref/match_driver.cc only builds Frame / KeyFrame / MapPoint /
MapLine / MapPlane objects from the C ABI's plain-array views and reads the assignments back.  Every decision - Frame::isInFrustum (points and lines),
Frame::GetFeaturesInArea over the reference's own feature grid, GetLinesInArea, descriptor gates, ratio tests, the rotation histogram,
PointDistanceFromPlane - is the reference's code.  Bar: identical match lists, counts and mbTrackInView flags; bit-identical projections / view cosines.
The golden fixture (tests/golden/match_reference.npz, tools/make_golden_ref.py) holds the reference's answers for the first case of each family."""
import ctypes as C
import os

import numpy as np

import oracle_lib
import ref_lib
from planarslam_b200 import synth_lines
from test_oracle_planematch import _scenario as plane_scenario
from test_oracle_search import scenario

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "match_reference.npz")
PLANE_TH = (0.05, 0.985, 0.08716, 0.9962)


def map_case(seed, th, nnr):
    fv, m, lf = scenario(f0=10 + seed, f1=11 + seed, seed=seed)
    m["skip"][::17] = 1
    pre = np.full(fv["n"], -1, np.int32)
    pre[::23] = 3
    return fv, m, th, nnr, pre


def last_case(seed, th, mono, ori):
    fv, m, lf = scenario(f0=10 + 2 * seed, f1=11 + 2 * seed + (seed == 3), seed=seed)
    lf["outlier"][::13] = 1
    pre = np.full(fv["n"], -1, np.int32)
    pre[::29] = 5
    return fv, lf, m, th, mono, ori, pre


def oracle_plane_match(T, fc, mc, bad, off, pts, th):
    L = oracle_lib.lib()
    L.orc_plane_match.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p] + [C.c_float] * 4 + [C.c_void_p] * 3
    om, ov, op = [np.zeros(len(fc), np.int32) for _ in range(3)]
    n = L.orc_plane_match(T.ctypes.data, len(fc), fc.ctypes.data, len(mc), mc.ctypes.data, bad.ctypes.data, off.ctypes.data, pts.ctypes.data, *th,
                          om.ctypes.data, ov.ctypes.data, op.ctypes.data)
    return n, om, ov, op


def gold_cases():
    """(name, oracle outputs as a flat list of arrays, reference callable) for the first case of every family."""
    fv, m, th, nnr, pre = map_case(0, 3.0, 0.8)
    yield "map", oracle_lib.search_by_projection_map(fv, m, th, nnr, pre), lambda: ref_lib.ref_search_by_projection_map(fv, m, th, nnr, pre)
    a = last_case(0, 15.0, False, True)
    yield "last", oracle_lib.search_by_projection_last(*a), lambda: ref_lib.ref_search_by_projection_last(*a)
    kf, f = synth_lines.make_bow_pair(0, n_kf=400, n_f=380, n_nodes=90)
    yield "bow", oracle_lib.search_by_bow(kf, f, 0.7, True), lambda: ref_lib.ref_search_by_bow(kf, f, 0.7, True)
    lfm = synth_lines.make_line_search(0)
    yield "line", oracle_lib.line_search_by_projection(*lfm, 3.0, 0.8), lambda: ref_lib.ref_line_search_by_projection(*lfm, 3.0, 0.8)
    T, fc, mc, bad, off, pts = plane_scenario(2, np.random.default_rng(3))
    yield "plane", oracle_plane_match(T, fc, mc, bad, off, pts, PLANE_TH), lambda: ref_lib.ref_plane_match(T, fc, mc, bad, off, pts, *PLANE_TH)


def test_matcher_oracles_match_reference_golden():
    g = np.load(GOLD)
    for name, o, _ in gold_cases():
        assert int(o[0]) == int(g[f"{name}_n"][0]), name
        for k, arr in enumerate(o[1:]):
            assert np.array_equal(arr, g[f"{name}_{k}"]), (name, k)


def test_search_by_projection_map_identical_to_compiled_reference():
    tot = 0
    for seed, th, nnr in ((0, 3.0, 0.8), (1, 1.0, 0.8), (2, 5.0, 0.9), (3, 3.0, 0.6), (4, 10.0, 0.8)):
        fv, m, th, nnr, pre = map_case(seed, th, nnr)
        n, matches, in_view = oracle_lib.search_by_projection_map(fv, m, th, nnr, pre)
        rn, rmatches, rin_view = ref_lib.ref_search_by_projection_map(fv, m, th, nnr, pre)
        assert n == rn and ref_lib.same(matches, rmatches) and ref_lib.same(in_view, rin_view), seed
        tot += n
    assert tot > 1500


def test_search_by_projection_last_identical_to_compiled_reference():
    tot = 0
    for seed, th, mono, ori in ((0, 15.0, False, True), (1, 7.0, False, True), (2, 15.0, True, False), (3, 30.0, False, True), (4, 15.0, True, True)):
        a = last_case(seed, th, mono, ori)
        n, matches = oracle_lib.search_by_projection_last(*a)
        rn, rmatches = ref_lib.ref_search_by_projection_last(*a)
        assert n == rn and ref_lib.same(matches, rmatches), seed
        tot += n
    assert tot > 1500


def test_search_by_bow_identical_to_compiled_reference():
    tot = 0
    for seed in range(4):
        kf, f = synth_lines.make_bow_pair(seed, **(dict(n_kf=400, n_f=380, n_nodes=90) if seed < 3 else {}))       # seed 3: BASELINE size (1000 x 1000, 300 nodes)
        for ratio, ori in ((0.7, True), (0.9, False), (0.75, True)):
            n, m = oracle_lib.search_by_bow(kf, f, ratio, ori)
            rn, rm = ref_lib.ref_search_by_bow(kf, f, ratio, ori)
            assert n == rn and ref_lib.same(m, rm), (seed, ratio, ori)
            tot += n
    assert tot > 1000


def test_lines_in_frustum_and_line_search_identical_to_compiled_reference():
    for seed in range(6):
        fr, pos, nrm, mx, mn = synth_lines.make_line_frustum(seed)
        a, b = oracle_lib.lines_in_frustum(fr, pos, nrm, mx, mn, 0.5), ref_lib.ref_lines_in_frustum(fr, pos, nrm, mx, mn, 0.5)
        iv = a["in_view"].astype(bool)
        assert np.array_equal(a["in_view"], b["in_view"]) and 60 < iv.sum() < 340
        for k in ("proj", "level", "view_cos"):                   # the tracking fields are only written for lines in view
            assert np.array_equal(a[k][iv], b[k][iv]), (seed, k)
    tot = 0
    for seed in range(6):
        f, m = synth_lines.make_line_search(seed, n_frame=40 + 20 * seed, n_map=120 + 30 * seed)
        for th, nnr in ((1.0, 0.6), (3.0, 0.8)):
            n, assigned = oracle_lib.line_search_by_projection(f, m, th, nnr)
            rn, rassigned = ref_lib.ref_line_search_by_projection(f, m, th, nnr)
            assert n == rn and ref_lib.same(assigned, rassigned), (seed, th)
            tot += n
    assert tot > 300


def test_plane_match_identical_to_compiled_reference():
    rng = np.random.default_rng(3)
    tot = 0
    for trial in range(12):
        T, fc, mc, bad, off, pts = plane_scenario(trial, rng)
        for th in (PLANE_TH, (0.1, 0.86, 0.08716, 0.9962)):       # TUM3.yaml thresholds; PlaneMatcher's defaults
            o, r = oracle_plane_match(T, fc, mc, bad, off, pts, th), ref_lib.ref_plane_match(T, fc, mc, bad, off, pts, *th)
            assert o[0] == r[0] and all(ref_lib.same(x, y) for x, y in zip(o[1:], r[1:])), (trial, th)
            tot += o[0]
    assert tot >= 20
