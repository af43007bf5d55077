"""GPU: the CUDA path against THE REFERENCE'S OWN FUNCTIONS, directly (no oracle in between).

oracle/_ref/libmatch_ref.so holds src/ORBmatcher.cc, LSDmatcher.cpp, PlaneMatcher.cpp, Frame.cc, KeyFrame.cc, MapPoint.cc, MapLine.cpp, MapPlane.cc,
Map.cc and Optimizer.cc compiled unmodified in the build container (oracle/ref/, `make -C oracle ref`); libtrack_ref.so holds src/Tracking.cc;
libpose_ref.so the reference's g2o + edges.  They travel to the GPU box prebuilt.  Each test calls the reference's function on objects built from the
same plain arrays the C ABI takes and compares with what the CUDA kernels return:

  ORBmatcher::SearchByProjection(Frame&, vector<MapPoint*>&, th)      src/ORBmatcher.cc:46-130      identical match lists / mbTrackInView
  ORBmatcher::SearchByProjection(Frame&, const Frame&, th, mono)      src/ORBmatcher.cc:1396-1535   identical match lists
  ORBmatcher::SearchByBoW(KeyFrame*, Frame&, vector<MapPoint*>&)      src/ORBmatcher.cc:160-292     identical match lists
  Frame::isInFrustum(MapLine*) + LSDmatcher::SearchByProjection       src/Frame.cc:369-437, src/LSDmatcher.cpp:141-211   bit-identical fields / lists
  PlaneMatcher::SearchMapByCoefficients                               src/PlaneMatcher.cpp:10-67    identical associations
  Optimizer::PoseOptimization / TranslationOptimization(Frame*)       src/Optimizer.cc:550-1275, 2995-3737   identical flags, pose 5e-6 rad / 2e-5 m
  Optimizer::LocalBundleAdjustment(KeyFrame*, bool*, Map*)            src/Optimizer.cc:1853-2678    identical erasures, poses 1e-6 (2e-5 on 20 % outliers)
  Tracking::TrackManhattanFrame                                       src/Tracking.cc:963-1137      rotation within 2e-6 per entry
  Frame::isLineGood, Frame::ComputeStereoFromRGBD                     src/Frame.cc:189-267, 603-621 bit-identical

(The bar of BASELINE.json for poses is 1e-4 rad / 1e-3 m.)  Where the libraries are absent, their recorded answers (ref_lib) stand in."""
import numpy as np
import pytest

import ref_lib
from planarslam_b200 import synth, synth_lba, synth_lines, synth_pose
from planarslam_b200.synth_manhattan import make_manhattan
from test_oracle_match_ref import PLANE_TH, last_case, map_case
from test_oracle_planematch import _scenario as plane_scenario

pytestmark = pytest.mark.gpu
FLAGS = ("outlier_pt", "outlier_line", "outlier_plane", "outlier_par", "outlier_ver")


def test_search_by_projection_map_cuda_vs_reference():
    from planarslam_b200.matcher import ORBmatcher
    tot = 0
    for seed, th, nnr in ((0, 3.0, 0.8), (1, 1.0, 0.8), (2, 5.0, 0.9), (3, 3.0, 0.6), (4, 10.0, 0.8)):
        fv, m, th, nnr, pre = map_case(seed, th, nnr)
        n, matches, in_view = ORBmatcher(nnr).SearchByProjection(fv, m, th, pre)
        rn, rmatches, rin_view = ref_lib.ref_search_by_projection_map(fv, m, th, nnr, pre)
        assert n == rn and ref_lib.same(matches, rmatches) and ref_lib.same(in_view, rin_view), seed
        tot += n
    assert tot > 1500


def test_search_by_projection_last_cuda_vs_reference():
    from planarslam_b200.matcher import ORBmatcher
    tot = 0
    for seed, th, mono, ori in ((0, 15.0, False, True), (1, 7.0, False, True), (2, 15.0, True, False), (3, 30.0, False, True), (4, 15.0, True, True)):
        fv, lf, m, th, mono, ori, pre = last_case(seed, th, mono, ori)
        n, matches = ORBmatcher(0.9, ori).SearchByProjectionLast(fv, lf, m, th, mono, pre)
        rn, rmatches = ref_lib.ref_search_by_projection_last(fv, lf, m, th, mono, ori, pre)
        assert n == rn and ref_lib.same(matches, rmatches), seed
        tot += n
    assert tot > 1500


def test_search_by_bow_cuda_vs_reference():
    from planarslam_b200._lib import Context
    from planarslam_b200.matcher import search_by_bow
    ctx = Context(640, 480, 1)
    tot = 0
    for seed in range(4):
        kf, f = synth_lines.make_bow_pair(seed, **(dict(n_kf=400, n_f=380, n_nodes=90) if seed < 3 else {}))
        for ratio, ori in ((0.7, True), (0.9, False), (0.75, True)):
            n, m = search_by_bow(ctx, kf, f, ratio, ori)
            rn, rm = ref_lib.ref_search_by_bow(kf, f, ratio, ori)
            assert n == rn and ref_lib.same(m, rm), (seed, ratio, ori)
            tot += n
    assert tot > 1000


def test_lines_in_frustum_and_line_search_cuda_vs_reference():
    from planarslam_b200._lib import Context
    from planarslam_b200.matcher import LSDmatcher, lines_in_frustum
    ctx = Context(640, 480, 1)
    for seed in range(6):
        fr, pos, nrm, mx, mn = synth_lines.make_line_frustum(seed)
        cnt, a = lines_in_frustum(ctx, fr, pos, nrm, mx, mn, 0.5)
        b = ref_lib.ref_lines_in_frustum(fr, pos, nrm, mx, mn, 0.5)
        iv = a["in_view"].astype(bool)
        assert np.array_equal(a["in_view"], b["in_view"]) and cnt == int(iv.sum()) and 60 < iv.sum() < 340
        for k in ("proj", "level", "view_cos"):
            assert np.array_equal(a[k][iv], b[k][iv]), (seed, k)
    tot = 0
    for seed in range(6):
        f, m = synth_lines.make_line_search(seed, n_frame=40 + 4 * seed, n_map=120 + 30 * seed)
        for th, nnr in ((1.0, 0.6), (3.0, 0.8)):
            n, assigned = LSDmatcher(nnr).SearchByProjection(f, m, th)
            rn, rassigned = ref_lib.ref_line_search_by_projection(f, m, th, nnr)
            assert n == rn and ref_lib.same(assigned, rassigned), (seed, th)
            tot += n
    assert tot > 200


def test_plane_match_cuda_vs_reference():
    from planarslam_b200.matcher import PlaneMatcher
    rng = np.random.default_rng(3)
    tot = 0
    for trial in range(12):
        T, fc, mc, bad, off, pts = plane_scenario(trial, rng)
        for th in (PLANE_TH, (0.1, 0.86, 0.08716, 0.9962)):
            n, m, v, p = PlaneMatcher(*th).SearchMapByCoefficients(T, fc, mc, bad, off, pts)
            r = ref_lib.ref_plane_match(T, fc, mc, bad, off, pts, *th)
            assert n == r[0] and ref_lib.same(m, r[1]) and ref_lib.same(v, r[2]) and ref_lib.same(p, r[3]), (trial, th)
            tot += n
    assert tot >= 20


def test_pose_and_translation_optimization_cuda_vs_reference():
    from planarslam_b200.optimizer import Optimizer
    opt = Optimizer()
    cases = [dict(seed=s, frame=3 * s) for s in range(8)]
    cases += [dict(seed=20 + s, frame=s, outlier_frac=0.25, rot_pert=0.05, trans_pert=0.08) for s in range(4)]
    cases += [dict(seed=30, frame=1, n_points=0, n_lines=0), dict(seed=7, frame=21, n_planes=0, n_par=0, n_ver=0), dict(seed=9, frame=5, n_points=40, n_lines=6)]
    probs = [synth_pose.make_pose_problem(**kw) for kw in cases]
    for translation_only in (False, True):
        res = opt.TranslationOptimizationBatch(probs) if translation_only else opt.PoseOptimizationBatch(probs)
        for kw, p, g in zip(cases, probs, res):
            r = ref_lib.ref_full_pose_optimization(p, translation_only)       # Optimizer::PoseOptimization(Frame*) itself; pose written back as float
            assert g["n_inliers"] == r["n_inliers"], (translation_only, kw)
            for k in FLAGS:
                if k in g and len(r[k]):
                    assert np.array_equal(g[k], r[k]), (translation_only, kw, k)
            da, dt = synth_pose.pose_error(g["Tcw_d"], r["Tcw"].astype(np.float64))
            assert da < 5e-6 and dt < 2e-5, (translation_only, kw, da, dt)


def test_local_bundle_adjustment_cuda_vs_reference():
    from planarslam_b200.lba import LocalBundleAdjuster
    ba = LocalBundleAdjuster()
    from test_oracle_lba_ref import SMALL
    small = dict(SMALL, line_kf_quirk=True)            # the cases of tests/test_oracle_lba_ref.py (oracle == reference there, on the CPU)
    cases = [dict(seed=s, **small) for s in (1, 10, 11)]
    cases += [dict(seed=2, n_kf=8, n_points=300, n_pt_obs=900, n_lines=0, n_line_obs=0, n_plane_obs=(0, 0, 0))]
    hard = [dict(seed=20 + s, **small, line_norm3=False, outlier_frac=0.2, plane_outlier_frac=0.25) for s in range(2)]
    big = [dict(seed=4, line_kf_quirk=True)]                               # BASELINE.json's local-map size
    n_erased = 0
    for kw in cases + hard + big:
        p = synth_lba.restrict_to_local_planes(synth_lba.make_lba_problem(**kw))
        g, r = ba.LocalBundleAdjustment(p), ref_lib.ref_full_local_bundle_adjustment(p)
        bad = r["pt_bad"][p["pt_obs_pt"]]
        assert np.array_equal(g["erase_pt"] | bad, r["erase_pt"]), kw
        assert np.array_equal(g["erase_pt"][bad == 0], r["erase_pt"][bad == 0]), kw
        if len(p["line_obs_line"]):
            assert np.array_equal(g["erase_line"] | r["line_bad"][p["line_obs_line"]], r["erase_line"]), kw
        for t in range(3):
            if len(p["plane_obs_plane"][t]):
                assert np.array_equal(g["erase_plane"][t] | r["plane_bad"][p["plane_obs_plane"][t]], r["erase_plane"][t]), (kw, t)
        tol = (2e-5, 5e-5) if kw in hard else (1e-6, 1e-6)
        for k in range(len(g["kf_Tcw_d"])):
            da, dt = synth_pose.pose_error(g["kf_Tcw_d"][k], r["kf_Tcw_d"][k])
            assert da < tol[0] and dt < tol[1], (kw, k, da, dt)
        assert np.median(np.abs(g["pt_Xw_d"] - r["pt_Xw_d"]).max(1)) < (2e-5 if kw in hard else 5e-6), kw    # the reference's result depends on its heap layout there
        n_erased += int(g["erase_pt"].sum())
    assert n_erased > 300


def test_track_manhattan_cuda_vs_reference():
    from planarslam_b200._lib import Context
    from planarslam_b200.manhattan import TrackManhattanFrame
    cases = [dict(seed=s) for s in range(8)] + [dict(seed=3, weights=(0.5, 0.5, 0.0), clutter=0.02, n_lines=0), dict(seed=4, weights=(1.0, 0.0, 0.0), clutter=0.0, n_lines=0),
                                                 dict(seed=7, n_normals=500, n_lines=5), dict(seed=8, perturb_deg=10.0, noise_deg=4.0), dict(seed=9, clutter=0.4)]
    data = [make_manhattan(**kw) for kw in cases]
    ctx = Context(640, 480, max_batch=1)
    res, _, _ = TrackManhattanFrame(ctx, np.stack([d[0] for d in data]), [d[1] for d in data], [d[2] for d in data])
    for f, d in enumerate(data):
        r = ref_lib.ref_track_manhattan_frame(d[0], d[1], d[2])            # Tracking::TrackManhattanFrame itself
        assert np.abs(res[f]["R"] - r).max() < 2e-6, (cases[f], np.abs(res[f]["R"] - r).max())


def test_is_line_good_and_stereo_cuda_vs_reference():
    from planarslam_b200._lib import Context
    from planarslam_b200.frame import ComputeStereoFromRGBD
    from planarslam_b200.lines import KEYLINE_DTYPE, LineSegment, isLineGood
    from planarslam_b200.orb import KEYPOINT_DTYPE
    nf = 4
    frames = [synth.render_frame(seed=s, frame=3 * s) for s in range(nf)]
    ctx = Context(640, 480, max_batch=nf)
    res = LineSegment(ctx).ExtractLineSegment(np.stack([f[0] for f in frames]), 40)          # the CUDA detector's own key lines feed the 3-D fit
    kl = np.zeros((nf, 40), KEYLINE_DTYPE)
    n_lines = np.zeros(nf, np.int32)
    for f in range(nf):
        n_lines[f] = len(res[f][0])
        kl[f, :n_lines[f]] = res[f][0]
    d16 = np.stack([f[1] if k % 2 == 0 else synth.noisy_depth(f[1], k, 0.1 + 0.05 * k, 0.004 * k) for k, f in enumerate(frames)])
    factor = np.float32(1.0 / synth.DEPTH_FACTOR)
    seeds, skips = np.array([1, 1, 5, 99], np.uint32), np.array([0, 13, 0, 250], np.int32)
    out, _ = isLineGood(ctx, kl, n_lines, d16, synth.TUM3_K, factor, seeds, skips)
    n_valid = 0
    for f in range(nf):
        dl, l3 = ref_lib.ref_full_lines3d_frame(kl[f, :n_lines[f]], d16[f].astype(np.float32) * factor, synth.TUM3_K, seed=int(seeds[f]), skip=int(skips[f]))   # Frame::isLineGood itself
        g = out[f, :n_lines[f]]
        g3 = np.concatenate([g["A"], g["B"]], 1)
        assert ref_lib.same(g3, l3) and ref_lib.same(g["depth"], dl), f       # mvLines3D, mvDepthLine
        assert np.array_equal(g["valid"].astype(bool), np.any(g3 != 0, axis=1)), f
        n_valid += int(g["valid"].sum())
    assert n_valid > 40
    # Frame::ComputeStereoFromRGBD itself
    rng = np.random.default_rng(5)
    kp = np.zeros((nf, 1000), KEYPOINT_DTYPE)
    for f in range(nf):
        kp["x"][f], kp["y"][f] = rng.uniform(16, 623, 1000).astype(np.float32), rng.uniform(16, 463, 1000).astype(np.float32)
    ur, dz = ComputeStereoFromRGBD(ctx, kp, np.full(nf, 1000, np.int32), d16, factor, 40.0)
    for f in range(nf):
        xy = np.stack([kp["x"][f], kp["y"][f]], 1)
        r = ref_lib.ref_full_compute_stereo_from_rgbd(xy, xy, d16[f].astype(np.float32) * factor, 40.0)
        assert ref_lib.same(ur[f], r[0]) and ref_lib.same(dz[f], r[1]), f
