"""CPU: the PoseOptimization oracle (oracle/poseopt.cc) pinned against THE REFERENCE'S OWN g2o: Thirdparty/g2o (sparse optimiser, BlockSolver_6_3, dense
solver, the modified Levenberg-Marquardt with its stop criterion, Huber kernel), SE3Quat / VertexSE3Expmap, the projection edges, include/EdgeLine.h,
g2oAddition (Plane3D, EdgePlane / EdgeParallelPlane / EdgeVerticalPlane with their numeric Jacobians) and src/Converter.cc compile unmodified from
/root/reference (oracle/_ref/libpose_ref.so) against an Eigen stand-in (oracle/ref/shims/Eigen/mini_eigen.hpp: Eigen's formulas, plain left-to-right
reductions).  Optimizer::PoseOptimization itself needs the Frame / Map object graph; its graph construction and four rounds are restated in
oracle/ref/pose_driver.cc.  Bar: identical inlier counts and outlier flags of every edge family, pose within 5e-6 rad / 2e-5 m (the task's bar is 1e-4 rad
/ 1e-3 m).  Not compared: LM iteration counts - at convergence the gain of a step is rounding noise, so accept / reject decisions (and with them the
"three small gains" stop criterion) depend on the summation order of whichever linear algebra library is underneath."""
import os

import numpy as np

import oracle_lib
import ref_lib
from planarslam_b200 import synth_pose

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "pose_reference.npz")
FLAGS = ("outlier_pt", "outlier_line", "outlier_plane", "outlier_par", "outlier_ver")
GOLD_CASES = [dict(seed=0, frame=0), dict(seed=4, frame=12, outlier_frac=0.2), dict(seed=7, frame=21, n_planes=0, n_par=0, n_ver=0), dict(seed=9, frame=5, n_points=40, n_lines=6)]


def _same(o, r, ang=5e-6, dist=2e-5):
    assert o["n_inliers"] == r["n_inliers"]
    for k in FLAGS:
        assert np.array_equal(o[k], r[k]), k
    da, dt = synth_pose.pose_error(o["Tcw_d"], r["Tcw_d"])
    assert da < ang and dt < dist, (da, dt)


def test_oracle_pose_matches_reference_golden():
    g = np.load(GOLD)
    for i, kw in enumerate(GOLD_CASES):
        o = oracle_lib.pose_optimization(synth_pose.make_pose_problem(**kw))
        _same(o, dict(Tcw_d=g[f"c{i}_Tcw_d"], n_inliers=int(g[f"c{i}_n"][0]), **{k: g[f"c{i}_{k}"] for k in FLAGS}))


def test_oracle_pose_agrees_with_compiled_reference_g2o():
    cases = [dict(seed=s, frame=3 * s) for s in range(8)]
    cases += [dict(seed=s, frame=2 * s, n_planes=0, n_par=0, n_ver=0) for s in range(4)]                     # analytic Jacobians only
    cases += [dict(seed=20 + s, frame=s, outlier_frac=0.25, rot_pert=0.05, trans_pert=0.08) for s in range(4)]   # many outliers, poor start
    cases += [dict(seed=30, frame=1, n_points=0, n_lines=0), dict(seed=31, frame=2, n_points=30, n_lines=0, n_planes=0, n_par=0, n_ver=0),
              dict(seed=32, frame=3, n_points=2, n_lines=0, n_planes=0, n_par=0, n_ver=0, outlier_frac=0.0)]  # planes only; few points; < 3 correspondences
    for kw in cases:
        p = synth_pose.make_pose_problem(**kw)
        _same(oracle_lib.pose_optimization(p), ref_lib.ref_pose_optimization(p))


def test_oracle_translation_optimization_agrees_with_compiled_reference_g2o():
    """Optimizer::TranslationOptimization (src/Optimizer.cc:2995-3737) with the reference's OnlyTranslation edges: identical inlier counts and flags,
    rotation untouched on both sides, translation within 5e-6 m."""
    cases = [dict(seed=s, frame=3 * s, rot_pert=0.0 if s % 2 == 0 else 0.003) for s in range(8)]
    cases += [dict(seed=40 + s, frame=s, outlier_frac=0.25, trans_pert=0.08) for s in range(3)]
    cases += [dict(seed=50, frame=4, n_points=2, n_lines=5, n_planes=3, outlier_frac=0.0), dict(seed=51, frame=6, n_points=25, n_lines=0, n_planes=0)]
    for kw in cases:
        p = synth_pose.make_pose_problem(**kw)
        o, r = oracle_lib.pose_optimization(p, translation_only=True), ref_lib.ref_translation_optimization(p)
        assert o["n_inliers"] == r["n_inliers"], kw
        for k in ("outlier_pt", "outlier_line", "outlier_plane"):
            assert np.array_equal(o[k], r[k]), (kw, k)
        assert np.allclose(o["Tcw_d"][:3, :3], r["Tcw_d"][:3, :3], rtol=0, atol=1e-12)
        assert np.linalg.norm(o["Tcw_d"][:3, 3] - r["Tcw_d"][:3, 3]) < 5e-6, kw


def test_oracle_pose_agrees_with_the_reference_functions_themselves():
    """Optimizer::PoseOptimization(Frame*) and Optimizer::TranslationOptimization(Frame*) called AS THEY ARE (src/Optimizer.cc compiled unmodified into
    libmatch_ref.so with Frame.cc / MapPoint.cc / MapLine.cpp / MapPlane.cc; oracle/ref/match_driver.cc only fills a Frame from the problem arrays and reads
    mTcw and the mvb*Outlier vectors back; the Plane.* settings arrive through the reference's Config::Get).  Nothing of the function is restated here.
    The reference writes the pose back as float (Converter::toCvMat), so the comparison is against the oracle's double pose to float rounding."""
    cases = [dict(seed=s, frame=3 * s) for s in range(8)]
    cases += [dict(seed=20 + s, frame=s, outlier_frac=0.25, rot_pert=0.05, trans_pert=0.08) for s in range(4)]
    cases += [dict(seed=30, frame=1, n_points=0, n_lines=0), dict(seed=7, frame=21, n_planes=0, n_par=0, n_ver=0), dict(seed=9, frame=5, n_points=40, n_lines=6)]
    for translation_only in (False, True):
        for kw in cases:
            p = synth_pose.make_pose_problem(**kw)
            o = oracle_lib.pose_optimization(p, translation_only=True) if translation_only else oracle_lib.pose_optimization(p)
            r = ref_lib.ref_full_pose_optimization(p, translation_only)
            assert o["n_inliers"] == r["n_inliers"], (translation_only, kw)
            for k in FLAGS:
                if k in o and len(r[k]):
                    assert np.array_equal(o[k], r[k]), (translation_only, kw, k)
            da, dt = synth_pose.pose_error(o["Tcw_d"], r["Tcw"].astype(np.float64))
            assert da < 5e-6 and dt < 2e-5, (translation_only, kw, da, dt)
