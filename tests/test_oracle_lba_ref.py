"""CPU: the LocalBundleAdjustment oracle (oracle/lba.cc) pinned against THE REFERENCE'S OWN g2o: SparseOptimizer, BlockSolver_6_3 (Schur complement over
the marginalised point / line-endpoint / plane vertices), OptimizationAlgorithmLevenberg, Huber kernels, VertexSE3Expmap / VertexSBAPointXYZ / VertexPlane
and the six binary edge types compile unmodified from /root/reference into oracle/_ref/libpose_ref.so against the Eigen stand-in; g2o's wrapper over
Eigen's sparse Cholesky is replaced by a dense stand-in (oracle/ref/shims/Thirdparty/g2o/g2o/solvers/linear_solver_eigen.h).
Optimizer::LocalBundleAdjustment (src/Optimizer.cc:1853-2678) needs the KeyFrame / Map object graph; its graph construction, optimize(5) -> chi-square gate
-> optimize(10) and the erase lists are restated in oracle/ref/lba_driver.cc on the plain-array problem of the C ABI.
Bar: identical erase flags of every edge family and identical iteration counts of both optimisations; key-frame poses within 5e-6 rad / 1e-5 m, points
within 5e-4 m (median 5e-6 m), plane coefficients 2e-5, line endpoints 5e-3 m with their point-to-line residuals within 2e-3 px (an endpoint has three
unknowns and one residual per observation, so with fewer than three observations it slides freely along the null space of its Hessian and only the LM
damping holds it: its position amplifies last-bit differences by 1/lambda, its residuals do not) (the double outputs; the task's bar is 1e-4 rad / 1e-3 m).  Why not tighter:
the stereo edge projects with a FLOAT reciprocal depth (types_six_dof_expmap.cpp:150-157, kept by the oracle), so its residual is a step function of the
estimate with ~3e-5 px steps; two double implementations whose estimates differ in the last bits land on different steps, and a point that keeps one or
two observations moves along its viewing ray by that noise times its depth uncertainty (~0.2 m/px at 3 m).  With monocular observations only the two
agree to 1e-10 rad / 2e-7 m (asserted below)."""
import os

import numpy as np

import oracle_lib
import ref_lib
from planarslam_b200 import synth_lba, synth_pose

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "lba_reference.npz")
SMALL = dict(n_kf=6, n_points=200, n_pt_obs=600, n_lines=20, n_line_obs=20, n_plane_obs=(6, 2, 1))
GOLD_CASES = [dict(seed=1, **SMALL), dict(seed=2, n_kf=8, n_fixed=2, n_points=300, n_pt_obs=900, n_lines=0, n_line_obs=0, n_plane_obs=(0, 0, 0)),
              dict(seed=3, n_kf=10, n_points=400, n_pt_obs=1200, n_lines=30, n_line_obs=40, n_plane_obs=(10, 3, 2), line_kf_quirk=True, line_norm3=False,
                   outlier_frac=0.15, plane_outlier_frac=0.3)]
FLOATS = (("kf_Tcw_d", None), ("pt_Xw_d", 5e-4), ("line_Xw_d", 5e-3), ("plane_Xw_d", 2e-5))


def _line_residuals(p, res):
    """EdgeLineProjectXYZ::computeError (include/EdgeLine.h) of both endpoints of every line observation under the optimised estimates."""
    out = np.zeros((len(p["line_obs_kf"]), 2))
    for j, (k, li) in enumerate(zip(p["line_obs_kf"], p["line_obs_line"])):
        T, K = res["kf_Tcw_d"][k], p["kf_K"][k].astype(np.float64)
        for s_ in range(2):
            X = T[:3, :3] @ res["line_Xw_d"][li, 3 * s_:3 * s_ + 3] + T[:3, 3]
            out[j, s_] = p["line_obs_l"][j] @ np.array([K[0] * X[0] / X[2] + K[2], K[1] * X[1] / X[2] + K[3], 1.0])
    return out


def _same(o, r, pose_tol=(5e-6, 1e-5), pt_scale=1.0):
    assert np.array_equal(o["erase_pt"], r["erase_pt"]) and np.array_equal(o["erase_line"], r["erase_line"])
    for t in range(3):
        assert np.array_equal(o["erase_plane"][t], r["erase_plane"][t]), t
    for k in range(len(o["kf_Tcw_d"])):
        da, dt = synth_pose.pose_error(o["kf_Tcw_d"][k], r["kf_Tcw_d"][k])
        assert da < pose_tol[0] and dt < pose_tol[1], (k, da, dt)
    for key, tol in FLOATS[1:]:
        if o[key].size:
            assert np.abs(o[key] - r[key]).max() < tol * pt_scale, key
    if o["pt_Xw_d"].size:
        assert np.median(np.abs(o["pt_Xw_d"] - r["pt_Xw_d"]).max(1)) < 5e-6 * pt_scale


def test_oracle_lba_matches_reference_golden():
    g = np.load(GOLD)
    for i, kw in enumerate(GOLD_CASES):
        o = oracle_lib.local_bundle_adjustment(synth_lba.make_lba_problem(**kw))
        r = {k: g[f"c{i}_{k}"] for k in ("kf_Tcw_d", "pt_Xw_d", "line_Xw_d", "plane_Xw_d", "erase_pt", "erase_line")}
        r["erase_plane"] = [g[f"c{i}_erase_plane{t}"] for t in range(3)]
        _same(o, r)


def test_oracle_lba_agrees_with_compiled_reference_g2o():
    cases = list(GOLD_CASES)
    cases += [dict(seed=10 + s, **SMALL) for s in range(4)]
    cases += [dict(seed=20 + s, **SMALL, line_norm3=False, outlier_frac=0.2, plane_outlier_frac=0.25) for s in range(4)]        # every gate fires
    cases += [dict(seed=30, n_kf=5, n_fixed=3, n_points=150, n_pt_obs=400, n_lines=10, n_line_obs=12, n_plane_obs=(4, 1, 1), mono_frac=1.0),   # mono only
              dict(seed=31, n_kf=5, n_points=150, n_pt_obs=400, n_lines=0, n_line_obs=0, n_plane_obs=(5, 2, 2), mono_frac=0.0),
              dict(seed=32, n_kf=12, n_points=500, n_pt_obs=1500, n_lines=40, n_line_obs=40, n_plane_obs=(12, 3, 2), rot_pert=0.01, trans_pert=0.03, pt_pert=0.05)]
    fired = np.zeros(5, int)
    for kw in cases:
        p = synth_lba.make_lba_problem(**kw)
        o, r = oracle_lib.local_bundle_adjustment(p), ref_lib.ref_local_bundle_adjustment(p)
        _same(o, r, *(((1e-9, 1e-9), 1e-3) if kw.get("mono_frac") == 1.0 else ()))
        if len(p["line_obs_kf"]):
            assert np.abs(_line_residuals(p, o) - _line_residuals(p, r)).max() < 2e-3, kw
        assert o["iterations"] == r["iterations"] and o["iterations"][0] == 5, (kw, o["iterations"], r["iterations"])
        fired += [int(o["erase_pt"].sum()), int(o["erase_line"].sum())] + [int(o["erase_plane"][t].sum()) for t in range(3)]
    assert fired[0] > 0 and fired[1] > 0 and fired[2] > 0, fired


def test_oracle_lba_full_size_agrees_with_compiled_reference_g2o():
    """BASELINE.json's local-map size (20 key frames, 1700 points, 5000 observations, 100 lines, 30 plane observations)."""
    p = synth_lba.make_lba_problem(4)
    _same(oracle_lib.local_bundle_adjustment(p), ref_lib.ref_local_bundle_adjustment(p))


def test_oracle_lba_agrees_with_the_reference_function_itself():
    """Optimizer::LocalBundleAdjustment(KeyFrame*, bool*, Map*) called AS IT IS (src/Optimizer.cc compiled unmodified into libmatch_ref.so with KeyFrame.cc,
    MapPoint.cc, MapLine.cpp, MapPlane.cc, Map.cc): oracle/ref/match_driver.cc builds the key frames (covisibility list, feature slots), map points / lines /
    planes and their observation maps from the problem arrays, calls the function, and reads back the poses / positions it wrote (float) and the feature
    slots it cleared.  The local / fixed key-frame discovery, graph construction, both optimisations, the gating, the erasures (with the bad-landmark cascade
    of EraseObservation) and the write-back are all the reference's.  A cleared slot means "this observation was erased" or "its landmark went bad";
    pt_bad / line_bad / plane_bad tell which.  Line edges hang on the current key frame (the reference's quirk), so the problems are made with line_kf_quirk."""
    small = dict(SMALL, line_kf_quirk=True)
    cases = [dict(seed=s, **small) for s in (1, 10, 11, 12)]
    cases += [dict(seed=2, n_kf=8, n_points=300, n_pt_obs=900, n_lines=0, n_line_obs=0, n_plane_obs=(0, 0, 0)),
              dict(seed=30, n_kf=5, n_points=150, n_pt_obs=400, n_lines=10, n_line_obs=12, n_plane_obs=(4, 1, 1), mono_frac=1.0, line_kf_quirk=True)]
    hard = [dict(seed=3, n_kf=10, n_points=400, n_pt_obs=1200, n_lines=30, n_line_obs=40, n_plane_obs=(10, 3, 2), line_kf_quirk=True, line_norm3=False,
                 outlier_frac=0.15, plane_outlier_frac=0.3)] + [dict(seed=20 + s, **small, line_norm3=False, outlier_frac=0.2, plane_outlier_frac=0.25) for s in range(3)]
    big = [dict(seed=4, line_kf_quirk=True)]                               # BASELINE.json's local-map size
    n_bad = n_erased = 0
    for kw in cases + hard + big:
        p = synth_lba.restrict_to_local_planes(synth_lba.make_lba_problem(**kw))
        o, r = oracle_lib.local_bundle_adjustment(p), ref_lib.ref_full_local_bundle_adjustment(p)
        assert np.array_equal(o["erase_pt"] | r["pt_bad"][p["pt_obs_pt"]], r["erase_pt"]), kw
        assert np.array_equal(o["erase_pt"][r["pt_bad"][p["pt_obs_pt"]] == 0], r["erase_pt"][r["pt_bad"][p["pt_obs_pt"]] == 0]), kw
        if len(p["line_obs_line"]):
            assert np.array_equal(o["erase_line"] | r["line_bad"][p["line_obs_line"]], r["erase_line"]), kw
        for t in range(3):
            if len(p["plane_obs_plane"][t]):
                assert np.array_equal(o["erase_plane"][t] | r["plane_bad"][p["plane_obs_plane"][t]], r["erase_plane"][t]), (kw, t)
        tol = (2e-5, 5e-5) if kw in hard else (1e-6, 1e-6)                  # the reference writes float poses back; "hard": see the module docstring
        for k in range(len(o["kf_Tcw_d"])):
            da, dt = synth_pose.pose_error(o["kf_Tcw_d"][k], r["kf_Tcw_d"][k])
            assert da < tol[0] and dt < tol[1], (kw, k, da, dt)
        # the reference iterates pointer-keyed containers (std::set / std::map of KeyFrame* / MapPoint*), so its summation order - and on the 20 %-outlier
        # problems the last digits of the result - changes with the heap layout from run to run (measured median 5.1e-6 .. 7.4e-6 on seed 3)
        assert np.median(np.abs(o["pt_Xw_d"] - r["pt_Xw_d"]).max(1)) < (2e-5 if kw in hard else 5e-6) and np.abs(o["pt_Xw_d"] - r["pt_Xw_d"]).max() < 2e-3, kw
        has = np.zeros(len(p["plane_Xw"]), bool)
        has[p["plane_obs_plane"][0]] = True
        if has.any():
            d = np.minimum(np.abs(o["plane_Xw_d"] - r["plane_Xw_d"]).max(1), np.abs(o["plane_Xw_d"] + r["plane_Xw_d"]).max(1))[has]
            assert d.max() < 5e-5, (kw, d.max())
        n_bad += int(r["pt_bad"].sum()); n_erased += int(o["erase_pt"].sum())
    assert n_bad > 50 and n_erased > 1000
