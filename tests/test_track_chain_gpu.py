"""GPU: the device-resident tracking chain (pslam_track_sequence, BASELINE.json config 3: TUM fr3-shaped synthetic 640x480 sequence, full
Tracking + PoseOptimization, pose tolerance 1e-4 rad / 1e-3 m) against THE SAME CHAIN RUN THROUGH THE REFERENCE'S OWN FUNCTIONS on the CPU:
src/ORBextractor.cc (liborb_ref), Frame::ComputeStereoFromRGBD, ORBmatcher::SearchByProjection x2 with Frame::isInFrustum and the reference's
feature grid, Optimizer::PoseOptimization(Frame*) (libmatch_ref: src/ORBmatcher.cc, Frame.cc, Optimizer.cc + Thirdparty/g2o compiled unmodified);
only the glue between them (Tracking::TrackWithMotionModel / TrackLocalMap / the velocity update: pose products, the outlier sweep, the skip
flags of SearchLocalPoints) is restated here in numpy with cv::Mat's float-storage / double-accumulation convention.  Where oracle/_ref is
absent, the recorded answers of those functions stand in (ref_lib); the key points fed on are the oracle's, checked equal to the reference's."""
import numpy as np
import pytest

import oracle_lib
import ref_lib
from planarslam_b200 import synth, synth_map, synth_pose

pytestmark = pytest.mark.gpu
N_FRAMES = 64


def _mm(a, b):
    return (np.asarray(a, np.float64) @ np.asarray(b, np.float64)).astype(np.float32)


def _inv_pose(T):
    R, t = T[:3, :3], T[:3, 3]
    out = np.eye(4, dtype=np.float32)
    out[:3, :3] = R.T
    out[:3, 3] = (-(R.T.astype(np.float64)) @ t.astype(np.float64)).astype(np.float32)
    return out


def _pose_problem(fa, matches, m, T0):
    idx = np.nonzero(matches >= 0)[0]
    k = fa["keys_un"][idx]
    inv_sigma2 = (np.float32(1.0) / (synth_map.SCALE_FACTORS ** 2).astype(np.float32)).astype(np.float32)
    z = np.zeros((0, 4), np.float32)
    p = dict(fx=synth.TUM3_K[0], fy=synth.TUM3_K[1], cx=synth.TUM3_K[2], cy=synth.TUM3_K[3], bf=40.0, Xw=np.ascontiguousarray(m["pos"][matches[idx]]),
             obs=np.ascontiguousarray(np.stack([k["x"], k["y"], fa["u_right"][idx]], 1), np.float32), inv_sigma2=np.ascontiguousarray(inv_sigma2[k["octave"]]),
             line_Xw=np.zeros((0, 6)), line_obs=np.zeros((0, 3)), plane_meas=z, plane_map=z, par_meas=z, par_map=z, ver_meas=z, ver_map=z,
             Tcw0=np.ascontiguousarray(T0, np.float32), **synth_pose.PLANE_SETTINGS)
    return p, idx


def _optimise(fa, matches, m, T):
    p, idx = _pose_problem(fa, matches, m, T)
    if len(idx) < 3:
        return T, len(idx), 0
    r = ref_lib.ref_full_pose_optimization(p, False)
    matches[idx[r["outlier_pt"] != 0]] = -1
    return np.ascontiguousarray(r["Tcw"], np.float32), len(idx), int(r["n_inliers"])


def _reference_chain(frames, m, T0):
    s_last, s_map = ref_lib.ref_search_by_projection_last, ref_lib.ref_search_by_projection_map
    poses, stats = [], []
    T = np.ascontiguousarray(T0, np.float32)
    last = vel = fa_prev = matches_prev = None
    for t, (g, d) in enumerate(frames):
        kps, desc = oracle_lib.orb_extract(g)
        rk, rd = ref_lib.ref_orb_extract(g)
        assert ref_lib.same(rk, kps) and ref_lib.same(rd, desc), t
        fa = synth_map.frame_arrays(kps, desc, d)
        matches = np.full(fa["n"], -1, np.int32)
        st = [0, 0, 0, 0]
        if t > 0:
            last = T
            T = _mm(vel, last) if t > 1 else last.copy()
            lf = dict(n=fa_prev["n"], keys=fa_prev["keys_un"], map_point=matches_prev, outlier=np.zeros(fa_prev["n"], np.uint8), Tcw=last)
            _, matches = s_last(synth_map.frame_view(fa, T), lf, m, 15.0, False, True, matches)
            matches = matches.copy()
            T, st[0], st[1] = _optimise(fa, matches, m, T)
        mm = dict(m)
        mm["skip"] = m["skip"].copy()
        mm["skip"][matches[matches >= 0]] = 1
        _, matches, _ = s_map(synth_map.frame_view(fa, T), mm, 3.0, 0.8, matches)
        matches = matches.copy()
        T, st[2], st[3] = _optimise(fa, matches, m, T)
        if t > 0:
            vel = _mm(T, _inv_pose(last))
        poses.append(T.copy()); stats.append(st)
        fa_prev, matches_prev = fa, matches
    return np.stack(poses), np.array(stats, np.int32)


def test_track_sequence_matches_the_reference_chain():
    from planarslam_b200._lib import Context
    from planarslam_b200.tracking import Tracker
    frames = [synth.render_frame(2, f)[:2] for f in range(N_FRAMES)]
    # map snapshot: the key points of every 8th frame, back-projected with the rendered depth at the true pose
    parts = []
    for f in range(0, N_FRAMES, 8):
        k, de = oracle_lib.orb_extract(frames[f][0])
        parts.append(synth_map.map_from_frame(synth_map.frame_arrays(k, de, frames[f][1]), synth_map.true_pose(f)))
    m = {key: np.concatenate([p[key] for p in parts]) for key in ("pos", "normal", "max_distance", "min_distance", "desc", "skip", "has_obs")}
    m["n"] = len(m["skip"])
    T0 = synth_map.true_pose(0).astype(np.float32)
    ref_poses, ref_stats = _reference_chain(frames, m, T0)
    ctx = Context(640, 480, max_batch=N_FRAMES)
    tr = Tracker(ctx)
    tr.set_map(m)
    poses, stats = tr.track(np.stack([f[0] for f in frames]), np.stack([f[1] for f in frames]), T0)
    worst = (0.0, 0.0)
    for t in range(N_FRAMES):
        da, dt = synth_pose.pose_error(poses[t], ref_poses[t])
        worst = (max(worst[0], da), max(worst[1], dt))
        assert da < 1e-4 and dt < 1e-3, (t, da, dt, stats[t], ref_stats[t])
        ea, et = synth_pose.pose_error(poses[t], synth_map.true_pose(t))
        assert ea < 5e-3 and et < 2e-2, (t, ea, et)                       # and the chain actually tracks the camera
    assert (stats[:, 3] > 100).all(), stats[:, 3].min()
    # the match / inlier counts agree frame by frame unless a pose differing in its last float digits moved a key point across a window border
    assert np.mean(np.all(stats == ref_stats, axis=1)) > 0.8, (stats[:8], ref_stats[:8])
    print("worst pose difference vs the reference chain:", worst)
