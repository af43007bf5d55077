"""CPU: the Manhattan-frame oracle (oracle/manhattan.cc) pinned against THE REFERENCE'S OWN Tracking::TrackManhattanFrame: src/Tracking.cc compiles unmodified
from /root/reference (oracle/_ref/libtrack_ref.so, linked against libmatch_ref.so) and oracle/ref/track_driver.cc calls the member function - with its
ProjectSN2Conic / ProjectSN2MF / MeanShift helpers, the R_cm aliasing and the final cv::SVD (the OpenCV Jacobi stand-in of oracle/cvsvd.h) - on a Tracking
object that only holds a default-constructed mCurrentFrame (the function reads no other state).  Bar: the returned rotation within 4e-7 per entry (1-3 float
ulp: the oracle does the closing SVD in float, the stand-in of cv::SVD in double), bit-identical when no SVD is applied (fewer than two axes found)."""
import os

import numpy as np

import oracle_lib
import ref_lib
from planarslam_b200.synth_manhattan import make_manhattan

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "manhattan_reference.npz")
CASES = [dict(seed=s) for s in range(8)] + [dict(seed=3, weights=(0.5, 0.5, 0.0), clutter=0.02, n_lines=0), dict(seed=4, weights=(1.0, 0.0, 0.0), clutter=0.0, n_lines=0),
                                            dict(seed=7, n_normals=500, n_lines=5), dict(seed=8, perturb_deg=10.0, noise_deg=4.0), dict(seed=9, clutter=0.4),
                                            dict(seed=10, n_lines=0), dict(seed=11, n_normals=60, n_lines=40)]


def test_manhattan_oracle_matches_reference_golden():
    g = np.load(GOLD)
    for i, kw in enumerate(CASES):
        R_last, normals, dirs, _ = make_manhattan(**kw)
        o = oracle_lib.track_manhattan_frame(R_last, normals, dirs)
        assert np.abs(o["R"] - g[f"R{i}"]).max() < 4e-7, kw


def test_manhattan_oracle_agrees_with_track_manhattan_frame_itself():
    n_svd = n_plain = 0
    for kw in CASES:
        R_last, normals, dirs, _ = make_manhattan(**kw)
        o = oracle_lib.track_manhattan_frame(R_last, normals, dirs)
        r = ref_lib.ref_track_manhattan_frame(R_last, normals, dirs)
        if o["svd_applied"]:
            assert np.abs(o["R"] - r).max() < 4e-7, (kw, np.abs(o["R"] - r).max())
            n_svd += 1
        else:
            assert np.array_equal(o["R"], r), kw
            n_plain += 1
    assert n_svd >= 10 and n_plain >= 1
