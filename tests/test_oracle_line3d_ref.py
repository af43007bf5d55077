"""CPU: the 3-D line-fit oracle (oracle/line3d.cc) pinned against THE REFERENCE'S OWN CODE: compPt3dCov, extract3dline_mahdist, verify3dLine,
mah_dist3d_pt_line and computeLine3d_svd of src/LineExtractor.cpp compiled unmodified (oracle/_ref/libline3d_ref.so, `make -C oracle ref`;
cv::Mat algebra and cv::SVD from the stand-ins of oracle/ref/shims/) drawing from libc's own rand().  Accept flags, inlier sets, end points
(including which end is A and which is B), directors and mvDepthLine must be IDENTICAL - on clean frames and on frames whose depth is corrupted
enough for the RANSAC to iterate, reject hypotheses and refit.  Golden copies in tests/golden/line3d_reference.npz."""
import os

import numpy as np

import oracle_lib
import ref_lib
from planarslam_b200 import synth

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "line3d_reference.npz")
KEYS = ("valid", "n_points", "n_inliers", "inliers", "lines3d", "depth_line", "director")
CASES = [(0, 0.0, 0.0, 1), (3, 0.15, 0.006, 5), (5, 0.3, 0.012, 9), (6, 0.45, 0.02, 2 ** 31 + 3)]       # (frame seed, outlier fraction, sigma [m], srand seed)


def case_inputs(s, frac, sigma):
    gray, d16, _, _ = synth.render_frame(seed=s, frame=3 * s)
    kl, _ = oracle_lib.extract_line_segments(gray, 40)
    if frac > 0:
        d16 = synth.noisy_depth(d16, s, frac, sigma)
    return kl, d16.astype(np.float32) * np.float32(1.0 / synth.DEPTH_FACTOR)


def test_oracle_line3d_matches_reference_golden():
    g = np.load(GOLD)
    for s, frac, sigma, seed in CASES:
        kl, depth = case_inputs(s, frac, sigma)
        o = oracle_lib.lines3d_frame(kl, depth, synth.TUM3_K, seed=seed)
        for k in KEYS:
            assert np.array_equal(o[k], g[f"c{s}_{k}"], equal_nan=(k == "director")), (s, k)


def test_oracle_line3d_identical_to_compiled_reference():
    n_valid = n_draws = 0
    for s in range(10):
        for frac, sigma in ((0.0, 0.0), (0.1 + 0.04 * s, 0.004 * (s + 1))):
            kl, depth = case_inputs(s, frac, sigma)
            for seed, skip in ((1, 0), (40 + s, 3 * s)):
                o = oracle_lib.lines3d_frame(kl, depth, synth.TUM3_K, seed=seed, skip=skip)
                r = ref_lib.ref_lines3d_frame(kl, depth, synth.TUM3_K, seed=seed, skip=skip)
                for k in KEYS:
                    assert ref_lib.same(o[k], r[k]), (s, frac, seed, k)
                n_valid += int(r["valid"].sum())
                n_draws += o["n_drawn"]
    assert n_valid > 800 and n_draws > 8000                      # the noisy frames make the RANSAC work: ~10 draws per line on average
    icl = (481.2, -480.0, 319.5, 239.5)                          # Examples/RGB-D/ICL.yaml: fy < 0
    kl, depth = case_inputs(2, 0.2, 0.01)
    o, r = oracle_lib.lines3d_frame(kl, depth, icl, seed=3), ref_lib.ref_lines3d_frame(kl, depth, icl, seed=3)
    assert all(ref_lib.same(o[k], r[k]) for k in KEYS)


def test_oracle_line3d_identical_to_frame_is_line_good_itself():
    """Frame::isLineGood(imGray, imDepth, K) called AS IT IS (src/Frame.cc + src/LineExtractor.cpp compiled unmodified into libmatch_ref.so): the sampling /
    back-projection loop that libline3d_ref's driver restates is the reference's here too.  mvDepthLine and mvLines3D bit-identical to the oracle."""
    n_valid = 0
    for s in range(10):
        for frac, sigma in ((0.0, 0.0), (0.1 + 0.04 * s, 0.004 * (s + 1))):
            kl, depth = case_inputs(s, frac, sigma)
            for seed, skip in ((1, 0), (40 + s, 3 * s)):
                o = oracle_lib.lines3d_frame(kl, depth, synth.TUM3_K, seed=seed, skip=skip)
                dl, l3 = ref_lib.ref_full_lines3d_frame(kl, depth, synth.TUM3_K, seed=seed, skip=skip)
                assert ref_lib.same(o["depth_line"], dl) and ref_lib.same(o["lines3d"], l3), (s, frac, seed)
                assert np.array_equal(o["valid"].astype(bool), np.any(o["lines3d"] != 0, axis=1)), (s, frac, seed)     # o["lines3d"] is l3
                n_valid += int(o["valid"].sum())
    assert n_valid > 800
