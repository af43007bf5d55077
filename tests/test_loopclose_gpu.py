"""GPU: the loop-closure / relocalisation consumer of the key-frame exchange (SURVEY.md 8 f3) through the C ABI - pslam_search_by_bow_kf,
pslam_bow_database_set, pslam_detect_loop_candidates, pslam_detect_relocalization_candidates - against the CPU oracle (bit-identical candidate lists, shared-word
counts, float scores, match lists) and directly against the reference's own compiled src/KeyFrameDatabase.cc / src/ORBmatcher.cc
(oracle/_ref/libmatch_ref.so, or its recorded answers where it is absent)."""
import numpy as np
import pytest

import oracle_lib
import ref_lib
from planarslam_b200 import synth_lines
from test_oracle_loopclose_ref import CASES

pytestmark = pytest.mark.gpu


def test_search_by_bow_kf_matches_oracle_and_reference():
    from planarslam_b200._lib import Context
    from planarslam_b200.matcher import search_by_bow_kf
    ctx = Context(640, 480, 1)
    tot = 0
    for seed in range(6):
        kf1, kf2 = synth_lines.make_bow_kf_pair(seed, n_kf=1000 if seed % 2 else 2000, n_f=1000, n_nodes=300 if seed < 4 else 40)
        for ratio, ori in ((0.75, True), (0.9, False), (0.6, True)):
            n, m = search_by_bow_kf(ctx, kf1, kf2, ratio, ori)
            on, om = oracle_lib.search_by_bow_kf(kf1, kf2, ratio, ori)
            assert n == on and np.array_equal(m, om), (seed, ratio, ori)
            if seed < 3:
                rn, rm = ref_lib.ref_search_by_bow_kf(kf1, kf2, ratio, ori)
                assert n == rn and ref_lib.same(m, rm)
            tot += n
    assert tot > 3000
    # distance exactly TH_LOW = 50 is rejected by this overload (bestDist1 < TH_LOW) and accepted by the (KeyFrame, Frame) one (<=)
    d1 = np.zeros((1, 32), np.uint8)
    d2 = np.zeros((1, 32), np.uint8)
    d2[0, :6] = 0xff
    d2[0, 6] = 0x03                                                           # 50 bits differ
    one = lambda d: dict(desc=d, angle=np.zeros(1, np.float32), has_mp=np.ones(1, np.uint8), node_id=np.array([7], np.int32), node_off=np.array([0, 1], np.int32),
                         node_feat=np.array([0], np.int32))
    n, m = search_by_bow_kf(ctx, one(d1), one(d2), 0.75, False)
    assert n == 0 and m[0] == -1 and oracle_lib.search_by_bow_kf(one(d1), one(d2), 0.75, False)[0] == 0
    d2[0, 6] = 0x01                                                           # 49 bits
    n, m = search_by_bow_kf(ctx, one(d1), one(d2), 0.75, False)
    assert n == 1 and m[0] == 0


@pytest.mark.parametrize("case", CASES, ids=lambda c: f"seed{c['seed']}")
def test_detect_candidates_match_oracle_and_reference(case):
    from planarslam_b200._lib import Context
    from planarslam_b200.matcher import KeyFrameDatabase
    ctx = Context(640, 480, 1)
    db = synth_lines.make_bow_database(**case)
    kfdb = KeyFrameDatabase(ctx, db["off"], db["word"], db["val"], db["covis"])
    for min_score in (0.0, 0.01, 0.03, 0.08):
        c, w, s = kfdb.DetectLoopCandidates(db["q_word"], db["q_val"], min_score, db["connected"])
        oc, ow, os_ = oracle_lib.detect_loop_candidates(db, min_score)
        assert np.array_equal(c, oc), (min_score, c, oc)
        assert np.array_equal(w, ow)
        assert np.array_equal(s, os_)                    # bit-identical floats, evaluated for the same key frames
        rc, rw, rs = ref_lib.ref_detect_loop_candidates(db, min_score)
        assert ref_lib.same(c, rc) and ref_lib.same(w, rw) and ref_lib.same(s, rs)
    n_kf = len(db["off"]) - 1
    rng = np.random.default_rng(case["seed"])
    for stale in (np.zeros(n_kf, np.float32), rng.uniform(0, 0.05, n_kf).astype(np.float32)):
        c, w, s = kfdb.DetectRelocalizationCandidates(db["q_word"], db["q_val"], stale)
        oc, ow, os_ = oracle_lib.detect_relocalization_candidates(db, stale)
        assert np.array_equal(c, oc) and np.array_equal(w, ow) and np.array_equal(s, os_)
        rc, rw, rs = ref_lib.ref_detect_relocalization_candidates(db, stale)
        assert ref_lib.same(c, rc) and ref_lib.same(w, rw) and ref_lib.same(s, rs)


def test_database_argument_checks():
    from planarslam_b200._lib import Context, PslamError
    from planarslam_b200.matcher import KeyFrameDatabase
    ctx = Context(640, 480, 1)
    with pytest.raises(PslamError):                    # words of a BowVector must ascend
        KeyFrameDatabase(ctx, [0, 2], [5, 5], [0.5, 0.5])
    kfdb = KeyFrameDatabase(ctx, [0, 2, 3], [1, 4, 4], [0.5, 0.5, 1.0], np.array([[1, -1], [7, -1]], np.int32))
    with pytest.raises(PslamError):                    # covisibility index outside the database
        kfdb.DetectLoopCandidates([4], [1.0], 0.0)
    empty = KeyFrameDatabase(ctx, [0], [], [])
    with pytest.raises(PslamError):
        empty.DetectLoopCandidates([4], [1.0], 0.0)
