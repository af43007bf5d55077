"""CPU: the loop-closure / relocalisation candidate oracle (oracle/loopclose.cc) pinned against THE REFERENCE'S OWN code: src/KeyFrameDatabase.cc
(DetectLoopCandidates :76-197, DetectRelocalizationCandidates :199-305), DBoW2's L1 scoring (Thirdparty/DBoW2/DBoW2/ScoringObject.cpp) and
src/ORBmatcher.cc (SearchByBoW(KeyFrame*, KeyFrame*, ...) :526-659), compiled unmodified into oracle/_ref/libmatch_ref.so; the driver only builds KeyFrame
objects (BowVectors, covisibility lists, map points) from the plain arrays."""
import os

import numpy as np
import pytest

import oracle_lib
import ref_lib
from planarslam_b200 import synth_lines

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "loopclose_reference.npz")

CASES = [dict(seed=0), dict(seed=1, n_kf=150, n_similar=25), dict(seed=2, n_kf=600, n_words=3000, words_per_kf=500, n_similar=80),
         dict(seed=3, n_kf=60, n_similar=0), dict(seed=4, n_kf=40, n_words=400, words_per_kf=120, n_similar=10), dict(seed=5, n_kf=1, n_similar=1),
         dict(seed=6, n_kf=300, n_words=100000, words_per_kf=900, n_similar=30)]
# the cases whose reference answers are committed as tests/golden/loopclose_reference.npz (tools/make_golden_loopclose.py)
GOLD_CASES, GOLD_MIN_SCORES, GOLD_KF_SEEDS = CASES[:5], (0.0, 0.03), (0, 1)


@pytest.mark.parametrize("case", CASES, ids=lambda c: f"seed{c['seed']}")
def test_detect_loop_candidates_identical_to_compiled_reference(case):
    db = synth_lines.make_bow_database(**case)
    some = 0
    for min_score in (0.0, 0.01, 0.03, 0.08):
        c, w, s = oracle_lib.detect_loop_candidates(db, min_score)
        rc, rw, rs = ref_lib.ref_detect_loop_candidates(db, min_score)
        assert ref_lib.same(c, rc), (min_score, c, rc)
        assert ref_lib.same(w, rw)
        assert ref_lib.same(s, rs)            # float scores bit-identical (and evaluated for the same key frames: the sentinel elsewhere)
        some += len(c)
    if case.get("n_similar", 40) >= 10:
        assert some > 0


@pytest.mark.parametrize("case", CASES, ids=lambda c: f"seed{c['seed']}")
def test_detect_relocalization_candidates_identical_to_compiled_reference(case):
    db = synth_lines.make_bow_database(**case)
    n_kf = len(db["off"]) - 1
    rng = np.random.default_rng(case["seed"])
    for stale in (np.zeros(n_kf, np.float32), rng.uniform(0, 0.05, n_kf).astype(np.float32)):     # mRelocScore left by earlier queries
        c, w, s = oracle_lib.detect_relocalization_candidates(db, stale)
        rc, rw, rs = ref_lib.ref_detect_relocalization_candidates(db, stale)
        assert ref_lib.same(c, rc), (c, rc)
        assert ref_lib.same(w, rw)
        assert ref_lib.same(s, rs)


def test_search_by_bow_kf_identical_to_compiled_reference():
    total = 0
    for seed in range(5):
        kf1, kf2 = synth_lines.make_bow_kf_pair(seed, **(dict(n_kf=400, n_f=380, n_nodes=90) if seed < 3 else {}))
        for ratio, ori in ((0.75, True), (0.75, False), (0.9, True), (0.6, True)):
            n, m = oracle_lib.search_by_bow_kf(kf1, kf2, ratio, ori)
            rn, rm = ref_lib.ref_search_by_bow_kf(kf1, kf2, ratio, ori)
            assert n == rn and ref_lib.same(m, rm)
            assert n == int((m >= 0).sum())
            total += n
    assert total > 1000


def _edge_databases():
    base = synth_lines.make_bow_database(seed=9, n_kf=50, n_words=600, words_per_kf=150, n_similar=12)
    yield "all connected", dict(base, connected=np.ones(50, np.uint8))
    empty_q = dict(base, q_word=np.zeros(0, np.int32), q_val=np.zeros(0))
    yield "empty query", empty_q
    off = base["off"].copy()
    cut = off[21] - off[20]                       # key frame 20 loses all its words
    word = np.concatenate([base["word"][:off[20]], base["word"][off[21]:]])
    val = np.concatenate([base["val"][:off[20]], base["val"][off[21]:]])
    off2 = off.copy(); off2[21:] -= cut
    yield "key frame without words", dict(base, off=off2, word=word, val=val)
    covis = base["covis"].copy(); covis[:, :] = -1
    yield "no covisibility", dict(base, covis=covis)
    covis = base["covis"].copy(); covis[:, 0] = 25
    yield "everyone's best neighbour is key frame 25", dict(base, covis=covis)


def test_candidate_edge_cases_identical_to_compiled_reference():
    for name, db in _edge_databases():
        for min_score in (0.0, 0.02, 0.9):
            c, w, s = oracle_lib.detect_loop_candidates(db, min_score)
            rc, rw, rs = ref_lib.ref_detect_loop_candidates(db, min_score)
            assert ref_lib.same(c, rc) and ref_lib.same(w, rw) and ref_lib.same(s, rs), (name, min_score)
        n_kf = len(db["off"]) - 1
        c, w, s = oracle_lib.detect_relocalization_candidates(db, np.full(n_kf, 0.01, np.float32))
        rc, rw, rs = ref_lib.ref_detect_relocalization_candidates(db, np.full(n_kf, 0.01, np.float32))
        assert ref_lib.same(c, rc) and ref_lib.same(w, rw) and ref_lib.same(s, rs), name


def test_oracle_matches_loopclose_golden():
    """The oracle against the committed answers of the reference's own code (no compiled reference needed: runs on the GPU box too)."""
    g = np.load(GOLD)
    for i, case in enumerate(GOLD_CASES):
        db = synth_lines.make_bow_database(**case)
        for j, ms in enumerate(GOLD_MIN_SCORES):
            c, w, s = oracle_lib.detect_loop_candidates(db, ms)
            assert np.array_equal(c, g[f"loop{i}_{j}_cand"]) and np.array_equal(w, g[f"loop{i}_{j}_words"]) and np.array_equal(s, g[f"loop{i}_{j}_score"]), (case, ms)
        stale = np.random.default_rng(case["seed"]).uniform(0, 0.05, len(db["off"]) - 1).astype(np.float32)
        c, w, s = oracle_lib.detect_relocalization_candidates(db, stale)
        assert np.array_equal(c, g[f"reloc{i}_cand"]) and np.array_equal(w, g[f"reloc{i}_words"]) and np.array_equal(s, g[f"reloc{i}_score"]), case
    for seed in GOLD_KF_SEEDS:
        kf1, kf2 = synth_lines.make_bow_kf_pair(seed, n_kf=400, n_f=380, n_nodes=90)
        n, m = oracle_lib.search_by_bow_kf(kf1, kf2, 0.75, True)
        assert n == int(g[f"bowkf{seed}_n"][0]) and np.array_equal(m, g[f"bowkf{seed}_match"]), seed
