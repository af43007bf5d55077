"""CPU: the DBoW2 oracle (oracle/bow_transform.cc) pinned against THE REFERENCE'S OWN CODE: Thirdparty/DBoW2 compiled unmodified from
/root/reference (oracle/_ref/libbow_ref.so, `make -C oracle ref`); synthetic vocabularies are written in the ORBvoc.txt format and read
by the reference's own loadFromTextFile.  BowVector (word ids, tf-idf values after L1 normalisation) and FeatureVector (node ids at
levelsup, feature index lists) must be IDENTICAL, and the L1 score of two bags equal.  Golden copies in tests/golden/bow_reference.npz."""
import os
import sys
import tempfile

import numpy as np

import oracle_lib
import ref_lib
from planarslam_b200 import synth_lines as sl

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
from make_golden_ref import BOW_CASES, bow_case  # noqa: E402

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "bow_reference.npz")
KEYS = ("word_id", "word_val", "node_id", "node_off", "node_feat")


def test_oracle_bow_transform_matches_reference_golden():
    g = np.load(GOLD)
    for seed, k, L, lu in BOW_CASES:
        voc, feats = bow_case(seed, k, L)
        o = oracle_lib.bow_transform(voc, feats, lu)
        for key in KEYS:
            assert np.array_equal(o[key], g[f"s{seed}_{key}"]), (seed, key)


def test_oracle_bow_transform_identical_to_compiled_reference():
    with tempfile.TemporaryDirectory() as td:
        for seed, (k, L) in enumerate([(10, 3), (10, 4), (6, 5), (9, 3), (2, 6)]):
            voc = sl.make_vocabulary(seed, k=k, L=L)
            path = os.path.join(td, f"voc{seed}.txt")
            ref_lib.write_vocabulary_txt(voc, path)
            rv = ref_lib.RefVocabulary(path)
            assert rv.size() == k ** L
            bags = []
            for lu in (4, 2, 0, L, 1):
                feats = sl.make_features_for_vocabulary(seed + 10 + lu, voc, 1000 if lu else 37)
                o, r = oracle_lib.bow_transform(voc, feats, lu), rv.transform(feats, lu)
                for key in KEYS:
                    assert ref_lib.same(o[key], r[key]), (seed, lu, key)
                bags.append(o)
            assert oracle_lib.bow_score_l1(bags[0], bags[1]) == rv.score(bags[0], bags[1])
            assert abs(rv.score(bags[0], bags[0]) - 1.0) < 1e-12
            empty = rv.transform(np.zeros((0, 32), np.uint8), 4)
            assert len(empty["word_id"]) == 0 and len(empty["node_id"]) == 0
