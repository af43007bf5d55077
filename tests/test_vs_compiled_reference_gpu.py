"""GPU: the CUDA path against THE REFERENCE'S OWN CODE, directly.  oracle/_ref/*.so are the reference's ORB extractor, plane extractor
and DBoW2 compiled unmodified in the build container (oracle/ref/, `make -C oracle ref`); they travel to the GPU box as prebuilt
libraries.  The CUDA outputs must be byte-identical to theirs (same bar as against the oracle, which the CPU suite proves identical
to these libraries).  Where the libraries are absent, their recorded answers (ref_lib) stand in."""
import os
import tempfile

import numpy as np
import pytest

import ref_lib
from planarslam_b200 import synth, synth_lines

pytestmark = pytest.mark.gpu


def test_orb_cuda_identical_to_reference_code():
    from planarslam_b200.orb import ORBextractor
    ext = ORBextractor(1000, 1.2, 8, 20, 7, max_batch=4)
    imgs = np.stack([synth.render_frame(2, 0)[0], synth.render_frame(2, 17)[0], synth.polygon_image(1), synth.render_frame(9, 4)[0]])
    kps, desc = ext.extract_batch(imgs)
    for f in range(len(imgs)):
        rk, rd = ref_lib.ref_orb_extract(imgs[f])                 # src/ORBextractor.cc, quadtree address ties = creation order
        assert len(kps[f]) == len(rk) >= 900, f
        assert ref_lib.same(rk, kps[f]), f"key points differ from the reference's ORBextractor, frame {f}"
        assert ref_lib.same(rd, desc[f]), f"descriptors differ from the reference's ORBextractor, frame {f}"


def _peac_vs_reference(depth, min_planes):
    from planarslam_b200.planes import PlaneDetection
    K = np.array([[535.4, 0, 320.1], [0, 539.2, 247.6], [0, 0, 1]], np.float32)
    scale = np.float32(1.0 / 5000.0)
    pd = PlaneDetection(max_batch=len(depth))
    res = pd.run_batch(depth, K, scale)
    n_planes = 0
    for f in range(len(depth)):
        labels, planes, members = res[f]
        rl, rp, rm = ref_lib.ref_peac_run(depth[f])               # src/PlaneExtractor.cpp + include/peac/*.hpp
        assert ref_lib.same(rl, labels), f"membershipImg differs from the reference's PEAC, frame {f}"
        assert len(planes) == len(rp), f
        for i, (d8, N) in enumerate(rp):
            assert planes["normal"][i].tobytes() == d8[0:3].tobytes() and planes["center"][i].tobytes() == d8[3:6].tobytes(), (f, i)
            assert planes["mse"][i] == d8[6] and planes["curvature"][i] == d8[7] and planes["N"][i] == N, (f, i)
            assert ref_lib.same(rm[i], members[i]), (f, i)
        n_planes += len(rp)
    assert n_planes >= min_planes


def test_peac_cuda_identical_to_reference_code():
    _peac_vs_reference(np.stack([synth.render_frame(2, f)[1] for f in (0, 17, 40, 55)]), 8)


def test_peac_cuda_identical_to_reference_code_many_planes():
    _peac_vs_reference(np.stack([synth.piecewise_planar_depth(2, n_rect=8), synth.piecewise_planar_depth(5, n_rect=11, curved=False),
                                 synth.piecewise_planar_depth(11, n_rect=17, curved=False)]), 20)


def test_bow_transform_cuda_identical_to_reference_code():
    from planarslam_b200._lib import Context
    from planarslam_b200.matcher import bow_transform
    ctx = Context(640, 480, 1)
    with tempfile.TemporaryDirectory() as td:
        for seed, (k, L, lup) in enumerate([(10, 4, 4), (10, 3, 2), (6, 5, 4)]):
            voc = synth_lines.make_vocabulary(seed, k=k, L=L)
            feats = synth_lines.make_features_for_vocabulary(seed, voc, n=1000)
            path = os.path.join(td, f"voc{seed}.txt")
            ref_lib.write_vocabulary_txt(voc, path)
            r = ref_lib.RefVocabulary(path).transform(feats, lup)        # Thirdparty/DBoW2 TemplatedVocabulary::transform
            g = bow_transform(ctx, voc, feats, lup)
            for key in ("word_id", "word_val", "node_id", "node_off", "node_feat"):
                assert ref_lib.same(g[key], r[key]), (seed, key)
