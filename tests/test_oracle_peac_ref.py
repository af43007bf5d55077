"""CPU: the PEAC oracle (oracle/peac.cc) pinned against THE REFERENCE'S OWN CODE.

  * live: src/PlaneExtractor.cpp + include/peac/*.hpp compiled unmodified from /root/reference (oracle/_ref/libpeac_ref.so, built by
    `make -C oracle ref` against the container stand-ins of oracle/ref/shims/ - cv::Mat as a typed buffer, and the 3x3 eigen-solver,
    which is the oracle's Jacobi because Eigen is not in this image).  Label image incl. the raw trail counters, plane parameters,
    supports and member lists must be IDENTICAL.  Where the library is absent, its recorded answers (ref_lib) stand in.
  * golden: the same outputs committed as tests/golden/peac_reference.npz (tools/make_golden_ref.py), checked everywhere."""
import os
import sys

import numpy as np

import oracle_lib
import ref_lib
from planarslam_b200 import synth

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
from make_golden_ref import PEAC_SCENES, digest, peac_scene  # noqa: E402

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "peac_reference.npz")


def test_oracle_peac_matches_reference_golden():
    g = np.load(GOLD)
    for kind, seed in PEAC_SCENES:
        o = oracle_lib.PeacOracle(peac_scene(kind, seed))
        key = f"{kind}{seed}"
        assert np.array_equal(o.labels, g[key + "_labels"].astype(np.int32)), key
        assert len(o.planes) == len(g[key + "_N"]) >= 3
        assert np.array_equal(np.stack([p[0] for p in o.planes]), g[key + "_planes"]), key         # normal, centre, mse, curvature: bit-exact
        assert np.array_equal(np.array([p[1][0] for p in o.planes]), g[key + "_N"]), key
        assert np.array_equal(np.stack([digest(m) for m in o.membership]), g[key + "_members_sha1"]), key


def test_oracle_peac_identical_to_compiled_reference():
    scenes = [synth.render_frame(seed=s, frame=3 * s)[1] for s in range(4)]
    scenes += [synth.piecewise_planar_depth(s, n_rect=6 + s, curved=(s % 2 == 0)) for s in range(12)]
    scenes += [synth.piecewise_planar_depth(40 + s, n_rect=20, noise_mm=6.0, hole_frac=0.04) for s in range(4)]      # noisy, many holes
    scenes.append(np.zeros((480, 640), np.uint16))                                                                       # no depth at all
    scenes.append(np.full((480, 640), 10000, np.uint16))                                                                 # one fronto-parallel plane
    n_planes = 0
    for k, d16 in enumerate(scenes):
        labels, planes, members = ref_lib.ref_peac_run(d16)
        o = oracle_lib.PeacOracle(d16)
        assert ref_lib.same(labels, o.labels), k
        assert len(planes) == len(o.planes), k
        for i, (d8, N) in enumerate(planes):
            if k == len(scenes) - 1:
                # constant depth: every block has the same MSE, so the merge order is decided by the reference's pointer-ordered sets and
                # heap ties (allocator-dependent, AHCPlaneSeg.hpp:188); the sums then round differently in the last bits
                assert np.allclose(d8, o.planes[i][0], rtol=0, atol=1e-12) and N == o.planes[i][1][0], (k, i)
            else:
                assert np.array_equal(d8, o.planes[i][0]) and N == o.planes[i][1][0], (k, i)
            assert ref_lib.same(members[i], o.membership[i]), (k, i)
        n_planes += len(planes)
    assert n_planes > 150


def test_oracle_peac_identical_to_compiled_reference_other_cameras_and_sizes():
    def same(d16, K, sc):
        labels, planes, members = ref_lib.ref_peac_run(d16, K, sc)
        o = oracle_lib.PeacOracle(d16, K, sc)
        assert ref_lib.same(labels, o.labels) and len(planes) == len(o.planes)
        for i, (d8, N) in enumerate(planes):
            assert np.array_equal(d8, o.planes[i][0]) and N == o.planes[i][1][0] and ref_lib.same(members[i], o.membership[i])
        return len(planes)
    tum, s5k = (535.4, 539.2, 320.1, 247.6), np.float32(1.0 / 5000.0)
    d = synth.render_frame(seed=3, frame=9)[1]
    assert same(d, (481.2, -480.0, 319.5, 239.5), s5k) >= 2                                      # Examples/RGB-D/ICL.yaml: fy < 0
    assert same((d // 5).astype(np.uint16), tum, np.float32(1.0 / 1000.0)) >= 2               # another DepthMapFactor
    assert same(synth.render_frame(seed=2, frame=6, width=1280, height=960)[1], (1070.8, 1078.4, 640.2, 495.2), s5k) >= 2
    assert same(synth.render_frame(seed=2, frame=6, width=320, height=240)[1], (267.7, 269.6, 160.0, 123.8), s5k) >= 1
    assert same(synth.piecewise_planar_depth(3)[:475, :633].copy(), tum, s5k) >= 5                # size not a multiple of the 10 x 10 block


def test_oracle_peac_fuzz_vs_compiled_reference():
    """Random image sizes (not multiples of the block size), cameras (some with fy < 0), patch counts, noise levels and hole fractions."""
    rng = np.random.default_rng(5)
    n_planes = 0
    for it in range(24):
        w, h = int(rng.integers(100, 700)), int(rng.integers(100, 520))
        d = synth.piecewise_planar_depth(100 + it, width=max(w, 200), height=max(h, 200), n_rect=int(rng.integers(3, 25)), noise_mm=float(rng.uniform(0.5, 12)),
                                         hole_frac=float(rng.uniform(0, 0.08)), curved=bool(it % 2))[:h, :w].copy()
        K = (float(rng.uniform(300, 700)), float(rng.uniform(300, 700)) * (1 if it % 5 else -1), w / 2 + float(rng.normal(0, 5)), h / 2 + float(rng.normal(0, 5)))
        labels, planes, members = ref_lib.ref_peac_run(d, K)
        o = oracle_lib.PeacOracle(d, K)
        assert ref_lib.same(labels, o.labels) and len(planes) == len(o.planes), (it, w, h)
        for i, (d8, N) in enumerate(planes):
            assert np.array_equal(d8, o.planes[i][0]) and N == o.planes[i][1][0] and ref_lib.same(members[i], o.membership[i]), (it, i)
        n_planes += len(planes)
    assert n_planes > 80
