"""CPU: the ORB oracle (oracle/orb.cc) pinned against THE REFERENCE'S OWN CODE.

  * live: src/ORBextractor.cc compiled unmodified from /root/reference (oracle/_ref/liborb_ref.so, `make -C oracle ref`) against the
    stand-ins of oracle/ref/shims/: containers plus the six OpenCV image primitives, which are the oracle's restatements pinned
    bit-for-bit to cv2 4.13 (tests/test_oracle_cvprims.py).  Cell grid, FAST threshold fallback, quadtree distribution, orientation,
    steered BRIEF and coordinate scaling are the reference's code.  Key points (all seven fields, output order) and descriptors must
    be BYTE-IDENTICAL.  DistributeOctTree breaks ties between equally populated nodes by heap address (src/ORBextractor.cc:684), i.e.
    by the allocator; the comparison runs the reference on a monotonic arena (address order = creation order, the documented
    convention of the oracle and the CUDA path) - with glibc malloc about 1 % of the key points change.
  * golden: outputs of that library committed as tests/golden/orb_reference.npz (tools/make_golden_ref.py), checked everywhere."""
import os
import sys

import numpy as np

import oracle_lib
import ref_lib
from planarslam_b200 import synth

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
from make_golden_ref import ORB_CASES, digest, orb_image  # noqa: E402

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "orb_reference.npz")


def _oracle(img, nfeatures=1000, scale=1.2, nlevels=8, ini_th=20, min_th=7):
    return oracle_lib.orb_extract(img, nfeatures, scale, nlevels, ini_th, min_th)


def test_oracle_orb_matches_reference_golden():
    g = np.load(GOLD)
    for name, ikw, okw in ORB_CASES:
        k, d = _oracle(orb_image(ikw), **okw)
        assert len(k) == int(g[name + "_n"][0]) > 400, name
        assert np.array_equal(digest(k), g[name + "_kps_sha1"]) and np.array_equal(digest(d), g[name + "_desc_sha1"]), name
        if name.startswith("tum"):
            assert np.array_equal(k.view(np.uint8).reshape(len(k), 28), g[name + "_kps"]) and np.array_equal(d, g[name + "_desc"]), name


def test_oracle_orb_identical_to_compiled_reference():
    cases = [(synth.render_frame(seed=s, frame=3 * s)[0], {}) for s in range(8)]
    g1 = synth.render_frame(seed=1, frame=3)[0]
    cases += [(g1, dict(nfeatures=500)), (g1, dict(nfeatures=2000)), (g1, dict(nlevels=4, scale=1.5)), (g1, dict(ini_th=40, min_th=10))]
    cases += [(synth.render_frame(seed=2, frame=6, width=1280, height=960)[0], dict(nfeatures=2000)), (synth.render_frame(seed=3, frame=9, width=320, height=240)[0], {})]
    cases += [(synth.polygon_image(11), {}), (np.full((480, 640), 90, np.uint8), {}), (np.random.default_rng(0).integers(0, 256, (480, 640), dtype=np.uint8), {})]
    total = 0
    for i, (img, kw) in enumerate(cases):
        k, d = ref_lib.ref_orb_extract(img, **kw)
        ok, od = _oracle(img, **kw)
        assert len(k) == len(ok), i
        assert ref_lib.same(k, ok), i
        assert ref_lib.same(d, od), i
        total += len(k)
    assert total > 15000


def test_allocator_dependence_of_the_reference_is_confined_to_ties():
    """With glibc malloc the reference still finds the same number of key points per level and all but the few that depend on which
    of several equally populated quadtree nodes is split last."""
    for s in (0, 4):
        img = synth.render_frame(seed=s, frame=3 * s)[0]
        k0, _ = ref_lib.ref_orb_extract(img, monotonic_alloc=False)
        k1, _ = _oracle(img)                                           # == the reference on the monotonic arena
        assert ref_lib.same(ref_lib.ref_orb_extract(img, monotonic_alloc=True)[0], k1)
        assert len(k0) == len(k1)
        assert np.array_equal(np.bincount(k0["octave"], minlength=8), np.bincount(k1["octave"], minlength=8))
        a = {(int(q["octave"]), float(q["x"]), float(q["y"])) for q in k0}
        b = {(int(q["octave"]), float(q["x"]), float(q["y"])) for q in k1}
        assert len(a - b) <= 0.03 * len(a)


def test_oracle_orb_fuzz_sizes_settings_and_content_vs_compiled_reference():
    """Random image sizes (160 .. 700 x 120 .. 520), content, feature counts, level counts and scale factors (pyramids whose top level stays above 40 px: the
    reference itself fails on smaller ones)."""
    import cv2
    rng = np.random.default_rng(2)
    done = 0
    for it in range(60):
        w, h = int(rng.integers(160, 700)), int(rng.integers(120, 520))
        nf, nl, sf = int(rng.choice([300, 1000, 1500])), int(rng.choice([4, 8])), float(rng.choice([1.2, 1.5]))
        if min(w, h) / sf ** (nl - 1) < 40 or w < 0.75 * h:      # portrait frames with (w - 32) / (h - 32) < 0.5 at some level give nIni = 0 root nodes in
            continue                                               # DistributeOctTree (src/ORBextractor.cc:543-550): the reference indexes an empty vector
        kind = it % 3
        if kind == 0:
            g = cv2.GaussianBlur(rng.integers(0, 256, (h, w), dtype=np.uint8), (0, 0), 1.5)
        elif kind == 1:
            g = np.zeros((h, w), np.uint8)
            for _ in range(25):
                cv2.fillPoly(g, [rng.integers(0, [w, h], (4, 2)).astype(np.int32)], int(rng.integers(40, 255)))
        else:
            g = synth.render_frame(seed=it, frame=it, width=w, height=h)[0]
        k, d = ref_lib.ref_orb_extract(g, nfeatures=nf, scale=sf, nlevels=nl)
        ok, od = _oracle(g, nfeatures=nf, scale=sf, nlevels=nl)
        assert len(k) == len(ok) and ref_lib.same(k, ok) and ref_lib.same(d, od), (it, w, h, nf, nl, sf)
        done += 1
    assert done >= 25
