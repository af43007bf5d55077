"""Frame::ComputeStereoFromRGBD (src/Frame.cc:603-621): oracle vs numpy on the CPU; C ABI vs oracle on the GPU (bit-exact)."""
import numpy as np
import pytest

import oracle_lib
from planarslam_b200 import synth


def _case(seed, n=1000):
    rng = np.random.default_rng(seed)
    _, d16, _, _ = synth.render_frame(seed=seed, frame=3 * seed)
    keys = np.stack([rng.uniform(16, 623, n), rng.uniform(16, 463, n)], 1).astype(np.float32)
    return keys, d16


def test_oracle_matches_numpy():
    keys, d16 = _case(1)
    factor, bf = np.float32(1.0 / synth.DEPTH_FACTOR), np.float32(40.0)
    depth = d16.astype(np.float32) * factor
    ur, dz = oracle_lib.compute_stereo_from_rgbd(keys, keys, depth, float(bf))
    d = depth[keys[:, 1].astype(int), keys[:, 0].astype(int)]
    ok = d > 0
    assert ok.sum() > 900 and (~ok).sum() > 0
    assert np.array_equal(dz[ok], d[ok]) and (dz[~ok] == -1).all() and (ur[~ok] == -1).all()
    assert np.array_equal(ur[ok], keys[ok, 0] - bf / d[ok])


@pytest.mark.gpu
def test_stereo_from_rgbd_gpu_matches_oracle():
    from planarslam_b200._lib import Context
    from planarslam_b200.frame import ComputeStereoFromRGBD
    from planarslam_b200.orb import KEYPOINT_DTYPE
    nf, cap = 3, 1200
    kp = np.zeros((nf, cap), KEYPOINT_DTYPE)
    n = np.array([1000, 1, 1200], np.int32)
    d16 = np.zeros((nf, 480, 640), np.uint16)
    xy = []
    for f in range(nf):
        k, d = _case(f + 2, cap)
        kp["x"][f], kp["y"][f] = k[:, 0], k[:, 1]
        d16[f] = d
        xy.append(k)
    factor, bf = np.float32(1.0 / synth.DEPTH_FACTOR), 40.0
    ctx = Context(640, 480, max_batch=nf)
    ur, dz = ComputeStereoFromRGBD(ctx, kp, n, d16, factor, bf)
    for f in range(nf):
        our, odz = oracle_lib.compute_stereo_from_rgbd(xy[f][:n[f]], xy[f][:n[f]], d16[f].astype(np.float32) * factor, bf)
        assert np.array_equal(ur[f, :n[f]], our) and np.array_equal(dz[f, :n[f]], odz), f
        assert (ur[f, n[f]:] == -1).all() and (dz[f, n[f]:] == -1).all()


def test_oracle_identical_to_frame_compute_stereo_from_rgbd_itself():
    """Frame::ComputeStereoFromRGBD called as it is (src/Frame.cc compiled unmodified into oracle/_ref/libmatch_ref.so)."""
    import ref_lib
    for seed in range(4):
        keys, d16 = _case(seed)
        keys_un = keys + np.float32(0.25) * (seed % 2)
        depth = d16.astype(np.float32) * np.float32(1.0 / synth.DEPTH_FACTOR)
        o, r = oracle_lib.compute_stereo_from_rgbd(keys, keys_un, depth, 40.0), ref_lib.ref_full_compute_stereo_from_rgbd(keys, keys_un, depth, 40.0)
        assert ref_lib.same(o[0], r[0]) and ref_lib.same(o[1], r[1]) and (o[1] > 0).sum() > 900
