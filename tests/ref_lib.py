"""ctypes access to oracle/_ref/*.so - the REFERENCE's own sources compiled in the build container (make -C oracle ref) against the
stand-in headers of oracle/ref/shims/.  Test infrastructure only; the libraries are prebuilt artefacts on the GPU box."""
import atexit
import ctypes as C
import functools
import hashlib
import inspect
import json
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_DIR = os.path.join(ROOT, "oracle", "_ref", *([os.environ["PSLAM_REF_VARIANT"]] if os.environ.get("PSLAM_REF_VARIANT") else []))   # PSLAM_REF_VARIANT=fast:
                                                                  # the -O3 build bench.py's CPU arm times (oracle/Makefile `fast`); parity tests use the default


def _load(name):
    path = os.path.join(REF_DIR, name)
    if not os.path.exists(path) and os.path.isdir("/root/reference/src"):
        subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), "ref"], check=True, stdout=subprocess.DEVNULL)
    return C.CDLL(path) if os.path.exists(path) else None


# Recorded answers.  The compiled reference exists only where the reference's sources were, so every ref_* call below that a test makes
# is answered, where its library is absent, from the outputs the library gave for the same arguments: tests/golden/reference_calls/<function>.npz,
# keyed by a SHA-1 of the arguments.  Running the tests with PSLAM_REF_RECORD=<dir> where the libraries are built writes <dir>/<function>.npz.
# A call with no recorded answer is an error, never a skip.  Outputs larger than DIGEST_OVER bytes of the functions recorded with digest=True
# (label maps, key points, descriptors, 3-D lines: only ever compared for equality) are kept as their SHA-1; compare them with same().
CALLS_DIR = os.path.join(ROOT, "tests", "golden", "reference_calls")
DIGEST_OVER = 256
_recording = {}


class Digest:
    """A recorded output array kept as its dtype, shape and SHA-1 of its bytes."""

    def __init__(self, descr, shape, sha1):
        self.descr, self.shape, self.sha1 = descr, tuple(shape), sha1

    def __len__(self):
        return self.shape[0]

    def matches(self, a) -> bool:
        a = np.ascontiguousarray(a)
        return str(a.dtype.descr) == self.descr and a.shape == self.shape and _sha1(a) == self.sha1


def _sha1(a):
    """SHA-1 of the values of a: every NaN and both zeros hash alike, as np.array_equal(equal_nan=True) compares them."""
    if a.dtype.kind == "f":
        a = np.where(np.isnan(a), np.nan, a + 0.0).astype(a.dtype)
    return hashlib.sha1(np.ascontiguousarray(a).tobytes()).hexdigest()


def same(a, b) -> bool:
    """a equals b, either of which may be a reference output kept as a Digest (NaNs compare equal, as in a Digest)."""
    if isinstance(b, Digest):
        a, b = b, a
    if isinstance(a, Digest):
        return a.matches(b)
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    if a.dtype.kind == "V" or b.dtype.kind == "V":             # records (key points): byte for byte, as a Digest hashes them
        return a.dtype.itemsize == b.dtype.itemsize and a.shape == b.shape and a.tobytes() == b.tobytes()
    return np.array_equal(a, b, equal_nan=a.dtype.kind == "f" and b.dtype.kind == "f")


def _feed(h, x):
    if isinstance(x, (np.ndarray, np.generic)):
        a = np.ascontiguousarray(x)
        h.update(f"a{a.dtype.descr}{a.shape}".encode())
        h.update(a.tobytes())
    elif isinstance(x, dict):
        h.update(b"d%d" % len(x))
        for k in sorted(x):
            _feed(h, k)
            _feed(h, x[k])
    elif isinstance(x, (list, tuple)):
        h.update(b"l%d" % len(x))
        for v in x:
            _feed(h, v)
    elif isinstance(x, RefVocabulary):
        _feed(h, x.text)
    else:
        h.update(f"{type(x).__name__}:{x!r}".encode())


def _flatten(x, arrays, digest, whole=(), omit=()):
    """JSON description of x whose arrays are appended to arrays.  whole: top-level keys / indices never digested; omit: top-level keys not stored."""
    if isinstance(x, np.ndarray):
        if digest and x.nbytes > DIGEST_OVER:
            a = np.ascontiguousarray(x)
            return {"digest": [str(a.dtype.descr), list(a.shape), _sha1(a)]}
        arrays.append(x)
        return {"a": len(arrays) - 1}
    if isinstance(x, np.generic):
        arrays.append(np.asarray(x))
        return {"s": len(arrays) - 1}
    if isinstance(x, dict):
        return {"d": [[k, _flatten(v, arrays, digest and k not in whole, whole=())] for k, v in x.items() if k not in omit]}
    if isinstance(x, (list, tuple)):
        return {"t" if isinstance(x, tuple) else "l": [_flatten(v, arrays, digest and i not in whole, whole=()) for i, v in enumerate(x)]}
    assert x is None or isinstance(x, (bool, int, float, str)), type(x)
    return {"v": x}


def _unflatten(spec, arrays):
    (kind, v), = spec.items()
    if kind == "a":
        return arrays[v].copy()
    if kind == "s":
        return arrays[v][()]
    if kind == "digest":
        return Digest(*v)
    if kind == "d":
        return {k: _unflatten(s, arrays) for k, s in v}
    if kind in ("t", "l"):
        items = [_unflatten(s, arrays) for s in v]
        return tuple(items) if kind == "t" else items
    return v


def _write_recording():
    out_dir = os.environ["PSLAM_REF_RECORD"]
    os.makedirs(out_dir, exist_ok=True)
    for name, calls in _recording.items():
        path = os.path.join(out_dir, name + ".npz")
        entries = dict(np.load(path)) if os.path.exists(path) else {}
        for key, (spec, arrays) in calls.items():
            entries[key + ".spec"] = np.array(json.dumps({"n": len(arrays), "out": spec}))
            for i, a in enumerate(arrays):
                entries[f"{key}.{i}"] = a
        np.savez_compressed(path, **entries)


_replay = {}
LBA_FLOAT_COPIES = ("kf_Tcw", "pt_Xw", "line_Xw", "plane_Xw")      # the float write-back next to the *_d doubles the tests compare


def _recorded(lib_getter, digest=False, whole=lambda args: (), omit=()):
    """Decorator of a ref_* function: live where lib_getter() finds the library (and recorded if PSLAM_REF_RECORD is set), replayed otherwise.
    Calls with impl != "ref" (the product's adapter) are never recorded.  whole(arguments): top-level outputs of that call stored whole even with
    digest=True; omit: keys of a dict result that no test reads, left out of the recording."""
    def wrap(fn):
        sig = inspect.signature(fn)

        @functools.wraps(fn)
        def call(*args, **kw):
            bound = sig.bind(*args, **kw)
            bound.apply_defaults()
            if bound.arguments.get("impl", "ref") != "ref":
                return fn(*args, **kw)
            live = lib_getter() is not None
            if live and not os.environ.get("PSLAM_REF_RECORD"):
                return fn(*args, **kw)
            h = hashlib.sha1(fn.__qualname__.encode())
            _feed(h, {k: v for k, v in bound.arguments.items() if k != "impl"})
            key = h.hexdigest()
            if live:
                out = fn(*args, **kw)
                if not _recording:
                    atexit.register(_write_recording)
                arrays = []
                spec = _flatten(out, arrays, digest, whole(bound.arguments), omit)
                _recording.setdefault(fn.__qualname__, {})[key] = (spec, arrays)
                return out
            if fn.__qualname__ not in _replay:
                path = os.path.join(CALLS_DIR, fn.__qualname__ + ".npz")
                _replay[fn.__qualname__] = np.load(path) if os.path.exists(path) else {}
            rec = _replay[fn.__qualname__]
            if key + ".spec" not in rec:
                raise LookupError(f"no recorded answer of the compiled reference for this call of {fn.__qualname__} (key {key}): record it with "
                                  "PSLAM_REF_RECORD=<dir> where oracle/_ref is built and add <dir>/*.npz to tests/golden/reference_calls/")
            spec = json.loads(str(rec[key + ".spec"]))
            return _unflatten(spec["out"], [rec[f"{key}.{i}"] for i in range(spec["n"])])
        return call
    return wrap


_peac = None


def peac_lib():
    global _peac
    if _peac is None:
        L = _load("libpeac_ref.so")
        if L is None:
            return None
        vp = C.c_void_p
        L.ref_peac_run.restype = vp
        L.ref_peac_run.argtypes = [vp, C.c_int, C.c_int] + [C.c_float] * 5
        L.ref_peac_free.argtypes = [vp]
        L.ref_peac_num_planes.argtypes = [vp]
        L.ref_peac_labels.argtypes = [vp, vp]
        L.ref_peac_plane.argtypes = [vp, C.c_int, vp, vp]
        L.ref_peac_membership.argtypes = [vp, C.c_int, vp, C.c_int]
        _peac = L
    return _peac


@_recorded(peac_lib, digest=True)
def ref_peac_run(depth16, K=(535.4, 539.2, 320.1, 247.6), scale=np.float32(1.0 / 5000.0)):
    """PlaneDetection::readDepthImage + runPlaneDetection of the reference itself.  Returns (labels int32 [h][w] = membershipImg,
    planes [(normal3 + center3 + mse + curvature, N)], plane_vertices_ lists)."""
    L = peac_lib()
    d = np.ascontiguousarray(depth16, np.uint16)
    h, w = d.shape
    p = C.c_void_p(L.ref_peac_run(d.ctypes.data, w, h, *[float(x) for x in K], float(np.float32(scale))))
    n = L.ref_peac_num_planes(p)
    labels = np.zeros((h, w), np.int32)
    L.ref_peac_labels(p, labels.ctypes.data)
    planes, members = [], []
    for i in range(n):
        d8, N = np.zeros(8), C.c_int()
        L.ref_peac_plane(p, i, d8.ctypes.data, C.byref(N))
        planes.append((d8, N.value))
        buf = np.zeros(h * w, np.int32)
        k = L.ref_peac_membership(p, i, buf.ctypes.data, h * w)
        members.append(buf[:k].copy())
    L.ref_peac_free(p)
    return labels, planes, members


def ref_peac_time(depth16, K=(535.4, 539.2, 320.1, 247.6), scale=np.float32(1.0 / 5000.0)):
    """Run the reference's plane extractor and drop the result (bench.py's CPU baseline)."""
    L = peac_lib()
    d = np.ascontiguousarray(depth16, np.uint16)
    p = C.c_void_p(L.ref_peac_run(d.ctypes.data, d.shape[1], d.shape[0], *[float(x) for x in K], float(np.float32(scale))))
    n = L.ref_peac_num_planes(p)
    L.ref_peac_free(p)
    return n


_orb = None


def orb_lib():
    global _orb
    if _orb is None:
        L = _load("liborb_ref.so")
        if L is None:
            return None
        L.ref_orb_extract.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
        _orb = L
    return _orb


@_recorded(orb_lib, digest=True, whole=lambda a: () if a["monotonic_alloc"] else (0,))
def ref_orb_extract(gray, nfeatures=1000, scale=1.2, nlevels=8, ini_th=20, min_th=7, monotonic_alloc=True, cap=8192):
    """Planar_SLAM::ORBextractor::operator() of the reference itself. Returns (key points as 28-byte records, descriptors [n][32]).
    monotonic_alloc: the library's allocations come from a bump arena, so the quadtree's address ties follow creation order."""
    from planarslam_b200._lib import KEYPOINT_DTYPE
    L = orb_lib()
    g = np.ascontiguousarray(gray, np.uint8)
    h, w = g.shape
    k, d = np.zeros(cap, KEYPOINT_DTYPE), np.zeros((cap, 32), np.uint8)
    n = L.ref_orb_extract(g.ctypes.data, w, h, nfeatures, scale, nlevels, ini_th, min_th, int(bool(monotonic_alloc)), k.ctypes.data, d.ctypes.data, cap)
    assert 0 <= n <= cap, n
    return k[:n].copy(), d[:n].copy()


_bow = None


def bow_lib():
    global _bow
    if _bow is None:
        L = _load("libbow_ref.so")
        if L is None:
            return None
        vp = C.c_void_p
        L.ref_voc_load.restype = vp
        L.ref_voc_load.argtypes = [C.c_char_p]
        L.ref_voc_free.argtypes = [vp]
        L.ref_voc_size.argtypes = [vp]
        L.ref_bow_transform.argtypes = [vp, vp, C.c_int, C.c_int] + [vp] * 6
        L.ref_bow_score.restype = C.c_double
        L.ref_bow_score.argtypes = [vp, vp, vp, C.c_int, vp, vp, C.c_int]
        _bow = L
    return _bow


def write_vocabulary_txt(voc: dict, path: str):
    """The ORBvoc.txt format TemplatedVocabulary::loadFromTextFile reads (Thirdparty/DBoW2/DBoW2/TemplatedVocabulary.h:1338-1434):
    'k L scoring weighting' then one line per node in id order: parent isLeaf 32 descriptor bytes weight.  No trailing newline (the
    loader's while(!f.eof()) would append an empty node)."""
    n = len(voc["word_id"])
    parent = np.zeros(n, np.int64)
    for p in range(n):
        parent[voc["child_id"][voc["child_off"][p]:voc["child_off"][p + 1]]] = p
    lines = [f"{voc['k']} {voc['L']} 0 0"]                     # L1_NORM, TF_IDF
    for i in range(1, n):
        leaf = int(voc["word_id"][i] >= 0)
        lines.append(f"{parent[i]} {leaf} " + " ".join(str(int(b)) for b in voc["desc"][i]) + f" {float(voc['weight'][i])!r}")
    with open(path, "w") as f:
        f.write("\n".join(lines))


class RefVocabulary:
    """ORBVocabulary of the reference (DBoW2 compiled from /root/reference) loaded from a text file."""

    def __init__(self, path: str):
        with open(path) as f:
            self.text = f.read()                   # what identifies the vocabulary in a recorded call
        self.L = bow_lib()
        if self.L is not None:
            self.h = C.c_void_p(self.L.ref_voc_load(path.encode()))
            assert self.h.value, "loadFromTextFile failed"

    @_recorded(bow_lib)
    def size(self):
        return self.L.ref_voc_size(self.h)

    @_recorded(bow_lib, digest=True)
    def transform(self, features: np.ndarray, levelsup: int = 4):
        f = np.ascontiguousarray(features, np.uint8)
        n = len(f)
        o = dict(word_id=np.zeros(n, np.int32), word_val=np.zeros(n), node_id=np.zeros(n, np.int32), node_off=np.zeros(n + 1, np.int32), node_feat=np.zeros(n, np.int32))
        cnt = np.zeros(2, np.int32)
        self.L.ref_bow_transform(self.h, f.ctypes.data, n, levelsup, o["word_id"].ctypes.data, o["word_val"].ctypes.data, o["node_id"].ctypes.data,
                                 o["node_off"].ctypes.data, o["node_feat"].ctypes.data, cnt.ctypes.data)
        nw, nn = int(cnt[0]), int(cnt[1])
        return dict(word_id=o["word_id"][:nw], word_val=o["word_val"][:nw], node_id=o["node_id"][:nn], node_off=o["node_off"][:nn + 1],
                    node_feat=o["node_feat"][:o["node_off"][nn]])

    @_recorded(bow_lib)
    def score(self, a: dict, b: dict) -> float:
        ia, va = np.ascontiguousarray(a["word_id"], np.int32), np.ascontiguousarray(a["word_val"], np.float64)
        ib, vb = np.ascontiguousarray(b["word_id"], np.int32), np.ascontiguousarray(b["word_val"], np.float64)
        return float(self.L.ref_bow_score(self.h, ia.ctypes.data, va.ctypes.data, len(ia), ib.ctypes.data, vb.ctypes.data, len(ib)))

    def __del__(self):
        try:
            self.L.ref_voc_free(self.h)
        except Exception:
            pass


_line3d = None


def line3d_lib():
    global _line3d
    if _line3d is None:
        L = _load("libline3d_ref.so")
        if L is None:
            return None
        L.ref_lines3d_frame.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_uint32, C.c_int] + [C.c_void_p] * 7
        _line3d = L
    return _line3d


@_recorded(line3d_lib, digest=True)
def ref_lines3d_frame(keylines, depth, cam, seed=1, skip=0):
    """The reference's compPt3dCov + extract3dline_mahdist (src/LineExtractor.cpp, libc rand() after srand(seed) and `skip` draws) inside a
    restated Frame::isLineGood loop.  Same outputs as oracle_lib.lines3d_frame (without the draw count)."""
    from oracle_lib import KEYLINE_DTYPE
    L = line3d_lib()
    kl = np.ascontiguousarray(keylines, KEYLINE_DTYPE)
    d = np.ascontiguousarray(depth, np.float32)
    n = len(kl)
    camv = np.asarray(cam, np.float32)
    o = dict(valid=np.zeros(n, np.uint8), depth_line=np.zeros(n, np.float32), lines3d=np.zeros((n, 6)), director=np.zeros((n, 3)),
             n_points=np.zeros(n, np.int32), n_inliers=np.zeros(n, np.int32), inliers=np.zeros(n, np.uint64))
    L.ref_lines3d_frame(kl.ctypes.data, n, d.ctypes.data, d.shape[1], d.shape[0], camv.ctypes.data, seed, skip, o["valid"].ctypes.data, o["depth_line"].ctypes.data,
                        o["lines3d"].ctypes.data, o["director"].ctypes.data, o["n_points"].ctypes.data, o["n_inliers"].ctypes.data, o["inliers"].ctypes.data)
    return o


_pose = None


def pose_lib():
    global _pose
    if _pose is None:
        L = _load("libpose_ref.so")
        if L is None:
            return None
        L.ref_pose_optimization.argtypes = [C.c_void_p] * 9
        L.ref_translation_optimization.argtypes = [C.c_void_p] * 7
        _pose = L
    return _pose


@_recorded(pose_lib)
def ref_pose_optimization(p: dict):
    """PoseOptimization run by the reference's own g2o, edges and Converter (compiled against the Eigen stand-in) on a planarslam_b200.synth_pose problem;
    the graph construction and the four optimise-and-classify rounds are restated in oracle/ref/pose_driver.cc.  Same keys as oracle_lib.pose_optimization."""
    import oracle_lib
    L = pose_lib()
    s = oracle_lib.pose_problem_struct(p)
    T0 = np.ascontiguousarray(p["Tcw0"], np.float32)
    Td = np.zeros((4, 4))
    o = [np.zeros(max(n, 1), np.uint8) for n in (s.n_points, s.n_lines, s.n_planes, s.n_par, s.n_ver)]
    it = np.zeros(4, np.int32)
    n = L.ref_pose_optimization(C.byref(s), T0.ctypes.data, Td.ctypes.data, *[a.ctypes.data for a in o], it.ctypes.data)
    return dict(Tcw_d=Td, n_inliers=n, outlier_pt=o[0][:s.n_points], outlier_line=o[1][:s.n_lines], outlier_plane=o[2][:s.n_planes], outlier_par=o[3][:s.n_par],
                outlier_ver=o[4][:s.n_ver], iterations=it)


@_recorded(pose_lib)
def ref_translation_optimization(p: dict):
    """TranslationOptimization by the reference's g2o and OnlyTranslation edges (oracle/ref/pose_driver.cc)."""
    import oracle_lib
    L = pose_lib()
    s = oracle_lib.pose_problem_struct(p)
    T0 = np.ascontiguousarray(p["Tcw0"], np.float32)
    Td = np.zeros((4, 4))
    o = [np.zeros(max(n, 1), np.uint8) for n in (s.n_points, s.n_lines, s.n_planes)]
    it = np.zeros(4, np.int32)
    n = L.ref_translation_optimization(C.byref(s), T0.ctypes.data, Td.ctypes.data, *[a.ctypes.data for a in o], it.ctypes.data)
    return dict(Tcw_d=Td, n_inliers=n, outlier_pt=o[0][:s.n_points], outlier_line=o[1][:s.n_lines], outlier_plane=o[2][:s.n_planes], iterations=it)


@_recorded(pose_lib, omit=LBA_FLOAT_COPIES)
def ref_local_bundle_adjustment(p: dict) -> dict:
    """LocalBundleAdjustment run by the reference's own g2o (BlockSolver_6_3 + Schur complement + Levenberg-Marquardt), edges and vertices on a
    planarslam_b200.synth_lba problem; the graph construction, the 5 + 10 iterations with the chi-square gating in between and the erase lists are
    restated in oracle/ref/lba_driver.cc.  Same keys as oracle_lib.local_bundle_adjustment."""
    from planarslam_b200 import lba as _lba
    L = pose_lib()
    L.ref_local_bundle_adjustment.argtypes = [C.c_void_p, C.c_void_p]
    s = _lba.problem_struct(p)
    r, o = _lba.result_struct(s)
    rc = L.ref_local_bundle_adjustment(C.byref(s), C.byref(r))
    assert rc == 0
    return _lba.finish(r, o)


_match = None


def match_lib():
    """oracle/_ref/libmatch_ref.so: the reference's ORBmatcher / LSDmatcher / PlaneMatcher with its Frame, KeyFrame, MapPoint, MapLine, MapPlane and Map
    classes, compiled unmodified; oracle/ref/match_driver.cc builds the objects from the C ABI's plain-array views."""
    global _match
    if _match is None:
        _match = _load("libmatch_ref.so")
    return _match


_adapter = None


def adapter_lib():
    """oracle/_ref/libadapter_ref.so: the entry points of match_driver.cc with the product's reference-typed adapter (include/pslam_reference_adapter.hpp) in place
    of the reference's functions (adp_* symbols; oracle/ref/adapter_driver.cc).  Needs libmatch_ref.so and the CUDA library."""
    global _adapter
    if _adapter is None and match_lib() is not None:
        path = os.path.join(REF_DIR, "libadapter_ref.so")
        if not os.path.exists(path) and os.path.isdir("/root/reference/src"):
            subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), "adapter"], check=True, stdout=subprocess.DEVNULL)
        _adapter = C.CDLL(path) if os.path.exists(path) else None
    return _adapter


def _impl(impl):
    return (match_lib(), "ref_") if impl == "ref" else (adapter_lib(), "adp_")


@_recorded(match_lib, digest=True, whole=lambda a: (1,))
def ref_search_by_projection_map(fv: dict, m: dict, th: float, nnratio: float, matches0: np.ndarray, impl: str = "ref"):
    """Tracking::SearchLocalPoints' frustum loop + ORBmatcher::SearchByProjection(Frame&, vector<MapPoint*>&, th) by the reference's own code
    (impl="adp": by the product's adapter class of the same signature, on the same objects).  Same arguments and returns as oracle_lib.search_by_projection_map."""
    import oracle_lib
    lib, pre = _impl(impl)
    fn = getattr(lib, pre + "search_by_projection_map")
    fn.argtypes = [C.c_void_p, C.c_void_p, C.c_float, C.c_float, C.c_void_p, C.c_void_p]
    matches = np.ascontiguousarray(matches0, np.int32).copy()
    in_view = np.zeros(max(m["n"], 1), np.uint8)
    n = fn(C.byref(oracle_lib.frame_view_struct(fv)), C.byref(oracle_lib.map_points_struct(m)), th, nnratio, matches.ctypes.data,
                                       in_view.ctypes.data)
    return n, matches, in_view[:m["n"]]


@_recorded(match_lib)
def ref_search_by_projection_last(fv: dict, lf: dict, m: dict, th: float, mono: bool, check_ori: bool, matches0: np.ndarray, impl: str = "ref"):
    """ORBmatcher::SearchByProjection(Frame& CurrentFrame, const Frame& LastFrame, th, bMono) by the reference's own code (impl="adp": the product's adapter)."""
    import oracle_lib
    lib, pre = _impl(impl)
    fn = getattr(lib, pre + "search_by_projection_last")
    fn.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_int, C.c_int, C.c_void_p]
    matches = np.ascontiguousarray(matches0, np.int32).copy()
    n = fn(C.byref(oracle_lib.frame_view_struct(fv)), C.byref(oracle_lib.last_frame_struct(lf)), C.byref(oracle_lib.map_points_struct(m)),
                                        th, int(mono), int(check_ori), matches.ctypes.data)
    return n, matches


@_recorded(match_lib, digest=True)
def ref_search_by_bow(kf: dict, frame: dict, nnratio: float = 0.7, check_orientation: bool = True, impl: str = "ref"):
    """ORBmatcher::SearchByBoW(KeyFrame*, Frame&, vector<MapPoint*>&) by the reference's own code (impl="adp": the product's adapter).  Same layout as
    oracle_lib.search_by_bow."""
    lib, pre = _impl(impl)
    fn = getattr(lib, pre + "search_by_bow")
    fn.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                    C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_int, C.c_void_p]
    k = {a: np.ascontiguousarray(b) for a, b in kf.items()}
    f = {a: np.ascontiguousarray(b) for a, b in frame.items()}
    nf = len(f["angle"])
    match = np.full(max(nf, 1), -1, np.int32)
    n = fn(len(k["angle"]), k["desc"].ctypes.data, k["angle"].ctypes.data, k["has_mp"].ctypes.data, len(k["node_id"]), k["node_id"].ctypes.data,
                            k["node_off"].ctypes.data, k["node_feat"].ctypes.data, nf, f["desc"].ctypes.data, f["angle"].ctypes.data, len(f["node_id"]),
                            f["node_id"].ctypes.data, f["node_off"].ctypes.data, f["node_feat"].ctypes.data, nnratio, 1 if check_orientation else 0,
                            match.ctypes.data)
    return n, match[:nf]


@_recorded(match_lib)
def ref_lines_in_frustum(frame: dict, pos, normal, max_distance, min_distance, cos_limit: float = 0.5):
    """Frame::isInFrustum(MapLine*, cosLimit) by the reference's own code.  Same arguments / returns as oracle_lib.lines_in_frustum."""
    L = match_lib()
    L.ref_lines_in_frustum.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float] + [C.c_void_p] * 4
    L.ref_lines_in_frustum.restype = None
    fv = np.concatenate([np.asarray(frame["Tcw"], np.float32).ravel(), np.array([frame[k] for k in ("fx", "fy", "cx", "cy", "min_x", "max_x", "min_y", "max_y",
                                                                                                      "log_scale_factor")], np.float32)])
    P, Nn = np.ascontiguousarray(pos, np.float64).reshape(-1, 6), np.ascontiguousarray(normal, np.float64).reshape(-1, 3)
    mx, mn = np.ascontiguousarray(max_distance, np.float32), np.ascontiguousarray(min_distance, np.float32)
    n = len(P)
    o = dict(in_view=np.zeros(n, np.uint8), proj=np.zeros((n, 4), np.float32), level=np.zeros(n, np.int32), view_cos=np.zeros(n, np.float32))
    L.ref_lines_in_frustum(fv.ctypes.data, n, P.ctypes.data, Nn.ctypes.data, mx.ctypes.data, mn.ctypes.data, cos_limit, o["in_view"].ctypes.data, o["proj"].ctypes.data,
                           o["level"].ctypes.data, o["view_cos"].ctypes.data)
    return o


@_recorded(match_lib, digest=True)
def ref_line_search_by_projection(frame: dict, map_lines: dict, th: float, nnratio: float, impl: str = "ref"):
    """LSDmatcher::SearchByProjection(Frame&, vector<MapLine*>&, th) by the reference's own code (impl="adp": the product's adapter).  Same layout as
    oracle_lib.line_search_by_projection."""
    lib, pre = _impl(impl)
    fn = getattr(lib, pre + "line_search_by_projection")
    fn.argtypes = [C.c_int] + [C.c_void_p] * 6 + [C.c_int, C.c_int] + [C.c_void_p] * 6 + [C.c_float, C.c_float, C.c_void_p]
    f = {k: np.ascontiguousarray(v) for k, v in frame.items()}
    m = {k: np.ascontiguousarray(v) for k, v in map_lines.items()}
    nf, nm = len(f["angle"]), len(m["level"])
    assigned = np.full(max(nf, 1), -1, np.int32)
    n = fn(nf, f["pt"].ctypes.data, f["angle"].ctypes.data, f["octave"].ctypes.data, f["desc"].ctypes.data,
                                        f["has_obs"].ctypes.data, f["scale_factors"].ctypes.data, len(f["scale_factors"]), nm, m["skip"].ctypes.data,
                                        m["level"].ctypes.data, m["view_cos"].ctypes.data, m["proj"].ctypes.data, m["desc"].ctypes.data,
                                        m["has_obs"].ctypes.data, th, nnratio, assigned.ctypes.data)
    return n, assigned[:nf]


@_recorded(match_lib, digest=True)
def ref_plane_match(T, fc, mc, bad, off, pts, dTh, aTh, verTh, parTh, impl: str = "ref"):
    """PlaneMatcher::SearchMapByCoefficients by the reference's own code (impl="adp": the product's adapter).  Returns (nmatches, match, vertical, parallel)."""
    lib, pre = _impl(impl)
    fn = getattr(lib, pre + "plane_match")
    fn.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p] + [C.c_float] * 4 + [C.c_void_p] * 3
    T, fc, mc = np.ascontiguousarray(T, np.float32), np.ascontiguousarray(fc, np.float32), np.ascontiguousarray(mc, np.float32)
    bad, off, pts = np.ascontiguousarray(bad, np.uint8), np.ascontiguousarray(off, np.int32), np.ascontiguousarray(pts, np.float32)
    om, ov, op = [np.zeros(max(len(fc), 1), np.int32) for _ in range(3)]
    n = fn(T.ctypes.data, len(fc), fc.ctypes.data, len(mc), mc.ctypes.data, bad.ctypes.data, off.ctypes.data, pts.ctypes.data, dTh, aTh, verTh, parTh,
                          om.ctypes.data, ov.ctypes.data, op.ctypes.data)
    return n, om[:len(fc)], ov[:len(fc)], op[:len(fc)]


@_recorded(match_lib)
def ref_full_pose_optimization(p: dict, translation_only: bool = False, impl: str = "ref"):
    """Optimizer::PoseOptimization(Frame*) / TranslationOptimization(Frame*) THEMSELVES (src/Optimizer.cc compiled unmodified into libmatch_ref.so) on a
    Frame built from a planarslam_b200.synth_pose problem.  Returns dict(Tcw float32 4x4 - the reference writes the pose back as float -, n_inliers, outlier_*)."""
    import oracle_lib
    lib, pre = _impl(impl)                     # impl="adp": pslam_adapter::ref::Optimizer::PoseOptimization(Frame*) on the same Frame
    fn = getattr(lib, pre + "full_pose_optimization")
    fn.argtypes = [C.c_void_p, C.c_void_p, C.c_int] + [C.c_void_p] * 6
    s = oracle_lib.pose_problem_struct(p)
    T0 = np.ascontiguousarray(p["Tcw0"], np.float32)
    T = np.zeros((4, 4), np.float32)
    o = [np.zeros(max(n, 1), np.uint8) for n in (s.n_points, s.n_lines, s.n_planes, s.n_par, s.n_ver)]
    n = fn(C.byref(s), T0.ctypes.data, int(translation_only), T.ctypes.data, *[a.ctypes.data for a in o])
    return dict(Tcw=T, n_inliers=n, outlier_pt=o[0][:s.n_points], outlier_line=o[1][:s.n_lines], outlier_plane=o[2][:s.n_planes],
                outlier_par=o[3][:s.n_par], outlier_ver=o[4][:s.n_ver])


@_recorded(match_lib, omit=LBA_FLOAT_COPIES)
def ref_full_local_bundle_adjustment(p: dict, impl: str = "ref") -> dict:
    """Optimizer::LocalBundleAdjustment(KeyFrame*, bool*, Map*) ITSELF (src/Optimizer.cc compiled unmodified into libmatch_ref.so) on a key-frame / landmark graph
    built from a planarslam_b200.synth_lba problem.  Keys of oracle_lib.local_bundle_adjustment (positions as the reference wrote them back: float) plus
    pt_bad / line_bad / plane_bad (landmarks the erasures turned bad: all their slots are cleared, not only the erased observation's)."""
    from planarslam_b200 import lba as _lba
    lib, pre = _impl(impl)
    fn = getattr(lib, pre + "full_local_bundle_adjustment")          # impl="adp": pslam_adapter::ref::Optimizer::LocalBundleAdjustment on the same object graph
    fn.argtypes = [C.c_void_p] * 5
    s = _lba.problem_struct(p)
    r, o = _lba.result_struct(s)
    bad = [np.zeros(max(n, 1), np.uint8) for n in (s.n_points, s.n_lines, s.n_planes)]
    rc = fn(C.byref(s), C.byref(r), *[b.ctypes.data for b in bad])
    assert rc == 0, rc
    out = _lba.finish(r, o)
    out["pt_bad"], out["line_bad"], out["plane_bad"] = bad[0][:s.n_points], bad[1][:s.n_lines], bad[2][:s.n_planes]
    return out


@_recorded(match_lib, digest=True)
def ref_full_compute_stereo_from_rgbd(keys_xy, keys_un_xy, depth, bf: float):
    """Frame::ComputeStereoFromRGBD itself (compiled src/Frame.cc).  Same arguments / returns as oracle_lib.compute_stereo_from_rgbd."""
    L = match_lib()
    L.ref_full_compute_stereo_from_rgbd.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_void_p]
    L.ref_full_compute_stereo_from_rgbd.restype = None
    k, ku, d = np.ascontiguousarray(keys_xy, np.float32), np.ascontiguousarray(keys_un_xy, np.float32), np.ascontiguousarray(depth, np.float32)
    ur, dz = np.zeros(len(k), np.float32), np.zeros(len(k), np.float32)
    L.ref_full_compute_stereo_from_rgbd(len(k), k.ctypes.data, ku.ctypes.data, d.ctypes.data, d.shape[1], d.shape[0], bf, ur.ctypes.data, dz.ctypes.data)
    return ur, dz


@_recorded(match_lib, digest=True)
def ref_full_lines3d_frame(keylines, depth, cam, seed=1, skip=0):
    """Frame::isLineGood itself (compiled src/Frame.cc + src/LineExtractor.cpp, libc rand() after srand(seed) and `skip` draws): (mvDepthLine, mvLines3D)."""
    from oracle_lib import KEYLINE_DTYPE
    L = match_lib()
    L.ref_full_lines3d_frame.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_uint32, C.c_int, C.c_void_p, C.c_void_p]
    L.ref_full_lines3d_frame.restype = None
    kl, d, camv = np.ascontiguousarray(keylines, KEYLINE_DTYPE), np.ascontiguousarray(depth, np.float32), np.asarray(cam, np.float32)
    dl, l3 = np.zeros(len(kl), np.float32), np.zeros((len(kl), 6))
    L.ref_full_lines3d_frame(kl.ctypes.data, len(kl), d.ctypes.data, d.shape[1], d.shape[0], camv.ctypes.data, seed, skip, dl.ctypes.data, l3.ctypes.data)
    return dl, l3


_track = None


def track_lib():
    """oracle/_ref/libtrack_ref.so: src/Tracking.cc compiled unmodified (links against libmatch_ref.so); oracle/ref/track_driver.cc calls TrackManhattanFrame."""
    global _track
    if _track is None and match_lib() is not None:
        _track = _load("libtrack_ref.so")
    return _track


@_recorded(track_lib)
def ref_track_manhattan_frame(R_last, normals, dirs):
    """Tracking::TrackManhattanFrame itself.  Returns the 3x3 float32 rotation it returns."""
    L = track_lib()
    L.ref_track_manhattan_frame.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]
    R = np.ascontiguousarray(R_last, np.float32).reshape(3, 3)
    nr, dr = np.ascontiguousarray(normals, np.float32).reshape(-1, 3), np.ascontiguousarray(dirs, np.float64).reshape(-1, 3)
    out = np.zeros((3, 3), np.float32)
    rc = L.ref_track_manhattan_frame(R.ctypes.data, nr.ctypes.data, len(nr), dr.ctypes.data, len(dr), out.ctypes.data)
    assert rc == 33, rc
    return out


@_recorded(match_lib, digest=True)
def ref_detect_loop_candidates(db: dict, min_score: float, sentinel: float = -1.0, impl: str = "ref"):
    """KeyFrameDatabase::DetectLoopCandidates by the reference's own code (src/KeyFrameDatabase.cc + DBoW2 L1 scoring).  Same layout as oracle_lib.detect_loop_candidates."""
    lib, pre = _impl(impl)
    fn = getattr(lib, pre + "detect_loop_candidates")
    fn.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int] + [C.c_void_p] * 4 + [C.c_int, C.c_void_p, C.c_float] + [C.c_void_p] * 3
    import oracle_lib
    d, n_kf, covis, stride = oracle_lib._db_args(db)
    cand, words, score = np.zeros(max(n_kf, 1), np.int32), np.zeros(max(n_kf, 1), np.int32), np.full(max(n_kf, 1), sentinel, np.float32)
    n = fn(d["q_word"].ctypes.data, d["q_val"].ctypes.data, len(d["q_word"]), n_kf, d["off"].ctypes.data, d["word"].ctypes.data,
                                     d["val"].ctypes.data, covis, stride, d["connected"].ctypes.data if "connected" in d else None, min_score,
                                     cand.ctypes.data, words.ctypes.data, score.ctypes.data)
    return cand[:n].copy(), words[:n_kf], score[:n_kf]


@_recorded(match_lib, digest=True)
def ref_detect_relocalization_candidates(db: dict, reloc_score: np.ndarray, impl: str = "ref"):
    lib, pre = _impl(impl)
    fn = getattr(lib, pre + "detect_relocalization_candidates")
    fn.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int] + [C.c_void_p] * 4 + [C.c_int] + [C.c_void_p] * 3
    import oracle_lib
    d, n_kf, covis, stride = oracle_lib._db_args(db)
    cand, words, score = np.zeros(max(n_kf, 1), np.int32), np.zeros(max(n_kf, 1), np.int32), np.ascontiguousarray(reloc_score, np.float32).copy()
    n = fn(d["q_word"].ctypes.data, d["q_val"].ctypes.data, len(d["q_word"]), n_kf, d["off"].ctypes.data, d["word"].ctypes.data,
                                               d["val"].ctypes.data, covis, stride, score.ctypes.data, cand.ctypes.data, words.ctypes.data)
    return cand[:n].copy(), words[:n_kf], score


@_recorded(match_lib, digest=True)
def ref_search_by_bow_kf(kf1: dict, kf2: dict, nnratio: float = 0.75, check_orientation: bool = True, impl: str = "ref"):
    """ORBmatcher::SearchByBoW(KeyFrame*, KeyFrame*, vector<MapPoint*>&) by the reference's own code (impl="adp": the product's adapter)."""
    import oracle_lib
    lib, pre = _impl(impl)
    return oracle_lib._bow_kf_call(getattr(lib, pre + "search_by_bow_kf"), kf1, kf2, nnratio, check_orientation)


@_recorded(match_lib)
def ref_line_search_by_descriptor(kf_desc, kf_has_ml, f_desc, impl: str = "ref"):
    """LSDmatcher::SearchByDescriptor(KeyFrame*, Frame&, vector<MapLine*>&) by the reference's own code (impl="adp": the product's adapter).  Returns (nmatches,
    match [n_f]: key line of the key frame whose map line the call stores into vpMapLineMatches[j], -1 NULL)."""
    lib, pre = _impl(impl)
    fn = getattr(lib, pre + "line_search_by_descriptor")
    fn.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    q, h, t = np.ascontiguousarray(kf_desc, np.uint8), np.ascontiguousarray(kf_has_ml, np.uint8), np.ascontiguousarray(f_desc, np.uint8)
    match = np.full(max(len(t), 1), -1, np.int32)
    n = fn(len(q), q.ctypes.data, h.ctypes.data, len(t), t.ctypes.data, match.ctypes.data)
    return n, match[:len(t)]
