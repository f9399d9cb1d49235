"""ctypes front-end of oracle/liborb_oracle.so (built by oracle/Makefile).  TEST INFRASTRUCTURE ONLY."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "liborb_oracle.so")

KP_DTYPE = np.dtype([("x", "<f4"), ("y", "<f4"), ("size", "<f4"), ("angle", "<f4"), ("response", "<f4"),
                     ("octave", "<i4"), ("class_id", "<i4")])
assert KP_DTYPE.itemsize == 28


def build(force: bool = False) -> str:
    srcs = [os.path.join(_HERE, f) for f in ("orb_ref.cpp", "match_ref.cpp", "occ_ref.cpp", "pipeline_ref.cpp",
                                             "Makefile")]
    if force or not os.path.exists(_SO) or any(os.path.getmtime(s) > os.path.getmtime(_SO) for s in srcs):
        subprocess.check_call(["make", "-C", _HERE, "-s"] + (["-B"] if force else []))
    return _SO


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            build()
        L = C.CDLL(_SO)
        L.orb_ref_create.restype = C.c_void_p
        L.orb_ref_create.argtypes = [C.c_int, C.c_float, C.c_int, C.c_int, C.c_int]
        L.orb_ref_destroy.argtypes = [C.c_void_p]
        L.orb_ref_extract.restype = C.c_int
        L.orb_ref_extract.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                      C.c_int, C.c_void_p]
        L.orb_ref_tables.argtypes = [C.c_void_p] + [C.c_void_p] * 6
        L.orb_ref_level_dims.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        L.orb_ref_get_level.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        L.orb_ref_resize.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int]
        L.orb_ref_blur.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        L.orb_ref_fast.restype = C.c_int
        L.orb_ref_fast.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int]
        L.orb_ref_fast_atan2.restype = C.c_float
        L.orb_ref_fast_atan2.argtypes = [C.c_float, C.c_float]
        L.orb_ref_descriptor.argtypes = [C.c_void_p, C.c_int, C.c_float, C.c_float, C.c_float, C.c_void_p]
        L.orb_ref_distribute.restype = C.c_int
        L.orb_ref_distribute.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                         C.c_void_p, C.c_int]
        _lib = L
    return _lib


def _p(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


class RefExtractor:
    """C++ oracle of ORB_SLAM2::ORBextractor (oracle/orb_ref.cpp)."""

    def __init__(self, nfeatures=1000, scaleFactor=1.2, nlevels=8, iniThFAST=20, minThFAST=7):
        self.L = lib()
        self.nlevels = nlevels
        self.nfeatures = nfeatures
        self.h = C.c_void_p(self.L.orb_ref_create(nfeatures, scaleFactor, nlevels, iniThFAST, minThFAST))
        sf, inv, s2, is2 = (np.zeros(nlevels, np.float32) for _ in range(4))
        nf = np.zeros(nlevels, np.int32)
        um = np.zeros(16, np.int32)
        self.L.orb_ref_tables(self.h, _p(sf), _p(inv), _p(s2), _p(is2), _p(nf), _p(um))
        self.mvScaleFactor, self.mvInvScaleFactor, self.mvLevelSigma2, self.mvInvLevelSigma2 = sf, inv, s2, is2
        self.mnFeaturesPerLevel, self.umax = nf, um
        self.candidates_per_level = np.zeros(nlevels, np.int32)

    def __del__(self):
        try:
            self.L.orb_ref_destroy(self.h)
        except Exception:
            pass

    def __call__(self, image: np.ndarray):
        if image is None or image.size == 0:
            return np.zeros(0, KP_DTYPE), np.zeros((0, 32), np.uint8)
        assert image.dtype == np.uint8 and image.ndim == 2
        cap = self.nfeatures + 3 * self.nlevels + 64
        kps = np.zeros(cap, KP_DTYPE)
        desc = np.zeros((cap, 32), np.uint8)
        n = self.L.orb_ref_extract(self.h, _p(image), image.shape[0], image.shape[1], image.strides[0], _p(kps),
                                   _p(desc), cap, _p(self.candidates_per_level))
        if n < 0:
            raise RuntimeError("orb_ref_extract failed: %d" % n)
        return kps[:n].copy(), desc[:n].copy()

    def level(self, l: int, bordered: bool = False) -> np.ndarray:
        w, h = C.c_int(), C.c_int()
        self.L.orb_ref_level_dims(self.h, l, C.byref(w), C.byref(h))
        shp = (h.value + 38, w.value + 38) if bordered else (h.value, w.value)
        out = np.zeros(shp, np.uint8)
        self.L.orb_ref_get_level(self.h, l, int(bordered), _p(out))
        return out


def resize(src: np.ndarray, dw: int, dh: int) -> np.ndarray:
    src = np.ascontiguousarray(src)
    dst = np.zeros((dh, dw), np.uint8)
    lib().orb_ref_resize(_p(src), src.shape[1], src.shape[0], _p(dst), dw, dh)
    return dst


def blur(src: np.ndarray) -> np.ndarray:
    src = np.ascontiguousarray(src)
    dst = np.zeros_like(src)
    lib().orb_ref_blur(_p(src), src.shape[1], src.shape[0], _p(dst))
    return dst


def fast(roi: np.ndarray, t: int) -> np.ndarray:
    roi = np.ascontiguousarray(roi)
    cap = roi.size
    out = np.zeros((cap, 3), np.int32)
    n = lib().orb_ref_fast(_p(roi), roi.shape[1], roi.shape[0], roi.strides[0], t, _p(out), cap)
    return out[:n]


def fast_atan2(y: float, x: float) -> float:
    return float(lib().orb_ref_fast_atan2(y, x))


def descriptor(img: np.ndarray, x: float, y: float, angle: float) -> np.ndarray:
    img = np.ascontiguousarray(img)
    d = np.zeros(32, np.uint8)
    lib().orb_ref_descriptor(_p(img), img.strides[0], x, y, angle, _p(d))
    return d


def distribute(kps: np.ndarray, minX, maxX, minY, maxY, N) -> np.ndarray:
    kps = np.ascontiguousarray(kps)
    out = np.zeros(max(len(kps), 1), KP_DTYPE)
    n = lib().orb_ref_distribute(_p(kps), len(kps), minX, maxX, minY, maxY, N, _p(out), len(out))
    if n < 0:
        raise RuntimeError("distribute failed %d" % n)
    return out[:n]


# ------------------------------------------------------------------------------------------------
# matcher / frame-glue oracle (oracle/match_ref.cpp); struct mirrors come from the ABI header mirror
# ------------------------------------------------------------------------------------------------
def _mlib():
    L = lib()
    if not getattr(L, "_match_ready", False):
        from orb_slam2_ssd_semantic_b200 import _abi
        L.match_ref_hamming.argtypes = [C.c_void_p, C.c_void_p]
        L.match_ref_projection_last.argtypes = [C.POINTER(_abi.OrbmFrame), C.POINTER(_abi.OrbmLast), C.c_float, C.c_int,
                                                C.c_float, C.c_int, C.c_void_p, C.POINTER(C.c_int)]
        L.match_ref_projection_points.argtypes = [C.POINTER(_abi.OrbmFrame), C.POINTER(_abi.OrbmTrackPoints),
                                                  C.c_float, C.c_float, C.c_void_p, C.POINTER(C.c_int)]
        L.match_ref_bow.argtypes = [C.POINTER(_abi.OrbmBow), C.POINTER(_abi.OrbmBow), C.c_float, C.c_int, C.c_void_p,
                                    C.POINTER(C.c_int)]
        L.frame_ref_stereo_unproject.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                                 C.c_void_p] + [C.c_float] * 5 + [C.c_void_p] * 4
        L.frame_ref_stereo_unproject.restype = None
        L._match_ready = True
    return L


def hamming(a, b) -> int:
    a = np.ascontiguousarray(a, np.uint8)
    b = np.ascontiguousarray(b, np.uint8)
    return int(_mlib().match_ref_hamming(_p(a), _p(b)))


def search_by_projection_last(cur, last, th, mono=False, nnratio=0.9, check_ori=True):
    """cur: _abi.FrameView, last: _abi.LastView -> (nmatches, cur2last)."""
    out = np.full(cur.n, -1, np.int32)
    nm = C.c_int(0)
    cs, ls = cur.struct(), last.struct()
    _mlib().match_ref_projection_last(C.byref(cs), C.byref(ls), float(th), int(mono), float(nnratio), int(check_ori),
                                      _p(out), C.byref(nm))
    return nm.value, out


def search_by_projection_points(F, pts, th, nnratio=0.8):
    out = np.full(F.n, -1, np.int32)
    nm = C.c_int(0)
    fs, ps = F.struct(), pts.struct()
    _mlib().match_ref_projection_points(C.byref(fs), C.byref(ps), float(th), float(nnratio), _p(out), C.byref(nm))
    return nm.value, out


def search_projected(F, queries, max_dist, claim_rule=1, check_ori=True):
    from orb_slam2_ssd_semantic_b200 import _abi
    L = _mlib()
    L.match_ref_projected.argtypes = [C.POINTER(_abi.OrbmFrame), C.POINTER(_abi.OrbmQueries), C.c_int, C.c_int, C.c_int,
                                      C.c_void_p, C.POINTER(C.c_int)]
    out = np.full(F.n, -1, np.int32)
    nm = C.c_int(0)
    fs, qs = F.struct(), queries.struct()
    L.match_ref_projected(C.byref(fs), C.byref(qs), int(max_dist), int(claim_rule), int(check_ori), _p(out), C.byref(nm))
    return nm.value, out


def search_by_bow(kf, f, nnratio=0.7, check_ori=True):
    out = np.full(f.n, -1, np.int32)
    nm = C.c_int(0)
    ks, fs = kf.struct(), f.struct()
    _mlib().match_ref_bow(C.byref(ks), C.byref(fs), float(nnratio), int(check_ori), _p(out), C.byref(nm))
    return nm.value, out


def search_by_bow_kf(kf1, kf2, nnratio=0.75, check_ori=True):
    from orb_slam2_ssd_semantic_b200 import _abi
    L = _mlib()
    L.match_ref_bow_kf.argtypes = [C.POINTER(_abi.OrbmBow), C.POINTER(_abi.OrbmBow), C.c_float, C.c_int, C.c_void_p,
                                   C.POINTER(C.c_int)]
    out = np.full(kf1.n, -1, np.int32)
    nm = C.c_int(0)
    a, b = kf1.struct(), kf2.struct()
    L.match_ref_bow_kf(C.byref(a), C.byref(b), float(nnratio), int(check_ori), _p(out), C.byref(nm))
    return nm.value, out


def stereo_unproject(kps, depth, Tcw, fx, fy, cx, cy, bf):
    """ComputeStereoFromRGBD + UnprojectStereo for every keypoint -> uright, depth, xw, valid."""
    n = len(kps)
    kf = np.ascontiguousarray(kps).view(np.float32).reshape(n, 7) if n else np.zeros((0, 7), np.float32)
    depth = np.ascontiguousarray(depth, np.float32)
    T = np.ascontiguousarray(Tcw, np.float32).reshape(16)
    ur = np.zeros(n, np.float32)
    dp = np.zeros(n, np.float32)
    xw = np.zeros((n, 3), np.float32)
    va = np.zeros(n, np.uint8)
    _mlib().frame_ref_stereo_unproject(_p(kf), 7, n, _p(depth), depth.shape[0], depth.shape[1], _p(T), fx, fy, cx, cy,
                                       bf, _p(ur), _p(dp), _p(xw), _p(va))
    return ur, dp, xw, va


def pipeline_run(gray, depth, Tcw, nthreads, nfeatures=1000, scale=1.2, nlevels=8, ini_th=20, min_th=7, fx=535.4,
                 fy=539.2, cx=320.1, cy=247.6, bf=40.0, th=15.0, nnratio=0.9, check_ori=True, last_obs=1, rgb=None,
                 kf_every=0):
    """Multi-threaded CPU baseline (oracle/pipeline_ref.cpp) -> (seconds, nkp, nmatch[, leaves]).  With rgb and
    kf_every > 0 every kf_every-th frame is also pushed through the occupancy oracle on its own mapping thread."""
    L = lib()
    L.pipeline_ref_run.restype = C.c_double
    L.pipeline_ref_run.argtypes = [C.c_void_p] * 3 + [C.c_int] * 3 + [C.c_int, C.c_float, C.c_int, C.c_int, C.c_int] + \
        [C.c_float] * 7 + [C.c_int] * 3 + [C.c_void_p] * 2 + [C.c_void_p, C.c_int, C.c_void_p]
    gray = np.ascontiguousarray(gray, np.uint8)
    depth = np.ascontiguousarray(depth, np.float32)
    T = np.ascontiguousarray(Tcw, np.float32).reshape(-1, 16)
    n, rows, cols = gray.shape
    nkp = np.zeros(n, np.int32)
    nm = np.zeros(n, np.int32)
    leaves = C.c_longlong(0)
    rgbp = None if rgb is None else np.ascontiguousarray(rgb, np.uint8)
    sec = L.pipeline_ref_run(_p(gray), _p(depth), _p(T), n, rows, cols, nfeatures, scale, nlevels, ini_th, min_th, fx, fy,
                             cx, cy, bf, th, nnratio, int(check_ori), last_obs, nthreads, _p(nkp), _p(nm),
                             None if rgbp is None else _p(rgbp), int(kf_every), C.byref(leaves))
    return sec, nkp, nm


# ------------------------------------------------------------------------------------------------
# occupancy oracle (oracle/occ_ref.cpp)
# ------------------------------------------------------------------------------------------------
class RefOccupancy:
    def __init__(self, **kw):
        from orb_slam2_ssd_semantic_b200._abi import OcmParams
        L = lib()
        L.occ_ref_create.restype = C.c_void_p
        L.occ_ref_create.argtypes = [C.POINTER(OcmParams)]
        L.occ_ref_destroy.argtypes = [C.c_void_p]
        L.occ_ref_default_params.argtypes = [C.POINTER(OcmParams)]
        L.occ_ref_constants.argtypes = [C.c_void_p, C.c_void_p]
        L.occ_ref_insert_keyframe.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p] + \
            [C.c_float] * 4 + [C.c_void_p]
        L.occ_ref_last_points.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.occ_ref_num_leaves.restype = C.c_longlong
        L.occ_ref_num_leaves.argtypes = [C.c_void_p]
        L.occ_ref_export_leaves.restype = C.c_longlong
        L.occ_ref_export_leaves.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong]
        L.occ_ref_ray.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        self.L = L
        p = OcmParams()
        L.occ_ref_default_params(C.byref(p))
        for k, v in kw.items():
            setattr(p, k, v)
        self.params = p
        self.h = C.c_void_p(L.occ_ref_create(C.byref(p)))

    def __del__(self):
        try:
            self.L.occ_ref_destroy(self.h)
        except Exception:
            pass

    def constants(self):
        out = np.zeros(4, np.float32)
        self.L.occ_ref_constants(self.h, _p(out))
        return out   # hit, miss, clamp_min, clamp_max (log-odds)

    def insert_keyframe(self, Tcw, depth, rgb, fx, fy, cx, cy, ground_label=None):
        depth = np.ascontiguousarray(depth, np.float32)
        rgb = np.ascontiguousarray(rgb, np.uint8)
        T = np.ascontiguousarray(Tcw, np.float32).reshape(16)
        lab = None if ground_label is None else np.ascontiguousarray(ground_label, np.uint8)
        return self.L.occ_ref_insert_keyframe(self.h, _p(depth), _p(rgb), depth.shape[0], depth.shape[1], _p(T), fx, fy,
                                              cx, cy, None if lab is None else _p(lab))

    def insert_keyframes_mt(self, depth, rgb, label, idx, Tcw, fx, fy, cx, cy, nthreads):
        """Batch form for the CPU baseline: GeneratePointCloud of the keyframes on `nthreads` threads, InsertScan in
        order.  depth [F,rows,cols] f32, rgb [F,rows,cols,3], label [F,rows,cols] u8 or None, idx = frames to insert,
        Tcw [len(idx),4,4]."""
        depth = np.ascontiguousarray(depth, np.float32)
        rgb = np.ascontiguousarray(rgb, np.uint8)
        lab = None if label is None else np.ascontiguousarray(label, np.uint8)
        idx = np.ascontiguousarray(idx, np.int32)
        T = np.ascontiguousarray(Tcw, np.float32).reshape(len(idx), 16)
        self.L.occ_ref_insert_keyframes_mt.argtypes = [C.c_void_p] * 4 + [C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p] + \
            [C.c_float] * 4 + [C.c_int]
        self.L.occ_ref_insert_keyframes_mt(self.h, _p(depth), _p(rgb), None if lab is None else _p(lab), depth.shape[1],
                                           depth.shape[2], _p(idx), len(idx), _p(T), fx, fy, cx, cy, int(nthreads))

    def last_points(self):
        cap = 1 << 20
        xyz = np.zeros((cap, 3), np.float32)
        rgb = np.zeros((cap, 3), np.uint8)
        lab = np.zeros(cap, np.uint8)
        n = self.L.occ_ref_last_points(self.h, _p(xyz), _p(rgb), _p(lab), cap)
        return xyz[:n].copy(), rgb[:n].copy(), lab[:n].copy()

    def export_leaves(self):
        n = self.L.occ_ref_num_leaves(self.h)
        keys = np.zeros((max(n, 1), 3), np.uint16)
        lo = np.zeros(max(n, 1), np.float32)
        m = self.L.occ_ref_export_leaves(self.h, _p(keys), _p(lo), n)
        return keys[:m], lo[:m]

    def ray(self, origin, end):
        o = np.ascontiguousarray(origin, np.float32)
        e = np.ascontiguousarray(end, np.float32)
        keys = np.zeros((4096, 3), np.uint16)
        n = self.L.occ_ref_ray(self.h, _p(o), _p(e), _p(keys), 4096)
        return None if n < 0 else keys[:n].copy()


def backproject_all(depth, Tcw, fx, fy, cx, cy):
    """T variant (src/pointcloudmapping.cc:131-194): every pixel, no gate -> rows*cols x 3 world points."""
    L = lib()
    L.occ_ref_backproject_all.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p] + [C.c_float] * 4 + [C.c_void_p]
    depth = np.ascontiguousarray(depth, np.float32)
    T = np.ascontiguousarray(Tcw, np.float32).reshape(16)
    out = np.zeros((depth.size, 3), np.float32)
    L.occ_ref_backproject_all(_p(depth), depth.shape[0], depth.shape[1], _p(T), fx, fy, cx, cy, _p(out))
    return out


def global_refilter(xyz, rgb, leaf):
    """T-variant global map refilter (src/pointcloudmapping.cc:491-493, PCL VoxelGrid) -> (xyz', rgb') in cell order."""
    L = lib()
    L.occ_ref_global_refilter.restype = C.c_longlong
    L.occ_ref_global_refilter.argtypes = [C.c_void_p, C.c_void_p, C.c_longlong, C.c_float, C.c_void_p, C.c_void_p,
                                          C.c_longlong]
    xyz = np.ascontiguousarray(xyz, np.float32).reshape(-1, 3)
    rgb = np.ascontiguousarray(rgb, np.uint8).reshape(-1, 3)
    n = xyz.shape[0]
    out = np.zeros((max(n, 1), 3), np.float32)
    out_rgb = np.zeros((max(n, 1), 3), np.uint8)
    m = L.occ_ref_global_refilter(_p(xyz), _p(rgb), n, float(np.float32(leaf)), _p(out), _p(out_rgb), max(n, 1))
    if m < 0:
        raise ValueError("global_refilter: %s" % ("index space overflows int" if m == -1 else "cap"))
    return out[:m].copy(), out_rgb[:m].copy()


def search_for_initialization(F1, F2, prev_xy, window=100, nnratio=0.9, check_ori=True):
    """SearchForInitialization (src/ORBmatcher.cc:523-660) -> (nmatches, matches12, updated vbPrevMatched)."""
    from orb_slam2_ssd_semantic_b200 import _abi
    L = _mlib()
    L.match_ref_initialization.argtypes = [C.POINTER(_abi.OrbmFrame), C.POINTER(_abi.OrbmFrame), C.c_void_p, C.c_int,
                                           C.c_float, C.c_int, C.c_void_p, C.POINTER(C.c_int)]
    prev = np.ascontiguousarray(prev_xy, np.float32).reshape(-1, 2).copy()
    out = np.full(F1.n, -1, np.int32)
    nm = C.c_int(0)
    a, b = F1.struct(), F2.struct()
    L.match_ref_initialization(C.byref(a), C.byref(b), _p(prev), int(window), float(nnratio), int(check_ori), _p(out),
                               C.byref(nm))
    return nm.value, out, prev


# ------------------------------------------------------------------------------------------------
# oracle/_ref/librefsrc.so: the REFERENCE'S OWN sources (src/ORBextractor.cc, ORBmatcher.cc, Frame.cc, KeyFrame.cc,
# MapPoint.cc, Map.cc) compiled unmodified against oracle/standin/ (see oracle/Makefile, target `ref`).  Same call
# signatures as the restatement above, so tests can assert restatement == reference sources.
_REFSO = os.path.join(_HERE, "_ref", "librefsrc.so")
_reflib = None


def refsrc_available() -> bool:
    return os.path.exists(_REFSO)


def reflib() -> C.CDLL:
    global _reflib
    if _reflib is None:
        if not os.path.exists(_REFSO):
            subprocess.check_call(["make", "-C", _HERE, "-s", "ref"])
        from orb_slam2_ssd_semantic_b200 import _abi
        L = C.CDLL(_REFSO)
        L.refsrc_orb_create.restype = C.c_void_p
        L.refsrc_orb_create.argtypes = [C.c_int, C.c_float, C.c_int, C.c_int, C.c_int]
        L.refsrc_orb_destroy.argtypes = [C.c_void_p]
        L.refsrc_orb_extract.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                         C.c_int, C.c_void_p]
        L.refsrc_orb_tables.argtypes = [C.c_void_p] + [C.c_void_p] * 6
        L.refsrc_orb_level_dims.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        L.refsrc_orb_get_level.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        L.refsrc_orb_distribute.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                            C.c_void_p, C.c_int]
        L.refsrc_hamming.argtypes = [C.c_void_p, C.c_void_p]
        PF, PL, PT, PB = (C.POINTER(_abi.OrbmFrame), C.POINTER(_abi.OrbmLast), C.POINTER(_abi.OrbmTrackPoints),
                          C.POINTER(_abi.OrbmBow))
        L.refsrc_projection_last.argtypes = [PF, PL, C.c_float, C.c_int, C.c_float, C.c_int, C.c_void_p, C.POINTER(C.c_int)]
        L.refsrc_projection_points.argtypes = [PF, PT, C.c_float, C.c_float, C.c_void_p, C.POINTER(C.c_int)]
        L.refsrc_bow.argtypes = [PB, PB, C.c_float, C.c_int, C.c_void_p, C.POINTER(C.c_int)]
        L.refsrc_bow_kf.argtypes = [PB, PB, C.c_float, C.c_int, C.c_void_p, C.POINTER(C.c_int)]
        L.refsrc_initialization.argtypes = [PF, PF, C.c_void_p, C.c_int, C.c_float, C.c_int, C.c_void_p, C.POINTER(C.c_int)]
        L.refsrc_frame_rgbd.argtypes = ([C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int,
                                         C.c_int, C.c_void_p] + [C.c_float] * 5 + [C.c_void_p] * 7 + [C.c_int, C.c_void_p])
        L.refsrc_is_in_frustum.argtypes = [PF, C.c_int] + [C.c_void_p] * 4 + [C.c_float] + [C.c_void_p] * 6
        _reflib = L
    return _reflib


class SrcExtractor:
    """ORB_SLAM2::ORBextractor of the reference (src/ORBextractor.cc compiled unmodified)."""

    def __init__(self, nfeatures=1000, scaleFactor=1.2, nlevels=8, iniThFAST=20, minThFAST=7):
        self.L = reflib()
        self.nlevels = nlevels
        self.h = self.L.refsrc_orb_create(nfeatures, scaleFactor, nlevels, iniThFAST, minThFAST)
        self.cap = nfeatures + 16 * nlevels + 64
        t = [np.zeros(nlevels, np.float32) for _ in range(4)] + [np.zeros(nlevels, np.int32), np.zeros(16, np.int32)]
        self.L.refsrc_orb_tables(self.h, *[_p(a) for a in t])
        (self.mvScaleFactor, self.mvInvScaleFactor, self.mvLevelSigma2, self.mvInvLevelSigma2,
         self.mnFeaturesPerLevel, self.umax) = t

    def __del__(self):
        if getattr(self, "h", None):
            self.L.refsrc_orb_destroy(self.h)
            self.h = None

    def __call__(self, image: np.ndarray):
        image = np.asarray(image)
        assert image.dtype == np.uint8 and image.ndim == 2
        if image.strides[1] != 1:
            image = np.ascontiguousarray(image)
        kps = np.zeros(self.cap, KP_DTYPE)
        desc = np.zeros((self.cap, 32), np.uint8)
        n = C.c_int(0)
        rc = self.L.refsrc_orb_extract(self.h, image.ctypes.data, image.shape[0], image.shape[1], image.strides[0],
                                       _p(kps), _p(desc), self.cap, C.byref(n))
        assert rc == 0
        return kps[:n.value].copy(), desc[:n.value].copy()

    def level(self, l: int, bordered: bool = False) -> np.ndarray:
        w, h = C.c_int(0), C.c_int(0)
        assert self.L.refsrc_orb_level_dims(self.h, l, C.byref(w), C.byref(h)) == 0
        B = 19 if bordered else 0
        out = np.zeros((h.value + 2 * B, w.value + 2 * B), np.uint8)
        self.L.refsrc_orb_get_level(self.h, l, int(bordered), _p(out))
        return out


def src_distribute(kps, minX, maxX, minY, maxY, N):
    kps = np.ascontiguousarray(kps, KP_DTYPE)
    out = np.zeros(len(kps) + 8, KP_DTYPE)
    n = reflib().refsrc_orb_distribute(_p(kps), len(kps), minX, maxX, minY, maxY, N, _p(out), len(out))
    assert n >= 0
    return out[:n].copy()


def src_hamming(a, b) -> int:
    a = np.ascontiguousarray(a, np.uint8)
    b = np.ascontiguousarray(b, np.uint8)
    return int(reflib().refsrc_hamming(_p(a), _p(b)))


def src_search_by_projection_last(cur, last, th, mono=False, nnratio=0.9, check_ori=True):
    out = np.full(cur.n, -1, np.int32)
    nm = C.c_int(0)
    cs, ls = cur.struct(), last.struct()
    reflib().refsrc_projection_last(C.byref(cs), C.byref(ls), float(th), int(mono), float(nnratio), int(check_ori),
                                    _p(out), C.byref(nm))
    return nm.value, out


def src_search_by_projection_points(F, pts, th, nnratio=0.8):
    out = np.full(F.n, -1, np.int32)
    nm = C.c_int(0)
    fs, ps = F.struct(), pts.struct()
    reflib().refsrc_projection_points(C.byref(fs), C.byref(ps), float(th), float(nnratio), _p(out), C.byref(nm))
    return nm.value, out


def src_search_by_bow(kf, f, nnratio=0.7, check_ori=True):
    out = np.full(f.n, -1, np.int32)
    nm = C.c_int(0)
    ks, fs = kf.struct(), f.struct()
    reflib().refsrc_bow(C.byref(ks), C.byref(fs), float(nnratio), int(check_ori), _p(out), C.byref(nm))
    return nm.value, out


def src_search_by_bow_kf(kf1, kf2, nnratio=0.75, check_ori=True):
    out = np.full(kf1.n, -1, np.int32)
    nm = C.c_int(0)
    a, b = kf1.struct(), kf2.struct()
    reflib().refsrc_bow_kf(C.byref(a), C.byref(b), float(nnratio), int(check_ori), _p(out), C.byref(nm))
    return nm.value, out


def src_search_for_initialization(F1, F2, prev_xy, window=100, nnratio=0.9, check_ori=True):
    prev = np.ascontiguousarray(prev_xy, np.float32).reshape(-1, 2).copy()
    out = np.full(F1.n, -1, np.int32)
    nm = C.c_int(0)
    a, b = F1.struct(), F2.struct()
    reflib().refsrc_initialization(C.byref(a), C.byref(b), _p(prev), int(window), float(nnratio), int(check_ori),
                                   _p(out), C.byref(nm))
    return nm.value, out, prev


def src_frame_rgbd(gray, depth, Tcw, fx, fy, cx, cy, bf, nfeatures=1000, scale=1.2, nlevels=8, ini_th=20, min_th=7,
                   dist=None):
    """The reference's RGB-D Frame constructor (src/Frame.cc:176-240) + UnprojectStereo per keypoint."""
    gray = np.ascontiguousarray(gray, np.uint8)
    depth = np.ascontiguousarray(depth, np.float32)
    T = np.ascontiguousarray(Tcw, np.float32).reshape(16)
    cap = nfeatures + 16 * nlevels + 64
    kps = np.zeros(cap, KP_DTYPE)
    desc = np.zeros((cap, 32), np.uint8)
    ur, dp, xw, va = np.zeros(cap, np.float32), np.zeros(cap, np.float32), np.zeros((cap, 3), np.float32), np.zeros(cap, np.uint8)
    n = C.c_int(0)
    d4 = None if dist is None else np.ascontiguousarray(dist, np.float32)
    rc = reflib().refsrc_frame_rgbd(_p(gray), _p(depth), gray.shape[0], gray.shape[1], nfeatures, scale, nlevels, ini_th,
                                    min_th, _p(T), fx, fy, cx, cy, bf, None if d4 is None else _p(d4), _p(kps), _p(desc),
                                    _p(ur), _p(dp), _p(xw), _p(va), cap, C.byref(n))
    assert rc == 0
    m = n.value
    return kps[:m].copy(), desc[:m].copy(), ur[:m].copy(), dp[:m].copy(), xw[:m].copy(), va[:m].copy()


def src_pipeline_run(gray, depth, Tcw, nthreads, nfeatures=1000, scale=1.2, nlevels=8, ini_th=20, min_th=7, fx=535.4,
                     fy=539.2, cx=320.1, cy=247.6, bf=40.0, th=15.0, nnratio=0.9, check_ori=True):
    """CPU baseline through the reference's OWN tracking sources (oracle/_ref/librefsrc.so): RGB-D Frame constructor +
    SearchByProjection(cur, last) per frame, frame-parallel -> (seconds, nkp, nmatch)."""
    L = reflib()
    L.refsrc_pipeline_run.restype = C.c_double
    L.refsrc_pipeline_run.argtypes = [C.c_void_p] * 3 + [C.c_int] * 3 + [C.c_int, C.c_float, C.c_int, C.c_int, C.c_int] + \
        [C.c_float] * 7 + [C.c_int] * 2 + [C.c_void_p] * 2
    gray = np.ascontiguousarray(gray, np.uint8)
    depth = np.ascontiguousarray(depth, np.float32)
    T = np.ascontiguousarray(Tcw, np.float32).reshape(-1, 16)
    n, rows, cols = gray.shape
    nkp = np.zeros(n, np.int32)
    nm = np.zeros(n, np.int32)
    sec = L.refsrc_pipeline_run(_p(gray), _p(depth), _p(T), n, rows, cols, nfeatures, scale, nlevels, ini_th, min_th, fx,
                                fy, cx, cy, bf, th, nnratio, int(check_ori), nthreads, _p(nkp), _p(nm))
    return sec, nkp, nm


# ------------------------------------------------------------------------------------------------
# flat oracles of the remaining matcher members + their reference-source / shim counterparts
class RefMapPoints(C.Structure):
    _fields_ = [("n", C.c_int), ("valid", C.c_void_p), ("bad", C.c_void_p), ("xw", C.c_void_p), ("normal", C.c_void_p),
                ("min_dist", C.c_void_p), ("max_dist", C.c_void_p), ("desc", C.c_void_p), ("obs", C.c_void_p)]


class MapPointsView:
    def __init__(self, xw, desc, valid=None, bad=None, normal=None, min_dist=None, max_dist=None, obs=None):
        f = lambda a, t: None if a is None else np.ascontiguousarray(a, t)
        self.xw = np.ascontiguousarray(xw, np.float32).reshape(-1, 3)
        self.n = len(self.xw)
        self.desc = np.ascontiguousarray(desc, np.uint8).reshape(-1, 32)
        self.valid, self.bad = f(valid, np.uint8), f(bad, np.uint8)
        self.normal = None if normal is None else np.ascontiguousarray(normal, np.float32).reshape(-1, 3)
        self.min_dist, self.max_dist, self.obs = f(min_dist, np.float32), f(max_dist, np.float32), f(obs, np.int32)

    def struct(self):
        s = RefMapPoints()
        s.n = self.n
        g = lambda a: None if a is None else a.ctypes.data
        s.valid, s.bad, s.xw, s.normal = g(self.valid), g(self.bad), g(self.xw), g(self.normal)
        s.min_dist, s.max_dist, s.desc, s.obs = g(self.min_dist), g(self.max_dist), g(self.desc), g(self.obs)
        return s


def search_best(KF, queries, gate=0, inv_level_sigma2=None):
    from orb_slam2_ssd_semantic_b200 import _abi
    L = _mlib()
    L.match_ref_best.argtypes = [C.POINTER(_abi.OrbmFrame), C.POINTER(_abi.OrbmQueries), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    bi = np.full(max(queries.n, 1), -1, np.int32)
    bd = np.full(max(queries.n, 1), 2 ** 31 - 1, np.int32)
    ks, qs = KF.struct(), queries.struct()
    is2 = None if inv_level_sigma2 is None else np.ascontiguousarray(inv_level_sigma2, np.float32)
    L.match_ref_best(C.byref(ks), C.byref(qs), int(gate), None if is2 is None else _p(is2), _p(bi), _p(bd))
    return bi[:queries.n], bd[:queries.n]


def search_for_triangulation(k1, k2, F12, epipole, sf2, sigma2_2, only_stereo=False, check_ori=True):
    from orb_slam2_ssd_semantic_b200 import _abi
    L = _mlib()
    L.match_ref_triangulation.argtypes = [C.POINTER(_abi.OrbmTriKF), C.POINTER(_abi.OrbmTriKF), C.c_void_p, C.c_float, C.c_float,
                                          C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_int)]
    F = np.ascontiguousarray(F12, np.float32).reshape(9)
    sf = np.ascontiguousarray(sf2, np.float32)
    s2 = np.ascontiguousarray(sigma2_2, np.float32)
    out = np.full(max(k1.n, 1), -1, np.int32)
    nm = C.c_int(0)
    a, b = k1.struct(), k2.struct()
    L.match_ref_triangulation(C.byref(a), C.byref(b), _p(F), float(epipole[0]), float(epipole[1]), _p(sf), _p(s2),
                              int(only_stereo), int(check_ori), _p(out), C.byref(nm))
    return nm.value, out[:k1.n]


_SHIMSO = os.path.join(_HERE, "_ref", "libshimsrc.so")
_shimlib = None


def shimlib() -> C.CDLL:
    """oracle/_ref/libshimsrc.so: the reference's Frame.cc / KeyFrame.cc / MapPoint.cc compiled against the B200 shims
    (needs a GPU at run time)."""
    global _shimlib
    if _shimlib is None:
        if not os.path.exists(_SHIMSO):
            subprocess.check_call(["make", "-C", _HERE, "-s", "shim"])
        _shimlib = C.CDLL(_SHIMSO)
    return _shimlib


class SrcMembers:
    """The remaining ORBmatcher members run on real Frame / KeyFrame / MapPoint graphs: prefix 'refsrc' = the reference's
    own ORBmatcher.cc, prefix 'shimsrc' = the B200 shim class on the same reference objects."""

    def __init__(self, prefix="refsrc"):
        self.L = reflib() if prefix == "refsrc" else shimlib()
        self.p = prefix

    def _f(self, name):
        return getattr(self.L, self.p + "_" + name)

    def search_by_projection_last(self, cur, last, th, mono=False, nnratio=0.9, check_ori=True):
        from orb_slam2_ssd_semantic_b200 import _abi
        f = self._f("projection_last")
        f.argtypes = [C.POINTER(_abi.OrbmFrame), C.POINTER(_abi.OrbmLast), C.c_float, C.c_int, C.c_float, C.c_int, C.c_void_p, C.POINTER(C.c_int)]
        out = np.full(cur.n, -1, np.int32)
        nm = C.c_int(0)
        cs, ls = cur.struct(), last.struct()
        f(C.byref(cs), C.byref(ls), float(th), int(mono), float(nnratio), int(check_ori), _p(out), C.byref(nm))
        return nm.value, out

    def search_by_projection_points(self, F, pts, th, nnratio=0.8):
        from orb_slam2_ssd_semantic_b200 import _abi
        f = self._f("projection_points")
        f.argtypes = [C.POINTER(_abi.OrbmFrame), C.POINTER(_abi.OrbmTrackPoints), C.c_float, C.c_float, C.c_void_p, C.POINTER(C.c_int)]
        out = np.full(F.n, -1, np.int32)
        nm = C.c_int(0)
        fs, ps = F.struct(), pts.struct()
        f(C.byref(fs), C.byref(ps), float(th), float(nnratio), _p(out), C.byref(nm))
        return nm.value, out

    def search_by_bow(self, kf, fr, nnratio=0.7, check_ori=True, kfkf=False):
        from orb_slam2_ssd_semantic_b200 import _abi
        f = self._f("bow_kf" if kfkf else "bow")
        f.argtypes = [C.POINTER(_abi.OrbmBow), C.POINTER(_abi.OrbmBow), C.c_float, C.c_int, C.c_void_p, C.POINTER(C.c_int)]
        out = np.full(kf.n if kfkf else fr.n, -1, np.int32)
        nm = C.c_int(0)
        a, b = kf.struct(), fr.struct()
        f(C.byref(a), C.byref(b), float(nnratio), int(check_ori), _p(out), C.byref(nm))
        return nm.value, out

    def search_for_initialization(self, F1, F2, prev_xy, window=100, nnratio=0.9, check_ori=True):
        from orb_slam2_ssd_semantic_b200 import _abi
        f = self._f("initialization")
        f.argtypes = [C.POINTER(_abi.OrbmFrame), C.POINTER(_abi.OrbmFrame), C.c_void_p, C.c_int, C.c_float, C.c_int, C.c_void_p, C.POINTER(C.c_int)]
        prev = np.ascontiguousarray(prev_xy, np.float32).reshape(-1, 2).copy()
        out = np.full(F1.n, -1, np.int32)
        nm = C.c_int(0)
        a, b = F1.struct(), F2.struct()
        f(C.byref(a), C.byref(b), _p(prev), int(window), float(nnratio), int(check_ori), _p(out), C.byref(nm))
        return nm.value, out, prev

    def projection_kf(self, cur, kf, kf_mps, already_found, th, orb_dist, nnratio=0.9, check_ori=True):
        from orb_slam2_ssd_semantic_b200 import _abi
        f = self._f("projection_kf")
        f.argtypes = [C.POINTER(_abi.OrbmFrame), C.POINTER(_abi.OrbmFrame), C.POINTER(RefMapPoints), C.c_void_p, C.c_float, C.c_int,
                      C.c_float, C.c_int, C.c_void_p, C.POINTER(C.c_int)]
        out = np.full(cur.n, -1, np.int32)
        nm = C.c_int(0)
        cs, ks, ms = cur.struct(), kf.struct(), kf_mps.struct()
        af = np.ascontiguousarray(already_found, np.uint8)
        f(C.byref(cs), C.byref(ks), C.byref(ms), _p(af), float(th), int(orb_dist), float(nnratio), int(check_ori), _p(out), C.byref(nm))
        return nm.value, out

    def projection_sim3(self, kf, Scw, pts, matched, th):
        from orb_slam2_ssd_semantic_b200 import _abi
        f = self._f("projection_sim3")
        f.argtypes = [C.POINTER(_abi.OrbmFrame), C.c_void_p, C.POINTER(RefMapPoints), C.c_void_p, C.c_int, C.POINTER(C.c_int)]
        m = np.ascontiguousarray(matched, np.int32).copy()
        S = np.ascontiguousarray(Scw, np.float32).reshape(16)
        nm = C.c_int(0)
        ks, ps = kf.struct(), pts.struct()
        f(C.byref(ks), _p(S), C.byref(ps), _p(m), int(th), C.byref(nm))
        return nm.value, m

    def fuse(self, kf, kf_mps, pts, in_kf, th, depth=None):
        from orb_slam2_ssd_semantic_b200 import _abi
        f = self._f("fuse")
        f.argtypes = [C.POINTER(_abi.OrbmFrame), C.POINTER(RefMapPoints), C.POINTER(RefMapPoints), C.c_void_p, C.c_float, C.c_void_p,
                      C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int)]
        slot = np.full(kf.n, -1, np.int32)
        rep = np.full(pts.n, -1, np.int32)
        krep = np.full(kf.n, -1, np.int32)
        nm = C.c_int(0)
        ks, ms, ps = kf.struct(), kf_mps.struct(), pts.struct()
        ik = np.ascontiguousarray(in_kf, np.uint8)
        f(C.byref(ks), C.byref(ms), C.byref(ps), _p(ik), float(th), None, _p(slot), _p(rep), _p(krep), C.byref(nm))
        return nm.value, slot, rep, krep

    def fuse_sim3(self, kf, kf_mps, Scw, pts, th):
        from orb_slam2_ssd_semantic_b200 import _abi
        f = self._f("fuse_sim3")
        f.argtypes = [C.POINTER(_abi.OrbmFrame), C.POINTER(RefMapPoints), C.c_void_p, C.POINTER(RefMapPoints), C.c_float, C.c_void_p,
                      C.c_void_p, C.POINTER(C.c_int)]
        slot = np.full(kf.n, -1, np.int32)
        rep = np.full(pts.n, -1, np.int32)
        nm = C.c_int(0)
        S = np.ascontiguousarray(Scw, np.float32).reshape(16)
        ks, ms, ps = kf.struct(), kf_mps.struct(), pts.struct()
        f(C.byref(ks), C.byref(ms), _p(S), C.byref(ps), float(th), _p(slot), _p(rep), C.byref(nm))
        return nm.value, slot, rep

    def search_by_sim3(self, kf1, kf2, mp1, mp2, matches12, s12, R12, t12, th):
        from orb_slam2_ssd_semantic_b200 import _abi
        f = self._f("search_by_sim3")
        f.argtypes = [C.POINTER(_abi.OrbmFrame), C.POINTER(_abi.OrbmFrame), C.POINTER(RefMapPoints), C.POINTER(RefMapPoints), C.c_void_p,
                      C.c_float, C.c_void_p, C.c_void_p, C.c_float, C.POINTER(C.c_int)]
        m = np.ascontiguousarray(matches12, np.int32).copy()
        R = np.ascontiguousarray(R12, np.float32).reshape(9)
        t = np.ascontiguousarray(t12, np.float32).reshape(3)
        nm = C.c_int(0)
        a, b, p1, p2 = kf1.struct(), kf2.struct(), mp1.struct(), mp2.struct()
        f(C.byref(a), C.byref(b), C.byref(p1), C.byref(p2), _p(m), float(s12), _p(R), _p(t), float(th), C.byref(nm))
        return nm.value, m

    def triangulation(self, k1, k2, Tcw1, Tcw2, cam, F12, only_stereo=False, nnratio=0.6, check_ori=True):
        from orb_slam2_ssd_semantic_b200 import _abi
        f = self._f("triangulation")
        f.argtypes = [C.POINTER(_abi.OrbmTriKF), C.POINTER(_abi.OrbmTriKF), C.c_void_p, C.c_void_p, C.POINTER(_abi.OrbmFrame), C.c_void_p,
                      C.c_int, C.c_float, C.c_int, C.c_void_p, C.POINTER(C.c_int), C.c_void_p]
        out = np.full(max(k1.n, 1), -1, np.int32)
        ep = np.zeros(2, np.float32)
        nm = C.c_int(0)
        a, b, cs = k1.struct(), k2.struct(), cam.struct()
        T1 = np.ascontiguousarray(Tcw1, np.float32).reshape(16)
        T2 = np.ascontiguousarray(Tcw2, np.float32).reshape(16)
        F = np.ascontiguousarray(F12, np.float32).reshape(9)
        f(C.byref(a), C.byref(b), _p(T1), _p(T2), C.byref(cs), _p(F), int(only_stereo), float(nnratio), int(check_ori), _p(out),
          C.byref(nm), _p(ep))
        return nm.value, out[:k1.n], ep

    def kf_best(self, kf, queries):
        from orb_slam2_ssd_semantic_b200 import _abi
        f = self._f("kf_best")
        f.argtypes = [C.POINTER(_abi.OrbmFrame), C.POINTER(_abi.OrbmQueries), C.c_void_p, C.c_void_p]
        bi = np.full(max(queries.n, 1), -1, np.int32)
        bd = np.full(max(queries.n, 1), 2 ** 31 - 1, np.int32)
        ks, qs = kf.struct(), queries.struct()
        f(C.byref(ks), C.byref(qs), _p(bi), _p(bd))
        return bi[:queries.n], bd[:queries.n]

    def frame_rgbd(self, gray, depth, Tcw, fx, fy, cx, cy, bf, nfeatures=1000):
        f = self._f("frame_rgbd")
        f.argtypes = ([C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int, C.c_int, C.c_void_p] +
                      [C.c_float] * 5 + [C.c_void_p] * 7 + [C.c_int, C.c_void_p])
        gray = np.ascontiguousarray(gray, np.uint8)
        depth = np.ascontiguousarray(depth, np.float32)
        T = np.ascontiguousarray(Tcw, np.float32).reshape(16)
        cap = nfeatures + 16 * 8 + 64
        kps = np.zeros(cap, KP_DTYPE)
        desc = np.zeros((cap, 32), np.uint8)
        ur, dp, xw, va = np.zeros(cap, np.float32), np.zeros(cap, np.float32), np.zeros((cap, 3), np.float32), np.zeros(cap, np.uint8)
        n = C.c_int(0)
        rc = f(_p(gray), _p(depth), gray.shape[0], gray.shape[1], nfeatures, 1.2, 8, 20, 7, _p(T), fx, fy, cx, cy, bf, None,
               _p(kps), _p(desc), _p(ur), _p(dp), _p(xw), _p(va), cap, C.byref(n))
        assert rc == 0
        m = n.value
        return kps[:m].copy(), desc[:m].copy(), ur[:m].copy(), dp[:m].copy(), xw[:m].copy(), va[:m].copy()

    def pipeline_run(self, gray, depth, Tcw, nthreads, nfeatures, fx, fy, cx, cy, bf, th=15.0, nnratio=0.9):
        f = self._f("pipeline_run")
        f.restype = C.c_double
        f.argtypes = [C.c_void_p] * 3 + [C.c_int] * 3 + [C.c_int, C.c_float, C.c_int, C.c_int, C.c_int] + [C.c_float] * 7 + \
            [C.c_int] * 2 + [C.c_void_p] * 2
        gray = np.ascontiguousarray(gray, np.uint8)
        depth = np.ascontiguousarray(depth, np.float32)
        T = np.ascontiguousarray(Tcw, np.float32).reshape(-1, 16)
        n, rows, cols = gray.shape
        nkp, nm = np.zeros(n, np.int32), np.zeros(n, np.int32)
        sec = f(_p(gray), _p(depth), _p(T), n, rows, cols, nfeatures, 1.2, 8, 20, 7, fx, fy, cx, cy, bf, th, nnratio, 1, nthreads,
                _p(nkp), _p(nm))
        return sec, nkp, nm


def is_in_frustum(F, xw, normal, min_dist, max_dist, cos_limit, log_sf, which="oracle"):
    """Frame::isInFrustum for n points -> (in_view, proj_x, proj_y, proj_xr, scale_level, view_cos).
    which = 'oracle' (restatement) or 'refsrc' (the reference's own Frame.cc / MapPoint.cc)."""
    from orb_slam2_ssd_semantic_b200 import _abi
    xw = np.ascontiguousarray(xw, np.float32).reshape(-1, 3)
    nr = np.ascontiguousarray(normal, np.float32).reshape(-1, 3)
    mn, mx = np.ascontiguousarray(min_dist, np.float32), np.ascontiguousarray(max_dist, np.float32)
    n = len(xw)
    iv = np.zeros(n, np.uint8)
    px, py, pxr, vc = [np.zeros(n, np.float32) for _ in range(4)]
    lvl = np.zeros(n, np.int32)
    fs = F.struct()
    if which == "oracle":
        L = _mlib()
        L.match_ref_is_in_frustum.argtypes = [C.POINTER(_abi.OrbmFrame), C.c_int] + [C.c_void_p] * 4 + [C.c_float, C.c_float] + [C.c_void_p] * 6
        L.match_ref_is_in_frustum(C.byref(fs), n, _p(xw), _p(nr), _p(mn), _p(mx), float(cos_limit), float(log_sf), _p(iv), _p(px), _p(py),
                                  _p(pxr), _p(lvl), _p(vc))
    else:
        reflib().refsrc_is_in_frustum(C.byref(fs), n, _p(xw), _p(nr), _p(mn), _p(mx), float(cos_limit), _p(iv), _p(px), _p(py), _p(pxr),
                                      _p(lvl), _p(vc))
    return iv, px, py, pxr, lvl, vc


def undistort(xy, K, dist):
    """Frame::UndistortKeyPoints on xy pairs (oracle restatement of cv::undistortPoints)."""
    L = lib()
    L.orb_ref_undistort.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    xy = np.ascontiguousarray(xy, np.float32).reshape(-1, 2)
    K = np.ascontiguousarray(K, np.float32).reshape(9)
    d = np.ascontiguousarray(dist, np.float32)
    out = np.zeros_like(xy)
    L.orb_ref_undistort(_p(xy), len(xy), _p(K), _p(d), len(d), _p(out))
    return out


def synth_vocabulary(seed=3, k=10, L=3, stop_frac=0.05):
    """A synthetic DBoW2-shaped vocabulary: k-ary tree of depth L, children = parent descriptor with ~24 random bits
    flipped, positive idf-like leaf weights (a few 0 = stopped words).  -> (parent, node_desc, weight) in node-id order
    (breadth first, so parent[i] < i and siblings have ascending ids)."""
    rng = np.random.default_rng(seed)
    parent, desc, level = [0], [np.zeros(32, np.uint8)], [0]
    frontier = [0]
    for lvl in range(1, L + 1):
        nxt = []
        for p in frontier:
            for _ in range(k):
                d = desc[p].copy() if p else rng.integers(0, 256, 32, dtype=np.uint8)
                if p:
                    bits = rng.integers(0, 256, 24 // lvl + 4)
                    for b in bits:
                        d[b >> 3] ^= np.uint8(1 << (b & 7))
                parent.append(p); desc.append(d); level.append(lvl)
                nxt.append(len(parent) - 1)
        frontier = nxt
    n = len(parent)
    weight = np.where(np.array(level) == L, rng.uniform(0.5, 9.0, n), 0.0)
    weight[(np.array(level) == L) & (rng.random(n) < stop_frac)] = 0.0
    return np.array(parent, np.int32), np.stack(desc).astype(np.uint8), weight.astype(np.float64)


def bow_transform_py(k, L, parent, node_desc, weight, desc, levelsup=4):
    """Pure-numpy restatement of TemplatedVocabulary::transform (TF-IDF, L1) -> (bow dict, featvec dict)."""
    n_nodes = len(parent)
    children = [[] for _ in range(n_nodes)]
    for i in range(1, n_nodes):
        children[parent[i]].append(i)
    word_of, nw = {}, 0
    for i in range(1, n_nodes):
        if not children[i]:
            word_of[i] = nw
            nw += 1
    bits = np.unpackbits(node_desc, axis=1)
    bow, fv = {}, {}
    for fi, d in enumerate(np.asarray(desc, np.uint8).reshape(-1, 32)):
        db = np.unpackbits(d)
        cur, lvl, nid = 0, 0, 0
        while children[cur]:
            lvl += 1
            ch = children[cur]
            dist = (bits[ch] != db).sum(1)
            cur = ch[int(np.argmin(dist))]          # argmin: first minimum
            if lvl == L - levelsup:
                nid = cur
        w = float(weight[cur])
        if w > 0:
            bow[word_of[cur]] = bow.get(word_of[cur], 0.0) + w
            fv.setdefault(nid, []).append(fi)
    norm = 0.0
    for key in sorted(bow):
        norm += abs(bow[key])
    if norm > 0:
        for key in bow:
            bow[key] /= norm
    return bow, fv


def src_bow_transform(k, L, parent, node_desc, weight, desc, prefix="refsrc"):
    """Frame::ComputeBoW of the reference (prefix refsrc: stand-in DBoW2 on the CPU; shimsrc: shim ORBVocabulary on the
    GPU) -> (bow dict, featvec dict)."""
    Lb = reflib() if prefix == "refsrc" else shimlib()
    f = getattr(Lb, prefix + "_bow_transform")
    f.argtypes = [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int] + [C.c_void_p] * 7
    parent = np.ascontiguousarray(parent, np.int32)
    node_desc = np.ascontiguousarray(node_desc, np.uint8)
    weight = np.ascontiguousarray(weight, np.float64)
    desc = np.ascontiguousarray(desc, np.uint8).reshape(-1, 32)
    n = len(desc)
    words, values = np.zeros(n + 1, np.uint32), np.zeros(n + 1, np.float64)
    node_ids, node_off, idx = np.zeros(n + 1, np.uint32), np.zeros(n + 2, np.int32), np.zeros(n + 1, np.uint32)
    nw, nn = C.c_int(0), C.c_int(0)
    f(k, L, len(parent), _p(parent), _p(node_desc), _p(weight), _p(desc), n, 4, _p(words), _p(values), C.byref(nw), _p(node_ids),
      _p(node_off), _p(idx), C.byref(nn))
    bow = {int(words[i]): float(values[i]) for i in range(nw.value)}
    fv = {int(node_ids[j]): [int(v) for v in idx[node_off[j]:node_off[j + 1]]] for j in range(nn.value)}
    return bow, fv


# ------------------------------------------------------------------------------------------------
# oracle/_ref/librefperfect.so: the `perfect` tree's OWN sources (perfect/src/Frame.cc with its masked RGB-D constructor,
# KeyFrame.cc, MapPoint.cc, Map.cc, ORBextractor.cc, ORBmatcher.cc) compiled unmodified (oracle/Makefile, target `perfect`).
_PERFSO = os.path.join(_HERE, "_ref", "librefperfect.so")
_perflib = None


def refperfect_available() -> bool:
    return os.path.exists(_PERFSO)


def perfect_frames(gray: np.ndarray, depth: np.ndarray, mask: np.ndarray, nfeatures=1000, scale=1.2, nlevels=8, ini_th=20,
                   min_th=7, fx=535.4, fy=539.2, cx=320.1, cy=247.6, bf=40.0):
    """The perfect tree's two RGB-D Frame constructors on one image pair: plain (perfect/src/Frame.cc:255) and masked
    (:328).  -> ((kps, desc) the plain frame keeps, (kps, desc) the masked frame keeps); kps = cv::KeyPoint records (mvKeys)."""
    global _perflib
    from orb_slam2_ssd_semantic_b200.extractor import KP_DTYPE
    if _perflib is None:
        if not os.path.exists(_PERFSO):
            subprocess.check_call(["make", "-C", _HERE, "-s", "perfect"])
        _perflib = C.CDLL(_PERFSO)
        _perflib.refperfect_frames.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int,
                                               C.c_int, C.c_int, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float,
                                               C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
    gray = np.ascontiguousarray(gray, np.uint8)
    depth = np.ascontiguousarray(depth, np.float32)
    mask = np.ascontiguousarray(mask, np.uint8)
    assert gray.shape == depth.shape == mask.shape
    cap = nfeatures + 3 * nlevels + 64
    ka, kb = np.zeros(cap, KP_DTYPE), np.zeros(cap, KP_DTYPE)
    da, db = np.zeros((cap, 32), np.uint8), np.zeros((cap, 32), np.uint8)
    na, nb = C.c_int(0), C.c_int(0)
    rc = _perflib.refperfect_frames(_p(gray), _p(depth), _p(mask), gray.shape[0], gray.shape[1], int(nfeatures), float(scale),
                                    int(nlevels), int(ini_th), int(min_th), float(fx), float(fy), float(cx), float(cy), float(bf),
                                    _p(ka), _p(da), C.byref(na), _p(kb), _p(db), C.byref(nb), cap)
    if rc != 0:
        raise RuntimeError("refperfect_frames: %d" % rc)
    return (ka[:na.value].copy(), da[:na.value].copy()), (kb[:nb.value].copy(), db[:nb.value].copy())
