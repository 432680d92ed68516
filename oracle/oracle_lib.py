"""ORACLE — TEST INFRASTRUCTURE ONLY.

ctypes bindings for oracle/liborbport.so (CPU restatement) and oracle/_ref/liborbref.so (the
reference's own ORBextractor.cc compiled verbatim against oracle/cvshim).  Only tests/,
__graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this
module; the product package (orb_slam2_b200/) never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
PORT_SO = os.path.join(HERE, "liborbport.so")
REF_SO = os.path.join(HERE, "_ref", "liborbref.so")
REFERENCE_ROOT = "/root/reference"

KP_DTYPE = np.dtype([("x", "<f4"), ("y", "<f4"), ("size", "<f4"), ("angle", "<f4"), ("response", "<f4"),
                     ("octave", "<i4"), ("class_id", "<i4")])
assert KP_DTYPE.itemsize == 28

_u8p = C.POINTER(C.c_uint8)
_f32p = C.POINTER(C.c_float)
_i32p = C.POINTER(C.c_int32)


def build(force: bool = False) -> None:
    """Compile the oracle: the restatement and the product's adapter libraries always, the verbatim reference build (_ref)
    only where the reference tree exists."""
    targets = ["port", "adapt"]
    if os.path.exists(os.path.join(REFERENCE_ROOT, "src", "ORBextractor.cc")):
        targets.append("ref")
    if force:
        subprocess.check_call(["make", "-C", HERE, "clean"], stdout=subprocess.DEVNULL)
    subprocess.check_call(["make", "-C", HERE] + targets, stdout=subprocess.DEVNULL)


def have_ref() -> bool:
    return os.path.exists(REF_SO)


def _p(a, t):
    return a.ctypes.data_as(t)


class _ExtractorBase:
    """Shared python face of the two CPU extractors (same call signature as the product's)."""

    def __init__(self, lib, prefix, nfeatures=2000, scale_factor=1.2, nlevels=8, ini_th=20, min_th=7):
        self._lib, self._px = lib, prefix
        self.nfeatures, self.nlevels = nfeatures, nlevels
        create = getattr(lib, prefix + "_create")
        create.restype = C.c_void_p
        create.argtypes = [C.c_int, C.c_float, C.c_int, C.c_int, C.c_int]
        self._h = C.c_void_p(create(nfeatures, scale_factor, nlevels, ini_th, min_th))
        ext = getattr(lib, prefix + "_extract")
        ext.restype = C.c_int
        ext.argtypes = [C.c_void_p, _u8p, C.c_int, C.c_int, C.c_int, C.c_void_p, _u8p, C.c_int]
        self._extract = ext
        tab = getattr(lib, prefix + "_tables")
        tab.restype = None
        tab.argtypes = [C.c_void_p, _f32p, _f32p, _f32p, _f32p, _i32p, _i32p]
        L = nlevels
        self.scale = np.zeros(L, np.float32); self.inv_scale = np.zeros(L, np.float32)
        self.sigma2 = np.zeros(L, np.float32); self.inv_sigma2 = np.zeros(L, np.float32)
        self.per_level = np.zeros(L, np.int32); self.umax = np.zeros(16, np.int32)
        tab(self._h, _p(self.scale, _f32p), _p(self.inv_scale, _f32p), _p(self.sigma2, _f32p),
            _p(self.inv_sigma2, _f32p), _p(self.per_level, _i32p), _p(self.umax, _i32p))

    def __del__(self):
        try:
            d = getattr(self._lib, self._px + "_destroy")
            d.restype = None
            d.argtypes = [C.c_void_p]
            d(self._h)
        except Exception:
            pass

    def __call__(self, img: np.ndarray):
        img = np.ascontiguousarray(img, dtype=np.uint8)
        h, w = img.shape
        cap = self.nfeatures + 64
        while True:
            kps = np.zeros(cap, KP_DTYPE)
            desc = np.zeros((cap, 32), np.uint8)
            n = self._extract(self._h, _p(img, _u8p), w, h, img.strides[0], kps.ctypes.data_as(C.c_void_p), _p(desc, _u8p), cap)
            if n <= cap:
                return kps[:n].copy(), desc[:n].copy()
            cap = n


class PortExtractor(_ExtractorBase):
    def __init__(self, *a, **k):
        lib = C.CDLL(PORT_SO)
        super().__init__(lib, "orbport", *a, **k)
        lib.orbport_level_size.argtypes = [C.c_void_p, C.c_int, _i32p, _i32p]
        lib.orbport_level_ptr.restype = C.c_void_p
        lib.orbport_level_ptr.argtypes = [C.c_void_p, C.c_int]
        lib.orbport_blur_ptr.restype = C.c_void_p
        lib.orbport_blur_ptr.argtypes = [C.c_void_p, C.c_int]
        lib.orbport_candidates.argtypes = [C.c_void_p, C.c_int, _i32p, C.c_int]
        lib.orbport_level_count.argtypes = [C.c_void_p, C.c_int]

    def _level(self, fn, level):
        w, h = C.c_int32(), C.c_int32()
        self._lib.orbport_level_size(self._h, level, C.byref(w), C.byref(h))
        p = fn(self._h, level)
        if not p:
            return None
        return np.ctypeslib.as_array(C.cast(p, _u8p), shape=(h.value, w.value)).copy()

    def level(self, level):
        return self._level(self._lib.orbport_level_ptr, level)

    def blurred(self, level):
        return self._level(self._lib.orbport_blur_ptr, level)

    def candidates(self, level):
        n = self._lib.orbport_candidates(self._h, level, None, 0)
        out = np.zeros((max(n, 1), 3), np.int32)
        self._lib.orbport_candidates(self._h, level, _p(out, _i32p), n)
        return out[:n]

    def level_count(self, level):
        return self._lib.orbport_level_count(self._h, level)


class RefExtractor(_ExtractorBase):
    """The reference's ORBextractor::operator() itself (verbatim source + shim + monotonic allocator)."""

    def __init__(self, *a, **k):
        lib = C.CDLL(REF_SO)
        super().__init__(lib, "orbref", *a, **k)
        lib.orbref_pyramid.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), _i32p, _i32p, _i32p]
        lib.orbref_distribute.argtypes = [C.c_void_p, _f32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                          C.c_int, _f32p, C.c_int]

    def level(self, level):
        p = C.c_void_p()
        w, h, s = C.c_int32(), C.c_int32(), C.c_int32()
        if self._lib.orbref_pyramid(self._h, level, C.byref(p), C.byref(w), C.byref(h), C.byref(s)) != 0:
            return None
        a = np.ctypeslib.as_array(C.cast(p, _u8p), shape=(h.value, s.value))
        return a[:, :w.value].copy()

    def distribute(self, xyr: np.ndarray, width: int, height: int, N: int):
        """DistributeOctTree on (x,y,response) rows relative to minBorder; returns selected rows in list order."""
        xyr = np.ascontiguousarray(xyr, np.float32)
        cap = len(xyr) + 8
        out = np.zeros((cap, 3), np.float32)
        n = self._lib.orbref_distribute(self._h, _p(xyr, _f32p), len(xyr), 16, 16 + width, 16, 16 + height, N, 0,
                                        _p(out, _f32p), cap)
        return out[:n]


def port_lib():
    lib = C.CDLL(PORT_SO)
    lib.orbport_distribute.argtypes = [_i32p, C.c_int, C.c_int, C.c_int, C.c_int, _i32p, C.c_int]
    lib.orbport_hamming.argtypes = [_u8p, _u8p]
    return lib


def port_distribute(xys: np.ndarray, width: int, height: int, N: int) -> np.ndarray:
    lib = port_lib()
    xys = np.ascontiguousarray(xys, np.int32)
    out = np.zeros((len(xys) + 8, 3), np.int32)
    n = lib.orbport_distribute(_p(xys, _i32p), len(xys), width, height, N, _p(out, _i32p), len(out))
    return out[:n]


def port_stereo(kL, dL, kR, dR, pyrL, pyrR, scale, inv_scale, bf, fx):
    """Frame::ComputeStereoMatches restatement. pyrL/pyrR: lists of tight uint8 level images.
    Returns (uRight, depth, sad) with -1 for 'no match'."""
    lib = C.CDLL(PORT_SO)
    nlev = len(pyrL)
    pyrL = [np.ascontiguousarray(p, np.uint8) for p in pyrL]
    pyrR = [np.ascontiguousarray(p, np.uint8) for p in pyrR]
    lw = np.array([p.shape[1] for p in pyrL], np.int32)
    lh = np.array([p.shape[0] for p in pyrL], np.int32)
    PL = (C.c_void_p * nlev)(*[p.ctypes.data for p in pyrL])
    PR = (C.c_void_p * nlev)(*[p.ctypes.data for p in pyrR])
    kL = np.ascontiguousarray(kL); kR = np.ascontiguousarray(kR)
    dL = np.ascontiguousarray(dL, np.uint8); dR = np.ascontiguousarray(dR, np.uint8)
    n = len(kL)
    ur = np.zeros(max(n, 1), np.float32); dp = np.zeros(max(n, 1), np.float32); sad = np.zeros(max(n, 1), np.int32)
    scale = np.ascontiguousarray(scale, np.float32); inv_scale = np.ascontiguousarray(inv_scale, np.float32)
    b = np.float32(bf) / np.float32(fx)
    lib.orbport_stereo.restype = C.c_int
    lib.orbport_stereo.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_float, C.c_float,
                                   C.c_void_p, C.c_void_p, C.c_void_p]
    lib.orbport_stereo(kL.ctypes.data, dL.ctypes.data, n, kR.ctypes.data, dR.ctypes.data, len(kR), PL, PR,
                       lw.ctypes.data, lh.ctypes.data, nlev, scale.ctypes.data, inv_scale.ctypes.data,
                       float(bf), float(b), ur.ctypes.data, dp.ctypes.data, sad.ctypes.data)
    return ur[:n], dp[:n], sad[:n]


# ---------------------------------------------------------------------------------------------- matchers (restatements)
def _plib():
    lib = C.CDLL(PORT_SO)
    lib.orbport_voc_load_text.restype = C.c_void_p
    lib.orbport_voc_random.restype = C.c_void_p
    return lib


def _a(x, dt):
    return None if x is None else np.ascontiguousarray(x, dt)


def _ptr(x):
    return None if x is None else C.c_void_p(x.ctypes.data)


def port_features_in_area(keys, bounds, x, y, r, min_level, max_level):
    lib = _plib()
    keys = _a(keys, KP_DTYPE)
    out = np.zeros(max(len(keys), 1), np.int32)
    lib.orbport_features_in_area.argtypes = [C.c_void_p, C.c_int] + [C.c_float] * 7 + [C.c_int, C.c_int, C.c_void_p, C.c_int]
    n = lib.orbport_features_in_area(_ptr(keys), len(keys), *[float(b) for b in bounds], float(x), float(y), float(r), min_level, max_level,
                                     _ptr(out), len(out))
    return out[:n]


def port_search_by_projection(F, mps, th, nnratio):
    """F: orb_slam2_b200.matcher.FrameView-like, mps: MapPointsView-like (duck typed)."""
    lib = _plib()
    k = _a(F.mvKeysUn, KP_DTYPE); d = _a(F.mDescriptors, np.uint8); ur = _a(F.mvuRight, np.float32); oc = _a(F.occupied, np.uint8)
    sf = _a(F.mvScaleFactors, np.float32)
    px = _a(mps.mTrackProjX, np.float32); py = _a(mps.mTrackProjY, np.float32); pxr = _a(mps.mTrackProjXR, np.float32)
    lv = _a(mps.mnTrackScaleLevel, np.int32); vc = _a(mps.mTrackViewCos, np.float32); md = _a(mps.descriptors, np.uint8)
    va = _a(mps.valid, np.uint8); ho = _a(mps.has_obs, np.uint8)
    match = np.full(max(len(px), 1), -1, np.int32)
    fn = lib.orbport_search_by_projection
    fn.restype = C.c_int
    fn.argtypes = [C.c_void_p] * 4 + [C.c_int] + [C.c_float] * 4 + [C.c_void_p, C.c_int] + [C.c_void_p] * 8 + [C.c_float, C.c_float, C.c_void_p]
    n = fn(_ptr(k), _ptr(d), _ptr(ur), _ptr(oc), len(k), *[float(b) for b in F.bounds], _ptr(sf), len(px), _ptr(px), _ptr(py), _ptr(pxr),
           _ptr(lv), _ptr(vc), _ptr(md), _ptr(va), _ptr(ho), float(th), float(np.float32(nnratio)), _ptr(match))
    return n, match[:len(px)]


def port_search_by_projection_last(Cur, Last, Tcw, K, bf, th, forward, backward, check_ori):
    lib = _plib()
    k = _a(Cur.mvKeysUn, KP_DTYPE); d = _a(Cur.mDescriptors, np.uint8); ur = _a(Cur.mvuRight, np.float32); oc = _a(Cur.occupied, np.uint8)
    sf = _a(Cur.mvScaleFactors, np.float32)
    lk = _a(Last.mvKeysUn, KP_DTYPE); wp = _a(Last.world_pos, np.float32); ld = _a(Last.descriptors, np.uint8)
    va = _a(Last.valid, np.uint8); ho = _a(Last.has_obs, np.uint8)
    T = _a(np.asarray(Tcw, np.float32)[:3, :4].reshape(12), np.float32)
    state = np.full(max(len(k), 1), -1, np.int32)
    fn = lib.orbport_search_by_projection_last
    fn.restype = C.c_int
    fn.argtypes = [C.c_void_p] * 4 + [C.c_int] + [C.c_float] * 4 + [C.c_void_p] * 6 + [C.c_int, C.c_void_p] + [C.c_float] * 6 + [C.c_int] * 3 + [C.c_void_p]
    n = fn(_ptr(k), _ptr(d), _ptr(ur), _ptr(oc), len(k), *[float(b) for b in Cur.bounds], _ptr(sf), _ptr(lk), _ptr(wp), _ptr(ld), _ptr(va),
           _ptr(ho), len(lk), _ptr(T), float(K[0]), float(K[1]), float(K[2]), float(K[3]), float(bf), float(th), int(forward), int(backward),
           int(check_ori), _ptr(state))
    return n, state[:len(k)]


def _log_scale(F):
    """Frame::mfLogScaleFactor = log(mfScaleFactor) (Frame.cc:71): glibc logf of the float scale factor."""
    v = getattr(F, "mfLogScaleFactor", None)
    if v is not None:
        return float(v)
    libm = C.CDLL("libm.so.6")
    libm.logf.restype = C.c_float
    libm.logf.argtypes = [C.c_float]
    return float(libm.logf(float(np.float32(F.mvScaleFactors[1]))))


def _points_args(P):
    wp = _a(P.world_pos, np.float32); md = _a(P.descriptors, np.uint8)
    mx = _a(P.max_distance, np.float32); mn = _a(P.min_distance, np.float32)
    va = _a(P.valid, np.uint8) if P.valid is not None else np.ones(len(wp), np.uint8)
    return wp, md, mx, mn, va


def port_search_by_projection_kf(Cur, P, Tcw, Ow, K, th, orb_dist, check_ori):
    """SearchByProjection(CurrentFrame, KeyFrame, sAlreadyFound, th, ORBdist) (ORBmatcher.cc:1472-1599)."""
    lib = _plib()
    k = _a(Cur.mvKeysUn, KP_DTYPE); d = _a(Cur.mDescriptors, np.uint8); oc = _a(Cur.occupied, np.uint8)
    sf = _a(Cur.mvScaleFactors, np.float32)
    wp, md, mx, mn, va = _points_args(P)
    ang = _a(P.angle, np.float32)
    T = _a(np.asarray(Tcw, np.float32)[:3, :4].reshape(12), np.float32); ow = _a(np.asarray(Ow, np.float32).reshape(3), np.float32)
    state = np.full(max(len(k), 1), -1, np.int32)
    fn = lib.orbport_search_by_projection_kf
    fn.restype = C.c_int
    fn.argtypes = ([C.c_void_p] * 3 + [C.c_int] + [C.c_float] * 4 + [C.c_void_p, C.c_int, C.c_float] + [C.c_void_p] * 6 + [C.c_int]
                   + [C.c_void_p] * 2 + [C.c_float] * 5 + [C.c_int, C.c_int, C.c_void_p])
    n = fn(_ptr(k), _ptr(d), _ptr(oc), len(k), *[float(b) for b in Cur.bounds], _ptr(sf), len(sf), _log_scale(Cur),
           _ptr(ang), _ptr(wp), _ptr(md), _ptr(mx), _ptr(mn), _ptr(va), len(wp), _ptr(T), _ptr(ow), float(K[0]), float(K[1]), float(K[2]),
           float(K[3]), float(th), int(orb_dist), int(check_ori), _ptr(state))
    return n, state[:len(k)]


def port_search_by_projection_sim3(KF, P, Tcw, Ow, K, th):
    """SearchByProjection(KeyFrame*, Scw, vpPoints, vpMatched, th) (ORBmatcher.cc:290-403); Tcw = [Rcw|tcw] with the scale divided out."""
    lib = _plib()
    k = _a(KF.mvKeysUn, KP_DTYPE); d = _a(KF.mDescriptors, np.uint8); oc = _a(KF.occupied, np.uint8)
    sf = _a(KF.mvScaleFactors, np.float32)
    wp, md, mx, mn, va = _points_args(P)
    nr = _a(P.normal, np.float32)
    T = _a(np.asarray(Tcw, np.float32)[:3, :4].reshape(12), np.float32); ow = _a(np.asarray(Ow, np.float32).reshape(3), np.float32)
    state = np.full(max(len(k), 1), -1, np.int32)
    fn = lib.orbport_search_by_projection_sim3
    fn.restype = C.c_int
    fn.argtypes = ([C.c_void_p] * 3 + [C.c_int] + [C.c_float] * 4 + [C.c_void_p, C.c_int, C.c_float] + [C.c_void_p] * 6 + [C.c_int]
                   + [C.c_void_p] * 2 + [C.c_float] * 4 + [C.c_int, C.c_void_p])
    n = fn(_ptr(k), _ptr(d), _ptr(oc), len(k), *[float(b) for b in KF.bounds], _ptr(sf), len(sf), _log_scale(KF),
           _ptr(wp), _ptr(md), _ptr(mx), _ptr(mn), _ptr(nr), _ptr(va), len(wp), _ptr(T), _ptr(ow), float(K[0]), float(K[1]), float(K[2]),
           float(K[3]), int(th), _ptr(state))
    return n, state[:len(k)]


def port_fuse(KF, P, Tcw, Ow, K, bf, th, scw):
    """Search part of Fuse(pKF, vpMapPoints, th) (ORBmatcher.cc:825-970) / Fuse(pKF, Scw, ...) (:972-1100)."""
    lib = _plib()
    k = _a(KF.mvKeysUn, KP_DTYPE); d = _a(KF.mDescriptors, np.uint8); sf = _a(KF.mvScaleFactors, np.float32)
    ur = _a(KF.mvuRight, np.float32) if KF.mvuRight is not None else None
    inv = _a(KF.mvInvLevelSigma2, np.float32) if KF.mvInvLevelSigma2 is not None else None
    wp, md, mx, mn, va = _points_args(P)
    nr = _a(P.normal, np.float32)
    T = _a(np.asarray(Tcw, np.float32)[:3, :4].reshape(12), np.float32); ow = _a(np.asarray(Ow, np.float32).reshape(3), np.float32)
    best = np.full(max(len(wp), 1), -1, np.int32)
    fn = lib.orbport_fuse
    fn.restype = C.c_int
    fn.argtypes = ([C.c_void_p] * 4 + [C.c_int] + [C.c_float] * 4 + [C.c_void_p, C.c_int, C.c_float] + [C.c_void_p] * 6 + [C.c_int]
                   + [C.c_void_p] * 2 + [C.c_float] * 6 + [C.c_int, C.c_void_p])
    n = fn(_ptr(k), _ptr(d), _ptr(ur) if ur is not None else None, _ptr(inv) if inv is not None else None, len(k),
           *[float(b) for b in KF.bounds], _ptr(sf), len(sf), _log_scale(KF), _ptr(wp), _ptr(md), _ptr(mx), _ptr(mn), _ptr(nr), _ptr(va),
           len(wp), _ptr(T), _ptr(ow), float(K[0]), float(K[1]), float(K[2]), float(K[3]), float(bf), float(th), int(scw), _ptr(best))
    return n, best[:len(wp)]


def port_search_by_sim3(KF1, KF2, P1, P2, T1w, T2w, S12, S21, K, th):
    """SearchBySim3 (ORBmatcher.cc:1102-1326)."""
    lib = _plib()
    k1 = _a(KF1.mvKeysUn, KP_DTYPE); d1 = _a(KF1.mDescriptors, np.uint8); sf1 = _a(KF1.mvScaleFactors, np.float32)
    k2 = _a(KF2.mvKeysUn, KP_DTYPE); d2 = _a(KF2.mDescriptors, np.uint8); sf2 = _a(KF2.mvScaleFactors, np.float32)
    b1 = _a(np.asarray(KF1.bounds, np.float32), np.float32); b2 = _a(np.asarray(KF2.bounds, np.float32), np.float32)
    wp1, md1, mx1, mn1, va1 = _points_args(P1)
    wp2, md2, mx2, mn2, va2 = _points_args(P2)
    mats = [_a(np.asarray(M, np.float32)[:3, :4].reshape(12), np.float32) for M in (T1w, T2w, S12, S21)]
    match = np.full(max(len(k1), 1), -1, np.int32)
    fn = lib.orbport_search_by_sim3
    fn.restype = C.c_int
    fn.argtypes = ([C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_float] * 2 + [C.c_int] + [C.c_void_p] * 10 + [C.c_void_p] * 4
                   + [C.c_float] * 5 + [C.c_void_p])
    n = fn(_ptr(k1), _ptr(d1), len(k1), _ptr(b1), _ptr(sf1), _log_scale(KF1), _ptr(k2), _ptr(d2), len(k2), _ptr(b2), _ptr(sf2),
           _log_scale(KF2), len(sf1), _ptr(wp1), _ptr(md1), _ptr(mx1), _ptr(mn1), _ptr(va1), _ptr(wp2), _ptr(md2), _ptr(mx2), _ptr(mn2),
           _ptr(va2), *[_ptr(M) for M in mats], float(K[0]), float(K[1]), float(K[2]), float(K[3]), float(th), _ptr(match))
    return n, match[:len(k1)]


def port_search_for_initialization(F1, F2, prev_matched, window, nnratio, check_ori):
    """SearchForInitialization (ORBmatcher.cc:405-520); returns (nmatches, vnMatches12, updated vbPrevMatched)."""
    lib = _plib()
    k1 = _a(F1.mvKeysUn, KP_DTYPE); d1 = _a(F1.mDescriptors, np.uint8)
    k2 = _a(F2.mvKeysUn, KP_DTYPE); d2 = _a(F2.mDescriptors, np.uint8)
    prev = np.ascontiguousarray(np.asarray(prev_matched, np.float32).reshape(-1, 2)).copy()
    m12 = np.full(max(len(k1), 1), -1, np.int32)
    fn = lib.orbport_search_for_initialization
    fn.restype = C.c_int
    fn.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int] + [C.c_float] * 4 + [C.c_void_p, C.c_int, C.c_float, C.c_int, C.c_void_p]
    n = fn(_ptr(k1), _ptr(d1), len(k1), _ptr(k2), _ptr(d2), len(k2), *[float(b) for b in F2.bounds], _ptr(prev), int(window),
           float(np.float32(nnratio)), int(check_ori), _ptr(m12))
    return n, m12[:len(k1)], prev


def port_distinctive_descriptor(desc):
    """MapPoint::ComputeDistinctiveDescriptors (MapPoint.cc:242-307) for one MapPoint's observation descriptors."""
    lib = _plib()
    d = _a(np.asarray(desc, np.uint8).reshape(-1, 32), np.uint8)
    fn = lib.orbport_distinctive_descriptor
    fn.restype = C.c_int
    fn.argtypes = [C.c_void_p, C.c_int]
    return int(fn(_ptr(d) if len(d) else None, len(d)))


def port_bow_score(bow1, bow2):
    """(L1 score, common words, first common word) of two BowVectors given as {word: value} dicts (ScoringObject.cpp:23-71)."""
    lib = _plib()
    w1 = _a(np.fromiter(bow1.keys(), np.uint32, len(bow1)), np.uint32); v1 = _a(np.fromiter(bow1.values(), np.float64, len(bow1)), np.float64)
    w2 = _a(np.fromiter(bow2.keys(), np.uint32, len(bow2)), np.uint32); v2 = _a(np.fromiter(bow2.values(), np.float64, len(bow2)), np.float64)
    fn = lib.orbport_bow_score_l1
    fn.restype = C.c_double
    fn.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    common = C.c_int32(0); first = C.c_uint32(0)
    s = fn(_ptr(w1) if len(w1) else None, _ptr(v1) if len(v1) else None, len(w1), _ptr(w2) if len(w2) else None,
           _ptr(v2) if len(v2) else None, len(w2), C.addressof(common), C.addressof(first))
    return float(s), common.value, first.value


def port_detect_reloc_candidates(kf_bows, n_words, q_bow, neigh):
    """KeyFrameDatabase::DetectRelocalizationCandidates (KeyFrameDatabase.cc:199-310) over keyframes added in list order."""
    lib = _plib()
    start = np.zeros(len(kf_bows) + 1, np.int32)
    start[1:] = np.cumsum([len(b) for b in kf_bows])
    kw = _a(np.concatenate([np.fromiter(b.keys(), np.uint32, len(b)) for b in kf_bows] + [np.zeros(0, np.uint32)]), np.uint32)
    kv = _a(np.concatenate([np.fromiter(b.values(), np.float64, len(b)) for b in kf_bows] + [np.zeros(0, np.float64)]), np.float64)
    qw = _a(np.fromiter(q_bow.keys(), np.uint32, len(q_bow)), np.uint32); qv = _a(np.fromiter(q_bow.values(), np.float64, len(q_bow)), np.float64)
    ng = _a(np.asarray(neigh, np.int32).reshape(len(kf_bows), 10), np.int32)
    out = np.zeros(max(len(kf_bows), 1), np.int32)
    fn = lib.orbport_detect_reloc_candidates
    fn.restype = C.c_int
    fn.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    n = fn(len(kf_bows), _ptr(start), _ptr(kw), _ptr(kv), int(n_words), _ptr(qw), _ptr(qv), len(qw), _ptr(ng), _ptr(out))
    return out[:n].copy()


def port_is_in_frustum(F, P, Tcw, Ow, K, mbf, viewing_cos_limit=0.5):
    """Frame::isInFrustum (Frame.cc:269-325) for every point of P; returns dict of the MapPoint track fields."""
    lib = _plib()
    wp, md, mx, mn, va = _points_args(P)
    nr = _a(P.normal, np.float32)
    T = _a(np.asarray(Tcw, np.float32)[:3, :4].reshape(12), np.float32); ow = _a(np.asarray(Ow, np.float32).reshape(3), np.float32)
    n = len(wp)
    inv = np.zeros(max(n, 1), np.uint8); px = np.zeros(max(n, 1), np.float32); py = np.zeros(max(n, 1), np.float32)
    pxr = np.zeros(max(n, 1), np.float32); lv = np.zeros(max(n, 1), np.int32); vc = np.zeros(max(n, 1), np.float32)
    fn = lib.orbport_is_in_frustum
    fn.restype = C.c_int
    fn.argtypes = [C.c_void_p] * 5 + [C.c_int, C.c_void_p, C.c_void_p] + [C.c_float] * 11 + [C.c_int] + [C.c_void_p] * 6
    cnt = fn(_ptr(wp), _ptr(nr), _ptr(mx), _ptr(mn), _ptr(va), n, _ptr(T), _ptr(ow), float(K[0]), float(K[1]), float(K[2]), float(K[3]),
             float(mbf), *[float(b) for b in F.bounds], float(viewing_cos_limit), _log_scale(F), len(F.mvScaleFactors), _ptr(inv), _ptr(px),
             _ptr(py), _ptr(pxr), _ptr(lv), _ptr(vc))
    return dict(count=cnt, in_view=inv[:n], proj_x=px[:n], proj_y=py[:n], proj_xr=pxr[:n], level=lv[:n], view_cos=vc[:n])


def port_detect_loop_candidates(kf_bows, n_words, q_bow, connected, neigh, min_score):
    """KeyFrameDatabase::DetectLoopCandidates (KeyFrameDatabase.cc:76-197) over keyframes added in list order."""
    lib = _plib()
    start = np.zeros(len(kf_bows) + 1, np.int32)
    start[1:] = np.cumsum([len(b) for b in kf_bows])
    kw = _a(np.concatenate([np.fromiter(b.keys(), np.uint32, len(b)) for b in kf_bows] + [np.zeros(0, np.uint32)]), np.uint32)
    kv = _a(np.concatenate([np.fromiter(b.values(), np.float64, len(b)) for b in kf_bows] + [np.zeros(0, np.float64)]), np.float64)
    qw = _a(np.fromiter(q_bow.keys(), np.uint32, len(q_bow)), np.uint32); qv = _a(np.fromiter(q_bow.values(), np.float64, len(q_bow)), np.float64)
    ng = _a(np.asarray(neigh, np.int32).reshape(len(kf_bows), 10), np.int32)
    cn = _a(np.asarray(connected, np.uint8), np.uint8)
    out = np.zeros(max(len(kf_bows), 1), np.int32)
    fn = lib.orbport_detect_loop_candidates
    fn.restype = C.c_int
    fn.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p]
    n = fn(len(kf_bows), _ptr(start), _ptr(kw), _ptr(kv), int(n_words), _ptr(qw), _ptr(qv), len(qw), _ptr(cn), _ptr(ng),
           float(np.float32(min_score)), _ptr(out))
    return out[:n].copy()


def _kf_args(kf):
    k = _a(kf.mvKeysUn, KP_DTYPE); d = _a(kf.mDescriptors, np.uint8)
    hm = _a(kf.has_mp, np.uint8) if kf.has_mp is not None else np.zeros(len(k), np.uint8)
    nd = _a(kf.mFeatVec.node_id, np.uint32); st = _a(kf.mFeatVec.start, np.int32); fi = _a(kf.mFeatVec.feat_idx, np.uint32)
    return k, d, hm, nd, st, fi


def port_search_by_bow(kf, F, nnratio, check_ori):
    lib = _plib()
    k1, d1, hm1, nd1, st1, fi1 = _kf_args(kf)
    k2, d2, _, nd2, st2, fi2 = _kf_args(F)
    match = np.full(max(len(k2), 1), -1, np.int32)
    fn = lib.orbport_search_by_bow_kf_f
    fn.restype = C.c_int
    fn.argtypes = [C.c_void_p] * 3 + [C.c_int, C.c_int] + [C.c_void_p] * 3 + [C.c_void_p] * 2 + [C.c_int, C.c_int] + [C.c_void_p] * 3 + [C.c_float, C.c_int, C.c_void_p]
    n = fn(_ptr(k1), _ptr(d1), _ptr(hm1), len(k1), len(nd1), _ptr(nd1), _ptr(st1), _ptr(fi1), _ptr(k2), _ptr(d2), len(k2), len(nd2),
           _ptr(nd2), _ptr(st2), _ptr(fi2), float(np.float32(nnratio)), int(check_ori), _ptr(match))
    return n, match[:len(k2)]


def port_search_by_bow_kf(kf1, kf2, nnratio, check_ori):
    lib = _plib()
    k1, d1, hm1, nd1, st1, fi1 = _kf_args(kf1)
    k2, d2, hm2, nd2, st2, fi2 = _kf_args(kf2)
    match = np.full(max(len(k1), 1), -1, np.int32)
    fn = lib.orbport_search_by_bow_kf_kf
    fn.restype = C.c_int
    fn.argtypes = ([C.c_void_p] * 3 + [C.c_int, C.c_int] + [C.c_void_p] * 3) * 2 + [C.c_float, C.c_int, C.c_void_p]
    n = fn(_ptr(k1), _ptr(d1), _ptr(hm1), len(k1), len(nd1), _ptr(nd1), _ptr(st1), _ptr(fi1), _ptr(k2), _ptr(d2), _ptr(hm2), len(k2),
           len(nd2), _ptr(nd2), _ptr(st2), _ptr(fi2), float(np.float32(nnratio)), int(check_ori), _ptr(match))
    return n, match[:len(k1)]


def port_search_for_triangulation(kf1, kf2, F12, epipole, only_stereo, check_ori):
    lib = _plib()
    k1, d1, hm1, nd1, st1, fi1 = _kf_args(kf1)
    k2, d2, hm2, nd2, st2, fi2 = _kf_args(kf2)
    ur1 = _a(kf1.mvuRight, np.float32); ur2 = _a(kf2.mvuRight, np.float32)
    f = _a(np.asarray(F12).reshape(9), np.float32)
    sf2 = _a(kf2.mvScaleFactors, np.float32); sg2 = _a(kf2.mvLevelSigma2, np.float32)
    pairs = np.zeros((max(len(k1), 1), 2), np.int32)
    fn = lib.orbport_search_for_triangulation
    fn.restype = C.c_int
    fn.argtypes = ([C.c_void_p] * 4 + [C.c_int, C.c_int] + [C.c_void_p] * 3) * 2 + [C.c_void_p, C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
    n = fn(_ptr(k1), _ptr(d1), _ptr(hm1), _ptr(ur1), len(k1), len(nd1), _ptr(nd1), _ptr(st1), _ptr(fi1), _ptr(k2), _ptr(d2), _ptr(hm2),
           _ptr(ur2), len(k2), len(nd2), _ptr(nd2), _ptr(st2), _ptr(fi2), _ptr(f), float(epipole[0]), float(epipole[1]), _ptr(sf2), _ptr(sg2),
           int(only_stereo), int(check_ori), _ptr(pairs))
    return pairs[:n]


class PortVocabulary:
    """CPU restatement of the DBoW2 tree (text loader, seeded random tree of ORBvoc's shape, transform)."""

    def __init__(self, handle):
        self._lib = _plib()
        self._h = C.c_void_p(handle)

    @staticmethod
    def random(k=10, L=6, seed=7):
        lib = _plib()
        lib.orbport_voc_random.argtypes = [C.c_int, C.c_int, C.c_uint]
        return PortVocabulary(lib.orbport_voc_random(k, L, seed))

    @staticmethod
    def load_text(path):
        lib = _plib()
        lib.orbport_voc_load_text.argtypes = [C.c_char_p]
        h = lib.orbport_voc_load_text(path.encode())
        if not h:
            raise IOError(path)
        return PortVocabulary(h)

    def export(self):
        self._lib.orbport_voc_nodes.argtypes = [C.c_void_p]
        n = self._lib.orbport_voc_nodes(self._h)
        parent = np.zeros(n, np.int32); leaf = np.zeros(n, np.uint8); word = np.zeros(n, np.int32)
        desc = np.zeros((n, 32), np.uint8); weight = np.zeros(n, np.float64)
        k, L = C.c_int(), C.c_int()
        self._lib.orbport_voc_export.argtypes = [C.c_void_p] * 6 + [C.POINTER(C.c_int), C.POINTER(C.c_int)]
        self._lib.orbport_voc_export(self._h, _ptr(parent), _ptr(leaf), _ptr(word), _ptr(desc), _ptr(weight), C.byref(k), C.byref(L))
        return dict(parent=parent, is_leaf=leaf, word_id=word, desc=desc, weight=weight, k=k.value, L=L.value)

    def save_text(self, path):
        e = self.export()
        with open(path, "w") as f:
            f.write(f"{e['k']} {e['L']} 0 0\n")
            for i in range(1, len(e["parent"])):
                f.write(f"{e['parent'][i]} {int(e['is_leaf'][i])} " + " ".join(str(int(b)) for b in e["desc"][i]) + f" {repr(float(e['weight'][i]))}\n")

    def transform_raw(self, desc, levelsup=4):
        d = _a(desc, np.uint8)
        n = len(d)
        word = np.zeros(max(n, 1), np.int32); weight = np.zeros(max(n, 1), np.float64); node = np.zeros(max(n, 1), np.int32)
        self._lib.orbport_voc_transform.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        self._lib.orbport_voc_transform(self._h, _ptr(d), n, levelsup, _ptr(word), _ptr(weight), _ptr(node))
        return word[:n], weight[:n], node[:n]

    def __del__(self):
        try:
            self._lib.orbport_voc_free.argtypes = [C.c_void_p]
            self._lib.orbport_voc_free(self._h)
        except Exception:
            pass


# ---------------------------------------------------------------------------------------------------------------------
# The reference's own src/ORBmatcher.cc, compiled verbatim (oracle/_ref/libmatchref.so, see oracle/Makefile and
# oracle/matchref_wrap.cpp).  These wrappers take the same view objects as the port_* functions above and return the
# results in the port's conventions, so a test can assert  port(x) == ref(x)  directly.
MATCHREF_SO = os.path.join(HERE, "_ref", "libmatchref.so")


def have_matchref() -> bool:
    return os.path.exists(MATCHREF_SO)


def _mlib():
    return C.CDLL(MATCHREF_SO)


def _f32(a, n=None):
    return _a(np.asarray(a, np.float32).reshape(-1) if n is None else np.asarray(a, np.float32).reshape(n), np.float32)


def _T12(T):
    return _a(np.asarray(T, np.float32)[:3, :4].reshape(12), np.float32)


def ref_descriptor_distance(a, b):
    lib = _mlib()
    a = _a(a, np.uint8); b = _a(b, np.uint8)
    lib.matchref_descriptor_distance.restype = C.c_int
    lib.matchref_descriptor_distance.argtypes = [C.c_void_p, C.c_void_p]
    return lib.matchref_descriptor_distance(_ptr(a), _ptr(b))


def ref_decompose_scw(Scw):
    """ORBmatcher.cc:298-303 with the shim's cv::Mat arithmetic -> (Tcw 3x4 = [Rcw|tcw], Ow)."""
    lib = _mlib()
    T = np.zeros(12, np.float32); ow = np.zeros(3, np.float32); s = _T12(Scw)
    lib.matchref_decompose_scw.argtypes = [C.c_void_p] * 3
    lib.matchref_decompose_scw(_ptr(s), _ptr(T), _ptr(ow))
    return T.reshape(3, 4), ow


def ref_sim3_mats(s12, R12, t12):
    lib = _mlib()
    S12 = np.zeros(12, np.float32); S21 = np.zeros(12, np.float32)
    r = _f32(R12, 9); t = _f32(t12, 3)
    lib.matchref_sim3_mats.argtypes = [C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.matchref_sim3_mats(float(np.float32(s12)), _ptr(r), _ptr(t), _ptr(S12), _ptr(S21))
    return S12.reshape(3, 4), S21.reshape(3, 4)


def ref_camera_center(Tcw):
    lib = _mlib()
    ow = np.zeros(3, np.float32); T = _T12(Tcw)
    lib.matchref_camera_center.argtypes = [C.c_void_p] * 2
    lib.matchref_camera_center(_ptr(T), _ptr(ow))
    return ow


def ref_epipole(Ow1, T2w, K2):
    lib = _mlib()
    o = _f32(Ow1, 3); T = _T12(T2w); ex = C.c_float(); ey = C.c_float()
    lib.matchref_epipole.argtypes = [C.c_void_p, C.c_void_p] + [C.c_float] * 4 + [C.c_void_p] * 2
    lib.matchref_epipole(_ptr(o), _ptr(T), *[float(x) for x in K2], C.addressof(ex), C.addressof(ey))
    return float(ex.value), float(ey.value)


def ref_forward_backward(TcwCur, TcwLast, mb, bMono):
    lib = _mlib()
    a = _T12(TcwCur); b = _T12(TcwLast); f = C.c_int(); w = C.c_int()
    lib.matchref_forward_backward.argtypes = [C.c_void_p, C.c_void_p, C.c_float, C.c_int, C.c_void_p, C.c_void_p]
    lib.matchref_forward_backward(_ptr(a), _ptr(b), float(mb), int(bMono), C.addressof(f), C.addressof(w))
    return bool(f.value), bool(w.value)


def _opt(a, dt):
    return _a(a, dt) if a is not None else None


def _p0(a):
    return _ptr(a) if a is not None else None


def ref_search_by_projection(F, mps, th, nnratio):
    """-> (nmatches, owner[F.N]): index of the map point in F.mvpMapPoints[idx] afterwards, -3 prior occupant, -1 none."""
    lib = _mlib()
    k = _a(F.mvKeysUn, KP_DTYPE); d = _a(F.mDescriptors, np.uint8); ur = _opt(F.mvuRight, np.float32); oc = _opt(F.occupied, np.uint8)
    sf = _a(F.mvScaleFactors, np.float32)
    px = _a(mps.mTrackProjX, np.float32); py = _a(mps.mTrackProjY, np.float32); pxr = _a(mps.mTrackProjXR, np.float32)
    lv = _a(mps.mnTrackScaleLevel, np.int32); vc = _a(mps.mTrackViewCos, np.float32); md = _a(mps.descriptors, np.uint8)
    va = _opt(mps.valid, np.uint8); ho = _opt(mps.has_obs, np.uint8)
    owner = np.full(max(len(k), 1), -1, np.int32)
    fn = lib.matchref_search_by_projection
    fn.restype = C.c_int
    fn.argtypes = [C.c_void_p] * 4 + [C.c_int] + [C.c_float] * 4 + [C.c_void_p, C.c_int, C.c_int] + [C.c_void_p] * 8 + [C.c_float, C.c_float, C.c_void_p]
    n = fn(_ptr(k), _ptr(d), _p0(ur), _p0(oc), len(k), *[float(b) for b in F.bounds], _ptr(sf), len(sf), len(px), _ptr(px), _ptr(py),
           _ptr(pxr), _ptr(lv), _ptr(vc), _ptr(md), _p0(va), _p0(ho), float(th), float(np.float32(nnratio)), _ptr(owner))
    return n, owner[:len(k)]


def owner_from_matches(F, mps, match):
    """What F.mvpMapPoints looks like after applying the port's per-map-point matches in order (ORBmatcher.cc:123)."""
    owner = np.where(np.asarray(F.occupied if F.occupied is not None else np.zeros(len(F.mvKeysUn)), bool), -3, -1).astype(np.int32)
    for i, f in enumerate(match):
        if f >= 0:
            owner[f] = i
    return owner


def owner_from_state(occupied, state):
    """Port state (>=0 query, -1 untouched, -2 culled) -> pointer view: index, -3 prior occupant, -1 NULL."""
    occ = np.asarray(occupied if occupied is not None else np.zeros(len(state)), bool)
    return np.where(state >= 0, state, np.where((state == -1) & occ, -3, -1)).astype(np.int32)


def ref_search_by_projection_last(Cur, Last, TcwCur, TcwLast, K, bf, mb, th, bMono, check_ori):
    lib = _mlib()
    k = _a(Cur.mvKeysUn, KP_DTYPE); d = _a(Cur.mDescriptors, np.uint8); ur = _opt(Cur.mvuRight, np.float32); oc = _opt(Cur.occupied, np.uint8)
    sf = _a(Cur.mvScaleFactors, np.float32)
    lk = _a(Last.mvKeysUn, KP_DTYPE); wp = _a(Last.world_pos, np.float32); ld = _a(Last.descriptors, np.uint8)
    va = _opt(Last.valid, np.uint8); ho = _opt(Last.has_obs, np.uint8)
    Tc = _T12(TcwCur); Tl = _T12(TcwLast)
    owner = np.full(max(len(k), 1), -1, np.int32)
    fn = lib.matchref_search_by_projection_last
    fn.restype = C.c_int
    fn.argtypes = ([C.c_void_p] * 4 + [C.c_int] + [C.c_float] * 4 + [C.c_void_p, C.c_int] + [C.c_void_p] * 5 + [C.c_int] + [C.c_void_p] * 2
                   + [C.c_float] * 7 + [C.c_int, C.c_int, C.c_void_p])
    n = fn(_ptr(k), _ptr(d), _p0(ur), _p0(oc), len(k), *[float(b) for b in Cur.bounds], _ptr(sf), len(sf), _ptr(lk), _ptr(wp), _ptr(ld),
           _p0(va), _p0(ho), len(lk), _ptr(Tc), _ptr(Tl), float(K[0]), float(K[1]), float(K[2]), float(K[3]), float(bf), float(mb),
           float(th), int(bMono), int(check_ori), _ptr(owner))
    return n, owner[:len(k)]


def ref_search_by_projection_kf(Cur, P, Tcw, K, th, orb_dist, check_ori):
    lib = _mlib()
    k = _a(Cur.mvKeysUn, KP_DTYPE); d = _a(Cur.mDescriptors, np.uint8); oc = _opt(Cur.occupied, np.uint8)
    sf = _a(Cur.mvScaleFactors, np.float32)
    wp, md, mx, mn, va = _points_args(P)
    ang = _a(P.angle, np.float32); T = _T12(Tcw)
    owner = np.full(max(len(k), 1), -1, np.int32)
    fn = lib.matchref_search_by_projection_kf
    fn.restype = C.c_int
    fn.argtypes = ([C.c_void_p] * 3 + [C.c_int] + [C.c_float] * 4 + [C.c_void_p, C.c_int, C.c_float] + [C.c_void_p] * 6 + [C.c_int]
                   + [C.c_void_p] + [C.c_float] * 5 + [C.c_int, C.c_int, C.c_void_p])
    n = fn(_ptr(k), _ptr(d), _p0(oc), len(k), *[float(b) for b in Cur.bounds], _ptr(sf), len(sf), _log_scale(Cur), _ptr(ang), _ptr(wp),
           _ptr(md), _ptr(mx), _ptr(mn), _ptr(va), len(wp), _ptr(T), float(K[0]), float(K[1]), float(K[2]), float(K[3]), float(th),
           int(orb_dist), int(check_ori), _ptr(owner))
    return n, owner[:len(k)]


def ref_search_by_projection_sim3(KF, P, Scw, K, th):
    lib = _mlib()
    k = _a(KF.mvKeysUn, KP_DTYPE); d = _a(KF.mDescriptors, np.uint8); oc = _opt(KF.occupied, np.uint8)
    sf = _a(KF.mvScaleFactors, np.float32)
    wp, md, mx, mn, va = _points_args(P)
    nr = _a(P.normal, np.float32); S = _T12(Scw)
    owner = np.full(max(len(k), 1), -1, np.int32)
    fn = lib.matchref_search_by_projection_sim3
    fn.restype = C.c_int
    fn.argtypes = ([C.c_void_p] * 3 + [C.c_int] + [C.c_float] * 4 + [C.c_void_p, C.c_int, C.c_float] + [C.c_void_p] * 6 + [C.c_int]
                   + [C.c_void_p] + [C.c_float] * 4 + [C.c_int, C.c_void_p])
    n = fn(_ptr(k), _ptr(d), _p0(oc), len(k), *[float(b) for b in KF.bounds], _ptr(sf), len(sf), _log_scale(KF), _ptr(wp), _ptr(md), _ptr(mx),
           _ptr(mn), _ptr(nr), _ptr(va), len(wp), _ptr(S), float(K[0]), float(K[1]), float(K[2]), float(K[3]), int(th), _ptr(owner))
    return n, owner[:len(k)]


def ref_search_by_bow(kf, F, nnratio, check_ori):
    lib = _mlib()
    k1, d1, hm1, nd1, st1, fi1 = _kf_args(kf)
    k2, d2, _, nd2, st2, fi2 = _kf_args(F)
    match = np.full(max(len(k2), 1), -1, np.int32)
    fn = lib.matchref_search_by_bow_kf_f
    fn.restype = C.c_int
    fn.argtypes = [C.c_void_p] * 3 + [C.c_int, C.c_int] + [C.c_void_p] * 3 + [C.c_void_p] * 2 + [C.c_int, C.c_int] + [C.c_void_p] * 3 + [C.c_float, C.c_int, C.c_void_p]
    n = fn(_ptr(k1), _ptr(d1), _ptr(hm1), len(k1), len(nd1), _ptr(nd1), _ptr(st1), _ptr(fi1), _ptr(k2), _ptr(d2), len(k2), len(nd2),
           _ptr(nd2), _ptr(st2), _ptr(fi2), float(np.float32(nnratio)), int(check_ori), _ptr(match))
    return n, match[:len(k2)]


def ref_search_by_bow_kf(kf1, kf2, nnratio, check_ori):
    lib = _mlib()
    k1, d1, hm1, nd1, st1, fi1 = _kf_args(kf1)
    k2, d2, hm2, nd2, st2, fi2 = _kf_args(kf2)
    match = np.full(max(len(k1), 1), -1, np.int32)
    fn = lib.matchref_search_by_bow_kf_kf
    fn.restype = C.c_int
    fn.argtypes = ([C.c_void_p] * 3 + [C.c_int, C.c_int] + [C.c_void_p] * 3) * 2 + [C.c_float, C.c_int, C.c_void_p]
    n = fn(_ptr(k1), _ptr(d1), _ptr(hm1), len(k1), len(nd1), _ptr(nd1), _ptr(st1), _ptr(fi1), _ptr(k2), _ptr(d2), _ptr(hm2), len(k2),
           len(nd2), _ptr(nd2), _ptr(st2), _ptr(fi2), float(np.float32(nnratio)), int(check_ori), _ptr(match))
    return n, match[:len(k1)]


def ref_search_for_triangulation(kf1, kf2, F12, Ow1, T2w, K2, only_stereo, check_ori):
    lib = _mlib()
    k1, d1, hm1, nd1, st1, fi1 = _kf_args(kf1)
    k2, d2, hm2, nd2, st2, fi2 = _kf_args(kf2)
    ur1 = _a(kf1.mvuRight, np.float32); ur2 = _a(kf2.mvuRight, np.float32)
    f = _f32(F12, 9); o = _f32(Ow1, 3); T = _T12(T2w)
    sf2 = _a(kf2.mvScaleFactors, np.float32); sg2 = _a(kf2.mvLevelSigma2, np.float32)
    pairs = np.zeros((max(len(k1), 1), 2), np.int32)
    fn = lib.matchref_search_for_triangulation
    fn.restype = C.c_int
    fn.argtypes = ([C.c_void_p] * 4 + [C.c_int, C.c_int] + [C.c_void_p] * 3) * 2 + [C.c_void_p] * 3 + [C.c_float] * 4 + [C.c_void_p] * 2 + [C.c_int] * 3 + [C.c_void_p]
    n = fn(_ptr(k1), _ptr(d1), _ptr(hm1), _ptr(ur1), len(k1), len(nd1), _ptr(nd1), _ptr(st1), _ptr(fi1), _ptr(k2), _ptr(d2), _ptr(hm2),
           _ptr(ur2), len(k2), len(nd2), _ptr(nd2), _ptr(st2), _ptr(fi2), _ptr(f), _ptr(o), _ptr(T), *[float(x) for x in K2], _ptr(sf2),
           _ptr(sg2), len(sf2), int(only_stereo), int(check_ori), _ptr(pairs))
    return pairs[:n].copy()


def ref_search_for_initialization(F1, F2, prev_matched, window, nnratio, check_ori):
    lib = _mlib()
    k1 = _a(F1.mvKeysUn, KP_DTYPE); d1 = _a(F1.mDescriptors, np.uint8)
    k2 = _a(F2.mvKeysUn, KP_DTYPE); d2 = _a(F2.mDescriptors, np.uint8)
    prev = np.ascontiguousarray(np.asarray(prev_matched, np.float32).reshape(-1, 2)).copy()
    m12 = np.full(max(len(k1), 1), -1, np.int32)
    fn = lib.matchref_search_for_initialization
    fn.restype = C.c_int
    fn.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int] + [C.c_float] * 4 + [C.c_void_p, C.c_int, C.c_float, C.c_int, C.c_void_p]
    n = fn(_ptr(k1), _ptr(d1), len(k1), _ptr(k2), _ptr(d2), len(k2), *[float(b) for b in F2.bounds], _ptr(prev), int(window),
           float(np.float32(nnratio)), int(check_ori), _ptr(m12))
    return n, m12[:len(k1)], prev


def ref_search_by_sim3(KF1, KF2, P1, P2, T1w, T2w, s12, R12, t12, K, th):
    lib = _mlib()
    k1 = _a(KF1.mvKeysUn, KP_DTYPE); d1 = _a(KF1.mDescriptors, np.uint8); sf1 = _a(KF1.mvScaleFactors, np.float32)
    k2 = _a(KF2.mvKeysUn, KP_DTYPE); d2 = _a(KF2.mDescriptors, np.uint8); sf2 = _a(KF2.mvScaleFactors, np.float32)
    b1 = _f32(KF1.bounds, 4); b2 = _f32(KF2.bounds, 4)
    wp1, md1, mx1, mn1, va1 = _points_args(P1)
    wp2, md2, mx2, mn2, va2 = _points_args(P2)
    Ta = _T12(T1w); Tb = _T12(T2w); r = _f32(R12, 9); t = _f32(t12, 3)
    match = np.full(max(len(k1), 1), -1, np.int32)
    fn = lib.matchref_search_by_sim3
    fn.restype = C.c_int
    fn.argtypes = ([C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_float] * 2 + [C.c_int] + [C.c_void_p] * 10 + [C.c_void_p] * 2
                   + [C.c_float, C.c_void_p, C.c_void_p] + [C.c_float] * 5 + [C.c_void_p])
    n = fn(_ptr(k1), _ptr(d1), len(k1), _ptr(b1), _ptr(sf1), _log_scale(KF1), _ptr(k2), _ptr(d2), len(k2), _ptr(b2), _ptr(sf2),
           _log_scale(KF2), len(sf1), _ptr(wp1), _ptr(md1), _ptr(mx1), _ptr(mn1), _ptr(va1), _ptr(wp2), _ptr(md2), _ptr(mx2), _ptr(mn2),
           _ptr(va2), _ptr(Ta), _ptr(Tb), float(np.float32(s12)), _ptr(r), _ptr(t), float(K[0]), float(K[1]), float(K[2]), float(K[3]),
           float(th), _ptr(match))
    return n, match[:len(k1)]


def ref_fuse(KF, P, Tcw_or_Scw, Ow, K, bf, th, scw):
    lib = _mlib()
    k = _a(KF.mvKeysUn, KP_DTYPE); d = _a(KF.mDescriptors, np.uint8); sf = _a(KF.mvScaleFactors, np.float32)
    ur = _opt(KF.mvuRight, np.float32); inv = _opt(KF.mvInvLevelSigma2, np.float32)
    wp, md, mx, mn, va = _points_args(P)
    nr = _a(P.normal, np.float32); T = _T12(Tcw_or_Scw); ow = _f32(Ow, 3)
    best = np.full(max(len(wp), 1), -1, np.int32)
    fn = lib.matchref_fuse
    fn.restype = C.c_int
    fn.argtypes = ([C.c_void_p] * 4 + [C.c_int] + [C.c_float] * 4 + [C.c_void_p, C.c_int, C.c_float] + [C.c_void_p] * 6 + [C.c_int]
                   + [C.c_void_p] * 2 + [C.c_float] * 6 + [C.c_int, C.c_void_p])
    n = fn(_ptr(k), _ptr(d), _p0(ur), _p0(inv), len(k), *[float(b) for b in KF.bounds], _ptr(sf), len(sf), _log_scale(KF), _ptr(wp),
           _ptr(md), _ptr(mx), _ptr(mn), _ptr(nr), _ptr(va), len(wp), _ptr(T), _ptr(ow), float(K[0]), float(K[1]), float(K[2]), float(K[3]),
           float(bf), float(th), int(scw), _ptr(best))
    return n, best[:len(wp)]


# ---------------------------------------------------------------------------------------------------------------------
# The reference's own src/Frame.cc compiled verbatim against its real include/Frame.h (oracle/_ref/libframeref.so,
# oracle/frameref_wrap.cpp): ComputeStereoMatches, the feature grid, isInFrustum.
FRAMEREF_SO = os.path.join(HERE, "_ref", "libframeref.so")


def have_frameref() -> bool:
    return os.path.exists(FRAMEREF_SO)


def ref_stereo(kL, dL, kR, dR, pyrL, pyrR, scale, inv_scale, bf, fx):
    """Frame::ComputeStereoMatches of the reference source; same arguments and outputs as port_stereo (without the SAD)."""
    lib = C.CDLL(FRAMEREF_SO)
    nlev = len(pyrL)
    pyrL = [np.ascontiguousarray(p, np.uint8) for p in pyrL]
    pyrR = [np.ascontiguousarray(p, np.uint8) for p in pyrR]
    lw = np.array([p.shape[1] for p in pyrL], np.int32)
    lh = np.array([p.shape[0] for p in pyrL], np.int32)
    PL = (C.c_void_p * nlev)(*[p.ctypes.data for p in pyrL])
    PR = (C.c_void_p * nlev)(*[p.ctypes.data for p in pyrR])
    kL = np.ascontiguousarray(kL); kR = np.ascontiguousarray(kR)
    dL = np.ascontiguousarray(dL, np.uint8); dR = np.ascontiguousarray(dR, np.uint8)
    n = len(kL)
    ur = np.zeros(max(n, 1), np.float32); dp = np.zeros(max(n, 1), np.float32)
    scale = np.ascontiguousarray(scale, np.float32); inv_scale = np.ascontiguousarray(inv_scale, np.float32)
    b = np.float32(bf) / np.float32(fx)
    lib.frameref_stereo.restype = C.c_int
    lib.frameref_stereo.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_float, C.c_float, C.c_void_p, C.c_void_p]
    lib.frameref_stereo(kL.ctypes.data, dL.ctypes.data, n, kR.ctypes.data, dR.ctypes.data, len(kR), PL, PR, lw.ctypes.data, lh.ctypes.data,
                        nlev, scale.ctypes.data, inv_scale.ctypes.data, float(bf), float(b), ur.ctypes.data, dp.ctypes.data)
    return ur[:n], dp[:n]


def ref_features_in_area(keys, bounds, x, y, r, min_level, max_level):
    lib = C.CDLL(FRAMEREF_SO)
    keys = _a(keys, KP_DTYPE)
    out = np.zeros(max(len(keys), 1), np.int32)
    lib.frameref_features_in_area.restype = C.c_int
    lib.frameref_features_in_area.argtypes = [C.c_void_p, C.c_int] + [C.c_float] * 7 + [C.c_int, C.c_int, C.c_void_p, C.c_int]
    n = lib.frameref_features_in_area(_ptr(keys), len(keys), *[float(b) for b in bounds], float(x), float(y), float(r), min_level,
                                      max_level, _ptr(out), len(out))
    return out[:n]


def ref_is_in_frustum(F, P, Tcw, K, mbf, viewing_cos_limit=0.5):
    """Frame::isInFrustum of the reference source; returns the same dict as port_is_in_frustum plus 'Ow' (mOw from SetPose)."""
    lib = C.CDLL(FRAMEREF_SO)
    wp, md, mx, mn, va = _points_args(P)
    nr = _a(P.normal, np.float32)
    T = _a(np.asarray(Tcw, np.float32)[:3, :4].reshape(12), np.float32)
    n = len(wp)
    inv = np.zeros(max(n, 1), np.uint8); px = np.zeros(max(n, 1), np.float32); py = np.zeros(max(n, 1), np.float32)
    pxr = np.zeros(max(n, 1), np.float32); lv = np.zeros(max(n, 1), np.int32); vc = np.zeros(max(n, 1), np.float32)
    ow = np.zeros(3, np.float32)
    fn = lib.frameref_is_in_frustum
    fn.restype = C.c_int
    fn.argtypes = [C.c_void_p] * 5 + [C.c_int, C.c_void_p] + [C.c_float] * 11 + [C.c_int] + [C.c_void_p] * 7
    cnt = fn(_ptr(wp), _ptr(nr), _ptr(mx), _ptr(mn), _ptr(va), n, _ptr(T), float(K[0]), float(K[1]), float(K[2]), float(K[3]), float(mbf),
             *[float(b) for b in F.bounds], float(viewing_cos_limit), _log_scale(F), len(F.mvScaleFactors), _ptr(inv), _ptr(px), _ptr(py),
             _ptr(pxr), _ptr(lv), _ptr(vc), _ptr(ow))
    return dict(count=cnt, in_view=inv[:n], proj_x=px[:n], proj_y=py[:n], proj_xr=pxr[:n], level=lv[:n], view_cos=vc[:n], Ow=ow)


# ---------------------------------------------------------------------------------------------------------------------
# The reference's DBoW2 and src/KeyFrameDatabase.cc compiled verbatim (oracle/_ref/libdbowref.so, oracle/dbowref_wrap.cpp).
DBOWREF_SO = os.path.join(HERE, "_ref", "libdbowref.so")


def have_dbowref() -> bool:
    return os.path.exists(DBOWREF_SO)


class RefVocabulary:
    """ORBVocabulary of the reference (DBoW2::TemplatedVocabulary<FORB::TDescriptor, FORB>), loaded with its own loadFromTextFile."""

    def __init__(self, text_path):
        self._lib = C.CDLL(DBOWREF_SO)
        self._lib.dbowref_voc_load_text.restype = C.c_void_p
        self._lib.dbowref_voc_load_text.argtypes = [C.c_char_p]
        self._h = self._lib.dbowref_voc_load_text(str(text_path).encode())
        if not self._h:
            raise RuntimeError("loadFromTextFile failed")
        self._lib.dbowref_voc_words.argtypes = [C.c_void_p]
        self.words = self._lib.dbowref_voc_words(self._h)

    def __del__(self):
        if getattr(self, "_h", None):
            self._lib.dbowref_voc_destroy.argtypes = [C.c_void_p]
            self._lib.dbowref_voc_destroy(self._h)
            self._h = None

    def transform(self, desc, levelsup):
        """-> (bow {word: value}, fv_node, fv_start, fv_idx)"""
        d = _a(desc, np.uint8)
        n = len(d)
        bw = np.zeros(max(n, 1), np.uint32); bv = np.zeros(max(n, 1), np.float64); nb = C.c_int(0)
        fn_ = np.zeros(max(n, 1), np.uint32); fs = np.zeros(max(n, 1) + 1, np.int32); fi = np.zeros(max(n, 1), np.uint32); nn = C.c_int(0)
        f = self._lib.dbowref_transform
        f.restype = C.c_int
        f.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int] + [C.c_void_p] * 7
        f(self._h, _ptr(d), n, int(levelsup), _ptr(bw), _ptr(bv), C.addressof(nb), _ptr(fn_), _ptr(fs), _ptr(fi), C.addressof(nn))
        k, a = nb.value, nn.value
        return dict(zip(bw[:k].tolist(), bv[:k].tolist())), fn_[:a].copy(), fs[:a + 1].copy(), fi[:fs[a]].copy()

    def score(self, bow1, bow2):
        w1 = _a(np.fromiter(bow1.keys(), np.uint32, len(bow1)), np.uint32); v1 = _a(np.fromiter(bow1.values(), np.float64, len(bow1)), np.float64)
        w2 = _a(np.fromiter(bow2.keys(), np.uint32, len(bow2)), np.uint32); v2 = _a(np.fromiter(bow2.values(), np.float64, len(bow2)), np.float64)
        f = self._lib.dbowref_score
        f.restype = C.c_double
        f.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
        return float(f(self._h, _ptr(w1) if len(w1) else None, _ptr(v1) if len(v1) else None, len(w1), _ptr(w2) if len(w2) else None,
                       _ptr(v2) if len(v2) else None, len(w2)))

    def detect_candidates(self, loop, kf_bows, q_bow, connected, neigh, min_score=0.0):
        start = np.zeros(len(kf_bows) + 1, np.int32)
        start[1:] = np.cumsum([len(b) for b in kf_bows])
        kw = _a(np.concatenate([np.fromiter(b.keys(), np.uint32, len(b)) for b in kf_bows] + [np.zeros(0, np.uint32)]), np.uint32)
        kv = _a(np.concatenate([np.fromiter(b.values(), np.float64, len(b)) for b in kf_bows] + [np.zeros(0, np.float64)]), np.float64)
        qw = _a(np.fromiter(q_bow.keys(), np.uint32, len(q_bow)), np.uint32); qv = _a(np.fromiter(q_bow.values(), np.float64, len(q_bow)), np.float64)
        ng = _a(np.asarray(neigh, np.int32).reshape(len(kf_bows), 10), np.int32)
        cn = _a(np.asarray(connected if connected is not None else np.zeros(len(kf_bows)), np.uint8), np.uint8)
        out = np.zeros(max(len(kf_bows), 1), np.int32)
        f = self._lib.dbowref_detect_candidates
        f.restype = C.c_int
        f.argtypes = [C.c_void_p, C.c_int, C.c_int] + [C.c_void_p] * 5 + [C.c_int, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p]
        n = f(self._h, int(loop), len(kf_bows), _ptr(start), _ptr(kw), _ptr(kv), _ptr(qw) if len(qw) else None, _ptr(qv) if len(qv) else None,
              len(qw), _ptr(cn), _ptr(ng), float(np.float32(min_score)), _ptr(out))
        return out[:n].tolist()

    def reloc_sequence(self, kf_bows, q_bows, neigh):
        """DetectRelocalizationCandidates for every query of `q_bows` IN SEQUENCE on one database (KeyFrame::mRelocScore persists)."""
        start = np.zeros(len(kf_bows) + 1, np.int32)
        start[1:] = np.cumsum([len(b) for b in kf_bows])
        kw = _a(np.concatenate([np.fromiter(b.keys(), np.uint32, len(b)) for b in kf_bows] + [np.zeros(0, np.uint32)]), np.uint32)
        kv = _a(np.concatenate([np.fromiter(b.values(), np.float64, len(b)) for b in kf_bows] + [np.zeros(0, np.float64)]), np.float64)
        qs = np.zeros(len(q_bows) + 1, np.int32)
        qs[1:] = np.cumsum([len(b) for b in q_bows])
        qw = _a(np.concatenate([np.fromiter(b.keys(), np.uint32, len(b)) for b in q_bows] + [np.zeros(1, np.uint32)]), np.uint32)
        qv = _a(np.concatenate([np.fromiter(b.values(), np.float64, len(b)) for b in q_bows] + [np.zeros(1, np.float64)]), np.float64)
        ng = _a(np.asarray(neigh, np.int32).reshape(len(kf_bows), 10), np.int32)
        stride = max(len(kf_bows), 1)
        out = np.zeros((len(q_bows), stride), np.int32); out_n = np.zeros(len(q_bows), np.int32)
        f = self._lib.dbowref_reloc_sequence
        f.restype = C.c_int
        f.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 3 + [C.c_int] + [C.c_void_p] * 5 + [C.c_int, C.c_void_p]
        f(self._h, len(kf_bows), _ptr(start), _ptr(kw), _ptr(kv), len(q_bows), _ptr(qs), _ptr(qw), _ptr(qv), _ptr(ng), _ptr(out), stride, _ptr(out_n))
        return [out[i, :out_n[i]].tolist() for i in range(len(q_bows))]


# ---------------------------------------------------------------------------------------------------------------------
# The reference's src/MapPoint.cc compiled verbatim against its real include/MapPoint.h (oracle/_ref/libmapref.so).
MAPREF_SO = os.path.join(HERE, "_ref", "libmapref.so")


def have_mapref() -> bool:
    return os.path.exists(MAPREF_SO)


def ref_predict_scale(max_distance, dist, log_scale, n_levels, use_frame=False):
    lib = C.CDLL(MAPREF_SO)
    mx = _a(max_distance, np.float32); ds = _a(dist, np.float32)
    out = np.zeros(max(len(mx), 1), np.int32)
    lib.mapref_predict_scale.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_int, C.c_int, C.c_void_p]
    lib.mapref_predict_scale(_ptr(mx), _ptr(ds), len(mx), float(np.float32(log_scale)), int(n_levels), int(use_frame), _ptr(out))
    return out[:len(mx)]


def port_predict_scale(max_distance, dist, log_scale, n_levels):
    lib = _plib()
    mx = _a(max_distance, np.float32); ds = _a(dist, np.float32)
    out = np.zeros(max(len(mx), 1), np.int32)
    lib.orbport_predict_scale.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_int, C.c_void_p]
    lib.orbport_predict_scale(_ptr(mx), _ptr(ds), len(mx), float(np.float32(log_scale)), int(n_levels), _ptr(out))
    return out[:len(mx)]


def ref_distance_invariance(max_distance, min_distance):
    lib = C.CDLL(MAPREF_SO)
    mx = _a(max_distance, np.float32); mn = _a(min_distance, np.float32)
    omx = np.zeros(max(len(mx), 1), np.float32); omn = np.zeros(max(len(mx), 1), np.float32)
    lib.mapref_distance_invariance.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    lib.mapref_distance_invariance(_ptr(mx), _ptr(mn), len(mx), _ptr(omx), _ptr(omn))
    return omx[:len(mx)], omn[:len(mx)]


def ref_distinctive_descriptor(desc, bad=None):
    """MapPoint::ComputeDistinctiveDescriptors of the reference source -> the chosen 32-byte descriptor (None if none)."""
    lib = C.CDLL(MAPREF_SO)
    d = _a(np.asarray(desc, np.uint8).reshape(-1, 32), np.uint8)
    b = _a(bad, np.uint8) if bad is not None else None
    out = np.zeros(32, np.uint8)
    lib.mapref_distinctive_descriptor.restype = C.c_int
    lib.mapref_distinctive_descriptor.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    ok = lib.mapref_distinctive_descriptor(_ptr(d) if len(d) else None, _ptr(b) if b is not None else None, len(d), _ptr(out))
    return out if ok else None


# ---------------------------------------------------------------------------------------------------------------------
# RGB-D leg of the Frame constructor (src/Frame.cc:119-178): UndistortKeyPoints, ComputeStereoFromRGBD, ComputeImageBounds.
def _rgbd_call(fn, keys, K4, dist, bf, depth):
    keys = _a(keys, KP_DTYPE)
    n = len(keys)
    K4 = _a(K4, np.float32); dist = _a(dist, np.float32); depth = _a(depth, np.float32)
    h, w = depth.shape
    ku = np.zeros(max(n, 1), KP_DTYPE); ur = np.zeros(max(n, 1), np.float32); dp = np.zeros(max(n, 1), np.float32); b4 = np.zeros(4, np.float32)
    return keys, n, K4, dist, depth, w, h, ku, ur, dp, b4


def ref_rgbd_frame(keys, K4, dist, bf, depth):
    """The reference's own UndistortKeyPoints + ComputeStereoFromRGBD + ComputeImageBounds (libframeref.so)."""
    lib = C.CDLL(FRAMEREF_SO)
    keys, n, K4, dist, depth, w, h, ku, ur, dp, b4 = _rgbd_call(None, keys, K4, dist, bf, depth)
    lib.frameref_rgbd.restype = C.c_int
    lib.frameref_rgbd.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_void_p, C.c_int, C.c_int] + [C.c_void_p] * 4
    cnt = lib.frameref_rgbd(_ptr(keys), n, _ptr(K4), _ptr(dist), len(dist), float(bf), _ptr(depth), w, h, _ptr(ku), _ptr(ur), _ptr(dp), _ptr(b4))
    return dict(keys_un=ku[:n], u_right=ur[:n], depth=dp[:n], bounds=b4, count=cnt)


def port_rgbd_frame(keys, K4, dist, bf, depth):
    """Restatement (oracle/orb_port_frame.cpp); same outputs as ref_rgbd_frame."""
    lib = _plib()
    keys, n, K4, dist, depth, w, h, ku, ur, dp, b4 = _rgbd_call(None, keys, K4, dist, bf, depth)
    lib.orbport_undistort_keypoints.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    lib.orbport_undistort_keypoints.restype = None
    lib.orbport_image_bounds.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    lib.orbport_image_bounds.restype = None
    lib.orbport_stereo_from_rgbd.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_void_p]
    lib.orbport_stereo_from_rgbd.restype = C.c_int
    lib.orbport_undistort_keypoints(_ptr(keys), n, _ptr(K4), _ptr(dist), len(dist), _ptr(ku))
    lib.orbport_image_bounds(w, h, _ptr(K4), _ptr(dist), len(dist), _ptr(b4))
    cnt = lib.orbport_stereo_from_rgbd(_ptr(keys), _ptr(ku), n, _ptr(depth), w, h, float(bf), _ptr(ur), _ptr(dp))
    return dict(keys_un=ku[:n], u_right=ur[:n], depth=dp[:n], bounds=b4, count=cnt)


def port_depth_to_float(raw, factor):
    lib = _plib()
    raw = _a(raw, np.uint16)
    out = np.zeros(raw.shape, np.float32)
    lib.orbport_depth_to_float.argtypes = [C.c_void_p, C.c_int, C.c_float, C.c_void_p]
    lib.orbport_depth_to_float.restype = None
    lib.orbport_depth_to_float(_ptr(raw), raw.size, float(np.float32(factor)), _ptr(out))
    return out


# ---------------------------------------------------------------------------------------------------------------------
# Batch helpers for bench.py's CPU arms (BASELINE configs[4]): keyframes built once, the timed sweep is the reference's loop.
def port_compute_bow(voc: "PortVocabulary", desc, levelsup=4):
    """(words[uint32], values[float64], FeatureVector CSR (node, start, idx)) — TemplatedVocabulary::transform with std::map bookkeeping."""
    lib = _plib()
    d = _a(desc, np.uint8)
    n = len(d)
    bw = np.zeros(max(n, 1), np.uint32); bv = np.zeros(max(n, 1), np.float64)
    fn_ = np.zeros(max(n, 1), np.uint32); fs = np.zeros(n + 1, np.int32); fi = np.zeros(max(n, 1), np.uint32)
    nb, nn = C.c_int32(0), C.c_int32(0)
    lib.orbport_compute_bow.restype = None
    lib.orbport_compute_bow.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int] + [C.c_void_p] * 7
    lib.orbport_compute_bow(voc._h, _ptr(d), n, levelsup, _ptr(bw), _ptr(bv), C.addressof(nb), _ptr(fn_), _ptr(fs), _ptr(fi), C.addressof(nn))
    return bw[:nb.value].copy(), bv[:nb.value].copy(), (fn_[:nn.value].copy(), fs[:nn.value + 1].copy(), fi[:fs[nn.value]].copy())


class PortScoreSweep:
    """KeyFrameDatabase scoring loop (src/KeyFrameDatabase.cc:127,:240) over many keyframes in one C call."""

    def __init__(self, kf_bows):
        self.lib = _plib()
        self.off = np.zeros(len(kf_bows) + 1, np.int32)
        self.off[1:] = np.cumsum([len(w) for w, _ in kf_bows])
        self.w = _a(np.concatenate([w for w, _ in kf_bows]) if kf_bows else np.zeros(0), np.uint32)
        self.v = _a(np.concatenate([v for _, v in kf_bows]) if kf_bows else np.zeros(0), np.float64)
        self.n = len(kf_bows)
        self.score = np.zeros(max(self.n, 1), np.float32); self.common = np.zeros(max(self.n, 1), np.int32)
        self.lib.orbport_bow_score_sweep.restype = None
        self.lib.orbport_bow_score_sweep.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]

    def __call__(self, qw, qv):
        qw = _a(qw, np.uint32); qv = _a(qv, np.float64)
        self.lib.orbport_bow_score_sweep(_ptr(qw), _ptr(qv), len(qw), _ptr(self.w), _ptr(self.v), _ptr(self.off), self.n, _ptr(self.score), _ptr(self.common))
        return self.score[:self.n], self.common[:self.n]


class RefBowSweep:
    """The reference's ORBmatcher::SearchByBoW(pKF, F, vpMapPointMatches) (src/ORBmatcher.cc:159-288, compiled verbatim) for one
    frame against many keyframes that are built once — what relocalisation / loop closing does with KeyFrames it already holds."""

    def __init__(self, kfs):
        self.lib = _mlib()
        L = self.lib
        L.matchref_kf_create.restype = C.c_void_p
        L.matchref_kf_create.argtypes = [C.c_void_p] * 3 + [C.c_int, C.c_int] + [C.c_void_p] * 3
        L.matchref_kf_destroy.argtypes = [C.c_void_p]
        L.matchref_frame_create.restype = C.c_void_p
        L.matchref_frame_create.argtypes = [C.c_void_p] * 2 + [C.c_int, C.c_int] + [C.c_void_p] * 3
        L.matchref_frame_destroy.argtypes = [C.c_void_p]
        L.matchref_search_by_bow_sweep.restype = C.c_int
        L.matchref_search_by_bow_sweep.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_float, C.c_int, C.c_void_p, C.c_void_p]
        self.h = []
        for kf in kfs:
            k, d, hm, nd, st, fi = _kf_args(kf)
            self.h.append(L.matchref_kf_create(_ptr(k), _ptr(d), _ptr(hm), len(k), len(nd), _ptr(nd), _ptr(st), _ptr(fi)))
        self.arr = (C.c_void_p * max(len(self.h), 1))(*self.h)
        self.nm = np.zeros(max(len(self.h), 1), np.int32)

    def frame(self, F):
        k, d, _, nd, st, fi = _kf_args(F)
        return self.lib.matchref_frame_create(_ptr(k), _ptr(d), len(k), len(nd), _ptr(nd), _ptr(st), _ptr(fi)), len(k)

    def free_frame(self, fh):
        self.lib.matchref_frame_destroy(fh[0])

    def sweep(self, fh, nnratio, check_ori, want_matches=False):
        match = np.full((len(self.h), max(fh[1], 1)), -1, np.int32) if want_matches else None
        self.lib.matchref_search_by_bow_sweep(self.arr, len(self.h), fh[0], float(np.float32(nnratio)), int(check_ori), _ptr(self.nm),
                                              _ptr(match) if want_matches else None)
        return self.nm[:len(self.h)].copy(), (match[:, :fh[1]] if want_matches else None)

    def __del__(self):
        try:
            for h in self.h:
                self.lib.matchref_kf_destroy(h)
        except Exception:
            pass
