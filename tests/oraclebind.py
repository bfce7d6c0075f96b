"""ctypes bindings for the plain-C oracle (oracle/liblsd_oracle.so) — test infrastructure."""
import ctypes as C
import os
import subprocess
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "oracle", "liblsd_oracle.so")
LSD_PARAMS = dict(sca=0.3, sig=0.6, angThre=22.5, denThre=0.7, pseBin=1024)
STAT_FIELDS = ["cells", "live_seeds", "grows", "grown_px", "small", "regrows", "rrr_passes", "nfa_calls",
               "nfa_px", "rejects", "accepts"]


class Stats(C.Structure):
    _fields_ = [(f, C.c_longlong) for f in STAT_FIELDS]


_lib = None


def build():
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "oracle"])


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(SO):
            build()
        L = C.CDLL(SO)
        L.lsdo_lsd.restype = C.c_int
        L.lsdo_lsd.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, C.c_double, C.c_int,
                               C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                               C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        L.lsdo_gauss_taps.restype = C.c_int
        L.lsdo_gauss_taps.argtypes = [C.c_double, C.c_double, C.c_void_p, C.c_int]
        L.lsdo_map_cache.restype = None
        L.lsdo_map_cache.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_void_p]
        L.lsdo_fa_scores.restype = C.c_int
        L.lsdo_fa_scores.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p,
                                     C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        L.lsdo_fa_legacy.restype = C.c_int
        L.lsdo_fa_legacy.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_double, C.c_double, C.c_double, C.c_void_p, C.c_int, C.c_int,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        L.lsdo_feature_scan.restype = C.c_int
        L.lsdo_feature_scan.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_double, C.c_void_p,
                                        C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
        _lib = L
    return _lib


def feature_scan(map_param, ranges, angles, least_point=3, thre_line=0.08, least_dist_m=0.5):
    """myrdp::FeatureScan restated (oracle/rdp_oracle.c); same dict as refbind.ref_feature_scan."""
    mp = np.asarray(map_param, np.float64)
    r = np.ascontiguousarray(ranges, np.float64); a = np.ascontiguousarray(angles, np.float64)
    lines = np.zeros((max(2 * len(r) + 2, 1), 10)); pts = np.zeros((400000, 2)); npts = C.c_int(0)
    lidar = np.zeros(2); imsz = np.zeros(2, np.int32)
    cap = 4096 * 4096
    im = np.zeros(cap, np.uint8)
    n = lib().lsdo_feature_scan(_p(mp), _p(r), _p(a), len(r), least_point, thre_line, least_dist_m, _p(lines), len(lines), _p(pts),
                                len(pts), C.byref(npts), _p(lidar), _p(imsz), _p(im), cap)
    w, h = int(imsz[0]), int(imsz[1])
    return dict(lines=lines[:n].copy(), pts=pts[:npts.value].copy(), lidar_pos=lidar, size=(w, h),
                line_im=im[:max(w, 0) * max(h, 0)].reshape(max(h, 0), max(w, 0)).copy())


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def lsd(map_u8, want_maps=True, want_line_im=True, max_lines=65536, **kw):
    p = dict(LSD_PARAMS); p.update(kw)
    m = np.ascontiguousarray(map_u8, dtype=np.uint8)
    rows, cols = m.shape
    W, H = int(np.floor(cols * p["sca"])), int(np.floor(rows * p["sca"]))
    out = {}
    if want_maps:
        out.update(map_out=np.zeros((rows, cols), np.uint8), gauss=np.zeros((H, W)), mag=np.zeros((H, W)),
                   deg=np.zeros((H, W)), used=np.zeros((H, W), np.uint8), labels=np.zeros((H, W), np.int32),
                   seeds=np.zeros((H * W, 3), np.int32))
    if want_line_im:
        out["line_im"] = np.zeros((rows, cols), np.uint8)
    rects = np.zeros((max_lines, 13)); lines = np.zeros((max_lines, 10))
    ns = C.c_int(0); st = Stats()
    g = out.get
    n = lib().lsdo_lsd(_p(m), cols, rows, p["sca"], p["sig"], p["angThre"], p["denThre"], p["pseBin"],
                       _p(g("map_out")), _p(g("gauss")), _p(g("mag")), _p(g("deg")), _p(g("used")), _p(g("labels")),
                       _p(g("seeds")), H * W if want_maps else 0, C.byref(ns), _p(rects), _p(lines), max_lines,
                       _p(g("line_im")), C.byref(st))
    if want_maps:
        out["seeds"] = out["seeds"][:ns.value].copy()
    out["n"] = n
    out["rects"] = rects[:n].copy(); out["lines"] = lines[:n].copy()
    out["stats"] = {f: getattr(st, f) for f in STAT_FIELDS}
    return out


def lsd_regrow_tols(map_u8, cap=1 << 20, **kw):
    """lsd() with the oracle's re-grow tap on: adds regrow_tols, the tolerance of every Refiner re-grow (:857) in call order"""
    L = lib()
    L.lsdo_set_regrow_tol_log.argtypes = [C.c_void_p, C.c_int]
    L.lsdo_regrow_tol_count.restype = C.c_int
    tols = np.zeros(cap)
    L.lsdo_set_regrow_tol_log(_p(tols), cap)
    try:
        out = lsd(map_u8, **kw)
        n = L.lsdo_regrow_tol_count()
    finally:
        L.lsdo_set_regrow_tol_log(None, 0)
    assert n < cap, "re-grow tap full"
    out["regrow_tols"] = tols[:n].copy()
    return out


def lsd_nfa_calls(map_u8, cap=1 << 20, **kw):
    """lsd() with the oracle's NFA tap on: adds nfa_calls, one row (allPix, aliPix, p, logNT, result) per RectangleNFACalculator
    call in call order"""
    L = lib()
    L.lsdo_set_nfa_log.argtypes = [C.c_void_p, C.c_int]
    L.lsdo_nfa_log_count.restype = C.c_int
    buf = np.zeros((cap, 5))
    L.lsdo_set_nfa_log(_p(buf), cap)
    try:
        out = lsd(map_u8, **kw)
        n = L.lsdo_nfa_log_count()
    finally:
        L.lsdo_set_nfa_log(None, 0)
    assert n < cap, "NFA tap full"
    out["nfa_calls"] = buf[:n].copy()
    return out


def nfa_tail(all_pix, ali_pix, p, logNT, few=0.0, near=0.0, margin=0.0):
    """lsdo_nfa_tail over arrays of tuples: (result, exit index, probe [n][5]); the probe counts each tail's break tests, those
    at m == 1, those at 0 < |1 - m| <= few, those inside (near, margin) of the device's fast break test, and those inside the
    margin without its |m^n| / |1 - m| term (lsd_oracle.h)"""
    L = lib()
    L.lsdo_nfa_tail_many.restype = None
    L.lsdo_nfa_tail_many.argtypes = [C.c_int] + [C.c_void_p] * 4 + [C.c_double] * 3 + [C.c_void_p] * 3
    a = np.ascontiguousarray(all_pix, np.int32); b = np.ascontiguousarray(ali_pix, np.int32)
    pp = np.ascontiguousarray(p, np.float64); ln = np.ascontiguousarray(logNT, np.float64)
    n = len(a)
    out = np.zeros(n); ex = np.zeros(n, np.int32); probe = np.zeros((n, 5), np.int32)
    L.lsdo_nfa_tail_many(n, _p(a), _p(b), _p(pp), _p(ln), few, near, margin, _p(out), _p(ex), _p(probe))
    return out, ex, probe


def log_gamma(xs):
    L = lib()
    L.lsdo_log_gamma.restype = C.c_double
    L.lsdo_log_gamma.argtypes = [C.c_int]
    return np.array([L.lsdo_log_gamma(int(x)) for x in xs])


def gauss_taps(sca=0.3, sig=0.6):
    buf = np.zeros(3 * 64)
    h = lib().lsdo_gauss_taps(sca, sig, _p(buf), len(buf))
    return h, buf[:3 * (2 * h + 1)].reshape(3, 2 * h + 1).copy()


def map_cache(map_u8, res):
    m = np.ascontiguousarray(map_u8, dtype=np.uint8)
    rows, cols = m.shape
    out = np.zeros((rows, cols))
    lib().lsdo_map_cache(_p(m), cols, rows, float(res), _p(out))
    return out


def fa_scores(scan_lines, map_lines, pts, mc, lidar_pose, last_pose):
    sl = np.ascontiguousarray(scan_lines, np.float64).reshape(-1, 10)
    ml = np.ascontiguousarray(map_lines, np.float64).reshape(-1, 10)
    pt = np.ascontiguousarray(pts, np.float64).reshape(-1, 2)
    mc = np.ascontiguousarray(mc, np.float64)
    rows, cols = mc.shape
    lp = np.asarray(lidar_pose, np.float64); la = np.asarray(last_pose, np.float64)
    cap = max(4 * len(sl) * len(ml), 4)
    idx = np.zeros((cap, 3), np.int32); val = np.zeros((cap, 4))
    n = lib().lsdo_fa_scores(_p(sl), len(sl), _p(ml), len(ml), _p(pt), len(pt), _p(mc), cols, rows, _p(lp), _p(la),
                             _p(idx), _p(val), cap)
    return idx[:n].copy(), val[:n].copy()


def fa_legacy(scan_lines, map_lines, resol, ori, lidar_pos, mc, ranges, angles, fn=None):
    """the catkin snapshot's FeatureAssociation restated (oracle/fa_legacy_oracle.c): (pose_all (T,15), est (3,), est_real (3,)).
    fn = a ros_fa entry point of oracle/_ref/libref_rosfa*.so instead of the restatement (same arguments, 15 x T matrix out)."""
    sl = np.ascontiguousarray(scan_lines, np.float64).reshape(-1, 10)
    ml = np.ascontiguousarray(map_lines, np.float64).reshape(-1, 10)
    mc = np.ascontiguousarray(mc, np.float64)
    rows, cols = mc.shape
    r = np.ascontiguousarray(ranges, np.float64); a = np.ascontiguousarray(angles, np.float64)
    lp = np.ascontiguousarray(lidar_pos, np.int32)
    cap = 4 * len(sl) * len(ml) + 4
    out = np.zeros((cap, 15)) if fn is None else np.zeros((15, cap))
    est = np.zeros(3); real = np.zeros(3)
    f = lib().lsdo_fa_legacy if fn is None else fn
    T = f(_p(sl), len(sl), _p(ml), len(ml), C.c_double(resol), C.c_double(ori[0]), C.c_double(ori[1]), _p(lp), cols, rows, _p(mc), _p(r), _p(a),
          len(r), _p(out), cap, _p(est), _p(real))
    return (out[:T].copy() if fn is None else out[:, :T].T.copy()), est, real


def feature_scan_many(map_param, frames):
    mp = np.asarray(map_param, np.float64)
    boff = np.zeros(len(frames) + 1, np.int32)
    boff[1:] = np.cumsum([len(r) for r, _ in frames])
    r = np.ascontiguousarray(np.concatenate([f[0] for f in frames]), np.float64)
    a = np.ascontiguousarray(np.concatenate([f[1] for f in frames]), np.float64)
    L = lib()
    L.lsdo_feature_scan_many.restype = C.c_longlong
    L.lsdo_feature_scan_many.argtypes = [C.c_void_p] * 4 + [C.c_int, C.c_void_p]
    npts = C.c_longlong(0)
    nl = L.lsdo_feature_scan_many(_p(mp), _p(r), _p(a), _p(boff), len(frames), C.byref(npts))
    return int(nl), int(npts.value)
