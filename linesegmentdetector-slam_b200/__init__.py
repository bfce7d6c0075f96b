"""Python (ctypes) face of liblsdb200.so — the B200-native LSD / association hot path.

The product is the C-ABI library declared in include/lsdb200.h; this module only marshals numpy
buffers into it for tests, bench.py and smoke().  There is no CPU fallback: importing works
anywhere, but creating a Context without the built library or without an sm_100 GPU raises.

Load it by path (the directory name is not a Python identifier):
    from __graft_entry__ import load_package; lsdb = load_package()
"""
import ctypes as C
import os
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(HERE, "liblsdb200.so")
LSD_DEFAULTS = dict(sca=0.3, sig=0.6, angThre=22.5, denThre=0.7, pseBin=1024)  # LSD/baseFunc.h:64-68
ERR_NAMES = {1: "CUDA", 2: "ARG", 3: "CAPACITY", 4: "TIMEOUT", 5: "NO_DEVICE"}
STAGES = ("stencil", "order", "grow")
STAT_FIELDS = ["cells", "live_seeds", "grows", "grown_px", "small", "regrows", "rrr_passes", "nfa_calls", "nfa_px",
               "rejects", "accepts", "spec_evals", "respec_evals", "chunks", "cyc_grow", "cyc_rect", "cyc_nfa", "cyc_wait",
               "cyc_retire", "cyc_spec", "cyc_respec", "cyc_map", "ns_map", "spare_", "rs_none", "rs_conflict", "rs_commit", "rs_lost_commit", "rs_pad0", "rs_pad1", "rs_pad2", "rs_pad3"]

LINE_DTYPE = np.dtype([("k", "f8"), ("b", "f8"), ("dx", "f8"), ("dy", "f8"), ("x1", "f8"), ("y1", "f8"), ("x2", "f8"),
                       ("y2", "f8"), ("len", "f8"), ("orient", "i4"), ("_pad", "i4")])
RECT_FIELDS = ["x1", "y1", "x2", "y2", "wid", "cX", "cY", "deg", "dx", "dy", "p", "prec", "logNFA"]
EST_DTYPE = np.dtype([("n_hyp", "i4"), ("n_kept", "i4"), ("best_x", "f8"), ("best_y", "f8"), ("best_ang", "f8"), ("best_score", "f8"),
                      ("mean_x", "f8"), ("mean_y", "f8"), ("mean_ang", "f8"), ("mean_score", "f8")])
SCAN_INFO_DTYPE = np.dtype([("n_lines", "i4"), ("n_pts", "i4"), ("im_cols", "i4"), ("im_rows", "i4"), ("lidar_x", "f8"), ("lidar_y", "f8")])
RDP_DEFAULTS = dict(least_point=3, thre_line=0.08, least_dist_m=0.5)  # LSD/baseFunc.h:70-72
HYP_DTYPE = np.dtype([("frame", "i4"), ("i_scan", "i4"), ("i_map", "i4"), ("i_pair", "i4"), ("x", "f8"), ("y", "f8"),
                      ("ang", "f8"), ("score", "f8")])
LEGACY_EST_DTYPE = np.dtype([("n_cols", "i4"), ("best_col", "i4"), ("best_score", "f8"), ("estimate_pose", "f8", (3,)),
                             ("estimate_pose_realworld", "f8", (3,))])   # lsdb_fa_legacy_estimate


class LsdbError(RuntimeError):
    pass


class _Params(C.Structure):
    _fields_ = [("sca", C.c_double), ("sig", C.c_double), ("angThre", C.c_double), ("denThre", C.c_double),
                ("pseBin", C.c_int), ("_pad", C.c_int)]


class _RdpParams(C.Structure):
    _fields_ = [("least_point", C.c_int), ("thre_line", C.c_double), ("least_dist_m", C.c_double)]


class _Stats(C.Structure):
    _fields_ = [(f, C.c_longlong) for f in STAT_FIELDS]


_lib = None


def lib():
    """The loaded C-ABI library; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise LsdbError(f"{SO_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                            "(nvcc, sm_100a).  There is no CPU fallback.")
        L = C.CDLL(SO_PATH)
        vp, ci, cd = C.c_void_p, C.c_int, C.c_double
        L.lsdb_version.restype = C.c_char_p
        L.lsdb_last_error.restype = C.c_char_p
        L.lsdb_last_error.argtypes = [vp]
        L.lsdb_create.argtypes = [C.POINTER(vp), ci, vp]
        L.lsdb_destroy.argtypes = [vp]; L.lsdb_destroy.restype = None
        L.lsdb_batch_create.argtypes = [vp, ci, vp, vp, C.POINTER(_Params), ci, C.POINTER(vp)]
        L.lsdb_batch_destroy.argtypes = [vp]; L.lsdb_batch_destroy.restype = None
        L.lsdb_batch_upload.argtypes = [vp, vp]
        L.lsdb_batch_run.argtypes = [vp]
        L.lsdb_batch_sync.argtypes = [vp]
        L.lsdb_batch_download.argtypes = [vp, vp, vp, vp]
        L.lsdb_batch_line_image.argtypes = [vp, ci, vp]
        L.lsdb_batch_line_images.argtypes = [vp, vp]
        L.lsdb_batch_planes.argtypes = [vp, ci, vp, vp, vp, vp, vp, ci, vp, vp]
        L.lsdb_batch_stage_ms.argtypes = [vp, vp]
        L.lsdb_batch_stats.argtypes = [vp, C.POINTER(_Stats)]
        L.lsdb_batch_map_stats.argtypes = [vp, ci, C.POINTER(_Stats)]
        L.lsdb_set_team_warps.argtypes = [vp, ci]
        L.lsdb_batch_launches.argtypes = [vp]
        L.lsdb_lsd.argtypes = [vp, vp, ci, ci, C.POINTER(_Params), vp, ci, vp, vp, vp]
        L.lsdb_map_cache.argtypes = [vp, vp, ci, ci, cd, cd, vp]
        L.lsdb_map_cache_fill.argtypes = [vp, vp, ci, ci, cd, cd, cd, vp]
        L.lsdb_batch_map_caches.argtypes = [vp, vp, cd, cd, vp]
        L.lsdb_fa_map_create_from_batch.argtypes = [vp, ci, C.POINTER(vp)]
        L.lsdb_stream.argtypes = [vp, C.POINTER(vp)]
        L.lsdb_batch_upload_device.argtypes = [vp, vp, vp]
        L.lsdb_batch_lines_device.argtypes = [vp, vp, vp, vp, vp, vp, C.c_longlong]
        L.lsdb_batch_line_images_device.argtypes = [vp, vp]
        L.lsdb_batch_map_caches_device.argtypes = [vp, vp]
        L.lsdb_multi_create.argtypes = [C.POINTER(vp), vp, ci]
        L.lsdb_multi_destroy.argtypes = [vp]; L.lsdb_multi_destroy.restype = None
        L.lsdb_multi_last_error.argtypes = [vp]; L.lsdb_multi_last_error.restype = C.c_char_p
        L.lsdb_multi_shard.argtypes = [ci, ci, ci, vp, vp]; L.lsdb_multi_shard.restype = None
        L.lsdb_multi_lsd.argtypes = [vp, ci, vp, vp, vp, C.POINTER(_Params), ci, vp, vp, vp]
        L.lsdb_read_map_param.argtypes = [C.c_char_p, vp, vp, vp, vp, vp]
        L.lsdb_read_map_value.argtypes = [C.c_char_p, ci, ci, vp]
        L.lsdb_read_map_cache.argtypes = [C.c_char_p, ci, ci, vp]
        L.lsdb_write_map_cache.argtypes = [C.c_char_p, ci, ci, vp]
        L.lsdb_fa_map_create.argtypes = [vp, vp, ci, ci, vp, ci, C.POINTER(vp)]
        L.lsdb_fa_map_destroy.argtypes = [vp]; L.lsdb_fa_map_destroy.restype = None
        L.lsdb_fa_score.argtypes = [vp, vp, ci, vp, vp, vp, vp, vp, vp, vp, ci, vp]
        L.lsdb_fa_score_kept.argtypes = [vp, vp, ci, vp, vp, vp, vp, vp, vp, cd, vp, ci, vp, vp]
        L.lsdb_fa_legacy.argtypes = [vp, vp, vp, ci, cd, cd, cd, vp, vp, vp, ci, vp, ci, vp, vp, vp]
        L.lsdb_fa_legacy_frames.argtypes = [vp, vp, ci, vp, vp, cd, cd, cd, vp, vp, vp, vp, vp, vp, ci, vp]
        L.lsdb_fa_estimate_frames.argtypes = [vp, vp, ci, vp, vp, vp, vp, vp, vp, vp]
        L.lsdb_fa_last_ms.argtypes = [vp]; L.lsdb_fa_last_ms.restype = C.c_float
        L.lsdb_feature_scan_frames.argtypes = [vp, cd, cd, cd, C.POINTER(_RdpParams), ci, vp, vp, vp, vp, vp, ci, vp, vp, ci, vp, vp,
                                               C.c_longlong, vp]
        L.lsdb_batch_upload_scan_rasters.argtypes = [vp, cd, cd, cd, C.POINTER(_RdpParams), ci, vp, vp, vp, vp]
        L.lsdb_scan_estimate_frames.argtypes = [vp, vp, cd, cd, cd, C.POINTER(_RdpParams), ci, vp, vp, vp, vp, vp, vp]
        L.lsdb_feature_scan_last_ms.argtypes = [vp]; L.lsdb_feature_scan_last_ms.restype = C.c_float
        _lib = L
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _params(kw):
    d = dict(LSD_DEFAULTS); d.update(kw or {})
    return _Params(d["sca"], d["sig"], d["angThre"], d["denThre"], int(d["pseBin"]), 0)


class Context:
    """lsdb_ctx: one per process/GPU.  `stream` = a cudaStream_t handle (int) or None."""

    def __init__(self, device=0, stream=None):
        self.h = C.c_void_p()
        self.device = int(device)
        rc = lib().lsdb_create(C.byref(self.h), int(device), C.c_void_p(stream) if stream else None)
        if rc:
            raise LsdbError(f"lsdb_create(device={device}) failed: {ERR_NAMES.get(rc, rc)} — an sm_100 (B200) GPU is "
                            "required; there is no CPU fallback")

    def check(self, rc, what):
        if rc:
            raise LsdbError(f"{what}: {ERR_NAMES.get(rc, rc)}: {lib().lsdb_last_error(self.h).decode()}")

    def close(self):
        if self.h:
            lib().lsdb_destroy(self.h)
            self.h = C.c_void_p()

    def set_team_warps(self, warps):
        """lsdb_set_team_warps: warps per map of the region stage for batches created from now on (0 = by batch size)."""
        self.check(lib().lsdb_set_team_warps(self.h, int(warps)), "lsdb_set_team_warps")

    def lsd(self, map_u8, want_line_im=True, want_remap=False, max_lines=4096, **params):
        """mylsd::myLineSegmentDetector on one host map (LSD/myLSD.h:132) through lsdb_lsd."""
        m = np.ascontiguousarray(map_u8, np.uint8)
        rows, cols = m.shape
        lines = np.zeros(max_lines, LINE_DTYPE)
        n = C.c_int(0)
        im = np.zeros((rows, cols), np.uint8) if want_line_im else None
        rm = np.zeros((rows, cols), np.uint8) if want_remap else None
        prm = _params(params)
        self.check(lib().lsdb_lsd(self.h, _p(m), cols, rows, C.byref(prm), _p(lines), max_lines, C.byref(n), _p(im), _p(rm)),
                   "lsdb_lsd")
        return dict(n=n.value, lines=lines[:n.value].copy(), line_im=im, map_out=rm)


def _ctx_map_cache(self, map_u8, res, max_dist=1.0, unreached=None):
    """mylsd::createMapCache (LSD/myLSD.h:131) through lsdb_map_cache: rows x cols f64 metres.  `unreached` = the value of the
    cells the brush fire never reaches when it is not max_dist (the catkin snapshot's 3-argument flavour stores 2)."""
    m = np.ascontiguousarray(map_u8, np.uint8)
    rows, cols = m.shape
    out = np.zeros((rows, cols), np.float64)
    if unreached is None:
        self.check(lib().lsdb_map_cache(self.h, _p(m), cols, rows, float(res), float(max_dist), _p(out)), "lsdb_map_cache")
    else:
        self.check(lib().lsdb_map_cache_fill(self.h, _p(m), cols, rows, float(res), float(max_dist), float(unreached), _p(out)), "lsdb_map_cache_fill")
    return out


Context.map_cache = _ctx_map_cache


def _ctx_stream(self):
    """lsdb_stream: the context's cudaStream_t handle (int); the device-memory calls of Batch enqueue their work there."""
    s = C.c_void_p()
    self.check(lib().lsdb_stream(self.h, C.byref(s)), "lsdb_stream")
    return s.value or 0


def _ctx_torch_stream(self):
    """the context's stream as a torch.cuda.ExternalStream"""
    import torch
    return torch.cuda.ExternalStream(self.stream, device=torch.device("cuda", self.device))


Context.stream = property(_ctx_stream)
Context.torch_stream = _ctx_torch_stream


class MultiContext:
    """One process, several GPUs: lsdb_multi_* (a batch of maps split contiguously over the devices, one host thread each)."""

    def __init__(self, devices):
        self.h = C.c_void_p()
        d = np.asarray(list(devices), np.int32)
        rc = lib().lsdb_multi_create(C.byref(self.h), _p(d), len(d))
        if rc != 0:
            raise LsdbError(f"lsdb_multi_create: {ERR_NAMES.get(rc, rc)}")
        self.n = len(d)

    def lsd(self, maps, max_lines=4096, want_rects=False, **params):
        ms = [np.ascontiguousarray(m, np.uint8) for m in maps]
        n = len(ms)
        cols = np.array([m.shape[1] for m in ms], np.int32); rows = np.array([m.shape[0] for m in ms], np.int32)
        ptrs = (C.c_void_p * max(n, 1))(*[m.ctypes.data for m in ms])
        prm = _Params(**dict(LSD_DEFAULTS, **params))
        counts = np.zeros(n, np.int32); lines = np.zeros((n, max_lines), LINE_DTYPE)
        rects = np.zeros((n, max_lines, 13)) if want_rects else None
        rc = lib().lsdb_multi_lsd(self.h, n, ptrs, _p(cols), _p(rows), C.byref(prm), max_lines, _p(counts), _p(lines), _p(rects))
        if rc != 0:
            raise LsdbError(f"lsdb_multi_lsd: {ERR_NAMES.get(rc, rc)}: {lib().lsdb_multi_last_error(self.h).decode()}")
        out = dict(counts=counts, lines=[lines[i, :counts[i]].copy() for i in range(n)])
        if want_rects:
            out["rects"] = [rects[i, :counts[i]].copy() for i in range(n)]
        return out

    def close(self):
        if self.h:
            lib().lsdb_multi_destroy(self.h)
            self.h = C.c_void_p()


def _io_check(rc, what, path):
    if rc != 0:
        raise LsdbError(f"{what}({path}): {ERR_NAMES.get(rc, rc)}")


def read_map_param(path):
    """mapParam.txt -> dict(cols, rows, res, ori_x, ori_y)  (LSD/main_on_windows.cpp:28-34)"""
    c, r = C.c_int(0), C.c_int(0); res, ox, oy = C.c_double(0), C.c_double(0), C.c_double(0)
    _io_check(lib().lsdb_read_map_param(os.fsencode(path), C.byref(c), C.byref(r), C.byref(res), C.byref(ox), C.byref(oy)), "lsdb_read_map_param", path)
    return dict(cols=c.value, rows=r.value, res=res.value, ori_x=ox.value, ori_y=oy.value)


def read_map_value(path, cols, rows):
    """mapValue*.txt -> rows x cols u8 (value & 0xFF, LSD/main_on_windows.cpp:38-46)"""
    out = np.zeros((rows, cols), np.uint8)
    _io_check(lib().lsdb_read_map_value(os.fsencode(path), cols, rows, _p(out)), "lsdb_read_map_value", path)
    return out


def read_map_cache(path, cols, rows):
    """mapCache.txt -> rows x cols f64 (LSD/test.cpp:11-17)"""
    out = np.zeros((rows, cols), np.float64)
    _io_check(lib().lsdb_read_map_cache(os.fsencode(path), cols, rows, _p(out)), "lsdb_read_map_cache", path)
    return out


def write_map_cache(path, cache):
    a = np.ascontiguousarray(cache, np.float64)
    _io_check(lib().lsdb_write_map_cache(os.fsencode(path), a.shape[1], a.shape[0], _p(a)), "lsdb_write_map_cache", path)


def _ctx_feature_scan(self, map_res, map_ori_x, map_ori_y, frames, want_rasters=False, capacity=None, raw=False, **rdp):
    """myrdp::FeatureScan (LSD/myRDP.h:63) for a list of frames [(ranges, angles), ...] through lsdb_feature_scan_frames
    (a sizing query, then the real call; `capacity` = (max_lines, max_pts) skips the query).  Returns one dict per frame:
    lines (LINE_DTYPE), pts (P,2), lidar_pos (2,), size (cols, rows) and, when asked for, line_im (rows x cols u8);
    raw=True returns the concatenated arrays (info, lines, line_off, pts, pt_off) instead."""
    nf = len(frames)
    boff = np.zeros(nf + 1, np.int32)
    for i, (r, _a) in enumerate(frames):
        boff[i + 1] = boff[i] + len(r)
    rng = np.ascontiguousarray(np.concatenate([np.asarray(r, np.float64) for r, _ in frames])) if nf else np.zeros(0)
    ang = np.ascontiguousarray(np.concatenate([np.asarray(a, np.float64) for _, a in frames])) if nf else np.zeros(0)
    d = dict(RDP_DEFAULTS); d.update(rdp)
    prm = _RdpParams(int(d["least_point"]), float(d["thre_line"]), float(d["least_dist_m"]))
    info = np.zeros(nf, SCAN_INFO_DTYPE)
    loff = np.zeros(nf + 1, np.int32); poff = np.zeros(nf + 1, np.int32); ioff = np.zeros(nf + 1, np.int64)
    args = (self.h, float(map_res), float(map_ori_x), float(map_ori_y), C.byref(prm), nf, _p(rng), _p(ang), _p(boff), _p(info))
    if capacity is None or want_rasters:
        self.check(lib().lsdb_feature_scan_frames(*args, None, 0, _p(loff), None, 0, _p(poff), None, 0, _p(ioff)), "lsdb_feature_scan_frames")
        capacity = (int(loff[-1]), int(poff[-1]))
    lines = np.empty(max(int(capacity[0]), 1), LINE_DTYPE); pts = np.empty((max(int(capacity[1]), 1), 2))
    im = np.zeros(max(int(ioff[-1]), 1), np.uint8) if want_rasters else None
    self.check(lib().lsdb_feature_scan_frames(*args, _p(lines), len(lines), _p(loff), _p(pts), len(pts), _p(poff), _p(im),
                                              0 if im is None else len(im), _p(ioff)), "lsdb_feature_scan_frames")
    if raw:
        return info, lines[:loff[-1]], loff, pts[:poff[-1]], poff
    out = []
    for f in range(nf):
        w, h = int(info[f]["im_cols"]), int(info[f]["im_rows"])
        rec = dict(lines=lines[loff[f]:loff[f + 1]].copy(), pts=pts[poff[f]:poff[f + 1]].copy(),
                   lidar_pos=np.array([info[f]["lidar_x"], info[f]["lidar_y"]]), size=(w, h))
        if want_rasters:
            rec["line_im"] = im[ioff[f]:ioff[f + 1]].reshape(max(h, 0), max(w, 0)).copy() if w > 0 and h > 0 else np.zeros((max(h, 0), max(w, 0)), np.uint8)
        out.append(rec)
    return out


def _marshal_sweeps(sweeps, rdp):
    nf = len(sweeps)
    boff = np.zeros(nf + 1, np.int32)
    for i, (r, _a) in enumerate(sweeps):
        boff[i + 1] = boff[i] + len(r)
    rng = np.ascontiguousarray(np.concatenate([np.asarray(r, np.float64) for r, _ in sweeps])) if nf else np.zeros(0)
    ang = np.ascontiguousarray(np.concatenate([np.asarray(a, np.float64) for _, a in sweeps])) if nf else np.zeros(0)
    d = dict(RDP_DEFAULTS); d.update(rdp)
    return nf, boff, rng, ang, _RdpParams(int(d["least_point"]), float(d["thre_line"]), float(d["least_dist_m"]))


def _ctx_feature_scan_info(self, map_res, map_ori_x, map_ori_y, sweeps, **rdp):
    """The sizing query of lsdb_feature_scan_frames: SCAN_INFO_DTYPE per sweep (lines, samples, raster size, lidarPos)."""
    nf, boff, rng, ang, prm = _marshal_sweeps(sweeps, rdp)
    info = np.zeros(nf, SCAN_INFO_DTYPE)
    loff = np.zeros(nf + 1, np.int32); poff = np.zeros(nf + 1, np.int32); ioff = np.zeros(nf + 1, np.int64)
    self.check(lib().lsdb_feature_scan_frames(self.h, float(map_res), float(map_ori_x), float(map_ori_y), C.byref(prm), nf, _p(rng), _p(ang),
                                              _p(boff), _p(info), None, 0, _p(loff), None, 0, _p(poff), None, 0, _p(ioff)),
               "lsdb_feature_scan_frames")
    return info


Context.feature_scan_info = _ctx_feature_scan_info
Context.feature_scan = _ctx_feature_scan
Context.feature_scan_last_ms = lambda self: float(lib().lsdb_feature_scan_last_ms(self.h))


class Batch:
    """lsdb_batch: device-resident buffers for a fixed list of map sizes."""

    def __init__(self, ctx, sizes, max_lines=4096, **params):
        self.ctx = ctx
        self.sizes = [(int(c), int(r)) for c, r in sizes]
        self.n = len(self.sizes)
        self.max_lines = max_lines
        self.sca = dict(LSD_DEFAULTS, **params)["sca"]
        cols = np.array([s[0] for s in self.sizes], np.int32); rows = np.array([s[1] for s in self.sizes], np.int32)
        self.h = C.c_void_p()
        prm = _params(params)
        ctx.check(lib().lsdb_batch_create(ctx.h, self.n, _p(cols), _p(rows), C.byref(prm), max_lines, C.byref(self.h)),
                  "lsdb_batch_create")

    def scaled(self, i):
        c, r = self.sizes[i]
        return int(np.floor(c * self.sca)), int(np.floor(r * self.sca))

    def upload(self, maps):
        """maps: list of C-contiguous uint8 arrays (rows x cols) or raw host pointers (ints)."""
        ptrs = (C.c_void_p * self.n)()
        keep = []
        for i, m in enumerate(maps):
            if isinstance(m, (int, np.integer)):
                ptrs[i] = int(m)
            else:
                a = np.ascontiguousarray(m, np.uint8); keep.append(a)
                assert a.shape == (self.sizes[i][1], self.sizes[i][0]), (a.shape, self.sizes[i])
                ptrs[i] = a.ctypes.data
        self._keep = keep
        self.ctx.check(lib().lsdb_batch_upload(self.h, C.cast(ptrs, C.c_void_p)), "lsdb_batch_upload")

    def upload_scan_rasters(self, map_res, map_ori_x, map_ori_y, sweeps, **rdp):
        """lsdb_batch_upload_scan_rasters: the FeatureScan rasters of `sweeps` become the batch's maps on the device
        (occupied = 1); the batch must have the raster sizes of Context.feature_scan_info.  Returns the scan info."""
        nf, boff, rng, ang, prm = _marshal_sweeps(sweeps, rdp)
        info = np.zeros(nf, SCAN_INFO_DTYPE)
        self.ctx.check(lib().lsdb_batch_upload_scan_rasters(self.h, float(map_res), float(map_ori_x), float(map_ori_y), C.byref(prm), nf,
                                                            _p(rng), _p(ang), _p(boff), _p(info)), "lsdb_batch_upload_scan_rasters")
        return info

    def upload_device(self, maps):
        """lsdb_batch_upload_device: the grids from device memory, copied device to device on the context stream.  maps: 2-D
        uint8 CUDA tensors (rows x cols; row-pitched views such as a column slice of a wider tensor work) or 2-D objects with a
        __cuda_array_interface__ of u1 whose last stride is 1.  The context stream first waits for torch's current stream, so
        grids produced there are ready (other producers must be ordered against Context.stream by the caller), and torch's
        current stream then waits for the copies, so that whatever it does next with the grids' memory comes after them.  The
        call returns without waiting for the copies."""
        import torch
        if len(maps) != self.n:
            raise ValueError(f"{len(maps)} maps for a batch of {self.n}")
        ptrs = (C.c_void_p * self.n)(); pitches = np.zeros(self.n, np.int64)
        for i, m in enumerate(maps):
            ptr, shape, pitch = _dev_grid(m)
            if shape != (self.sizes[i][1], self.sizes[i][0]):
                raise ValueError(f"map {i}: shape {shape}, batch expects {(self.sizes[i][1], self.sizes[i][0])}")
            ptrs[i] = ptr; pitches[i] = pitch
        ext = self.ctx.torch_stream()
        cur = torch.cuda.current_stream(ext.device)
        ext.wait_stream(cur)
        self.ctx.check(lib().lsdb_batch_upload_device(self.h, C.cast(ptrs, C.c_void_p), _p(pitches)), "lsdb_batch_upload_device")
        cur.wait_stream(ext)
        self._keep_dev = list(maps)   # memory that torch does not own must outlive the copies

    def _device_out(self, what, call):
        """call(), which writes torch allocations of the current stream on the context stream, between two stream waits: the
        context stream first waits for torch's current stream, where the outputs were allocated; torch's current stream then
        waits for the context stream, so that its consumers see the results, and a later reuse of the outputs' memory (torch
        reuses a freed block on the stream that allocated it) comes after the writes.  That wait stands in for record_stream,
        which would tie the tensors to the context's stream: a tensor freed after Context.close() would then make torch record
        an event on a destroyed stream.  Nothing is synchronised."""
        import torch
        ext = self.ctx.torch_stream()
        cur = torch.cuda.current_stream(ext.device)
        ext.wait_stream(cur)
        self.ctx.check(call(), what)
        cur.wait_stream(ext)

    def lines_device(self, max_total=None, want_rects=False):
        """lsdb_batch_lines_device: the segment tables of the last run, built on the device, as CUDA tensors: counts (n,) int32,
        offsets (n+1,) int32, status (n,) int32 (0, or LSDB_ERR_CAPACITY = 3 / LSDB_ERR_TIMEOUT = 4), lines (max_total, 80) uint8
        lsdb_line records (line_fields() views them) and with want_rects rects (max_total, 13) float64.  Map i's records are rows
        offsets[i] .. offsets[i] + counts[i] - 1.  max_total defaults to n * max_lines, which always suffices.  Nothing is
        synchronised: torch's current stream waits for the results."""
        import torch
        max_total = self.n * self.max_lines if max_total is None else int(max_total)
        if max_total < 0:
            raise ValueError("max_total must be >= 0")
        dev = torch.device("cuda", self.ctx.device)
        counts = torch.empty(self.n, dtype=torch.int32, device=dev)
        offsets = torch.empty(self.n + 1, dtype=torch.int32, device=dev)
        status = torch.empty(self.n, dtype=torch.int32, device=dev)
        lines = torch.empty((max_total, LINE_DTYPE.itemsize), dtype=torch.uint8, device=dev)
        rects = torch.empty((max_total, 13), dtype=torch.float64, device=dev) if want_rects else None
        ptr = lambda t: (t.data_ptr() or None) if t is not None else None  # noqa: E731  (an empty tensor has no storage)
        self._device_out("lsdb_batch_lines_device",
                         lambda: lib().lsdb_batch_lines_device(self.h, ptr(counts), ptr(offsets), ptr(status), ptr(lines), ptr(rects), max_total))
        out = dict(counts=counts, offsets=offsets, status=status, lines=lines)
        if want_rects:
            out["rects"] = rects
        return out

    def _packed(self, out, dtype, what):
        """a packed per-map CUDA buffer (map i after the rows*cols elements of the maps before it) and its per-map views"""
        import torch
        total = sum(c * r for c, r in self.sizes)
        if out is None:
            out = torch.empty(total, dtype=dtype, device=torch.device("cuda", self.ctx.device))
        elif not (isinstance(out, torch.Tensor) and out.is_cuda and out.dtype == dtype and out.is_contiguous() and out.numel() >= total):
            raise ValueError(f"{what}: out must be a contiguous CUDA {dtype} tensor of at least {total} elements")
        flat, views, o = out.view(-1), [], 0
        for c, r in self.sizes:
            views.append(flat[o:o + r * c].view(r, c))
            o += r * c
        return out, views

    def line_images_device(self, out=None):
        """lsdb_batch_line_images_device: lineIm of every map rasterised on the device into one packed uint8 CUDA tensor (`out`
        or a new one).  Returns (packed tensor, [rows x cols view per map]); nothing is synchronised."""
        import torch
        out, views = self._packed(out, torch.uint8, "line_images_device")
        self._device_out("lsdb_batch_line_images_device", lambda: lib().lsdb_batch_line_images_device(self.h, out.data_ptr()))
        return out, views

    def map_caches_device(self, out=None):
        """lsdb_batch_map_caches_device: the caches the last map_caches() left, copied into one packed float64 CUDA tensor (`out`
        or a new one).  Returns (packed tensor, [rows x cols view per map]); nothing is synchronised."""
        import torch
        out, views = self._packed(out, torch.float64, "map_caches_device")
        self._device_out("lsdb_batch_map_caches_device", lambda: lib().lsdb_batch_map_caches_device(self.h, out.data_ptr()))
        return out, views

    def run(self):
        self.ctx.check(lib().lsdb_batch_run(self.h), "lsdb_batch_run")

    def sync(self):
        self.ctx.check(lib().lsdb_batch_sync(self.h), "lsdb_batch_sync")

    def download(self, want_lines=True, want_rects=False):
        counts = np.zeros(self.n, np.int32)
        lines = np.zeros((self.n, self.max_lines), LINE_DTYPE) if want_lines else None
        rects = np.zeros((self.n, self.max_lines, 13)) if want_rects else None
        self.ctx.check(lib().lsdb_batch_download(self.h, _p(counts), _p(lines), _p(rects)), "lsdb_batch_download")
        out = dict(counts=counts)
        if want_lines:
            out["lines"] = [lines[i, :counts[i]].copy() for i in range(self.n)]
        if want_rects:
            out["rects"] = [rects[i, :counts[i]].copy() for i in range(self.n)]
        return out

    def counts(self):
        counts = np.zeros(self.n, np.int32)
        self.ctx.check(lib().lsdb_batch_download(self.h, _p(counts), None, None), "lsdb_batch_download")
        return counts

    def line_image(self, i):
        c, r = self.sizes[i]
        im = np.zeros((r, c), np.uint8)
        self.ctx.check(lib().lsdb_batch_line_image(self.h, i, _p(im)), "lsdb_batch_line_image")
        return im

    def line_images(self, outs=None):
        """lineIm of every map, rasterised on the device (lsdb_batch_line_images).  `outs`: list of rows x cols u8 arrays to
        fill (e.g. views of pinned memory), default fresh arrays."""
        if outs is None:
            outs = [np.zeros((r, c), np.uint8) for c, r in self.sizes]
        ptrs = (C.c_void_p * self.n)(*[o.ctypes.data for o in outs])
        self.ctx.check(lib().lsdb_batch_line_images(self.h, ptrs), "lsdb_batch_line_images")
        return outs

    def map_caches(self, res, max_dist=1.0, unreached=None, download=True):
        """mylsd::createMapCache of every map of the batch, on the device, from the uploaded source planes
        (lsdb_batch_map_caches).  `res`: one resolution for all maps or one per map; `unreached` = the value of the cells
        the brush fire never reaches (default max_dist; the catkin snapshot stores 2).  The caches stay on the device for
        FaMap.from_batch; with download=True they also come back as a list of rows x cols f64 arrays, else None."""
        r = np.ascontiguousarray(np.broadcast_to(np.asarray(res, np.float64), (self.n,)))
        outs = [np.empty((rows, cols)) for cols, rows in self.sizes] if download else None
        ptrs = (C.c_void_p * self.n)(*[o.ctypes.data for o in outs]) if download else None
        self.ctx.check(lib().lsdb_batch_map_caches(self.h, _p(r), float(max_dist), float(max_dist if unreached is None else unreached), ptrs),
                       "lsdb_batch_map_caches")
        return outs

    def planes(self, i):
        W, H = self.scaled(i)
        mag = np.zeros((H, W)); deg = np.zeros((H, W)); used = np.zeros((H, W), np.uint8)
        labels = np.zeros((H, W), np.int32); seeds = np.zeros(H * W, np.int32); ns = C.c_int(0); mg = C.c_double(0)
        self.ctx.check(lib().lsdb_batch_planes(self.h, i, _p(mag), _p(deg), _p(used), _p(labels), _p(seeds), H * W,
                                               C.byref(ns), C.byref(mg)), "lsdb_batch_planes")
        return dict(mag=mag, deg=deg, used=used, labels=labels, seeds=seeds[:ns.value].copy(), max_grad=mg.value)

    def stage_ms(self):
        ms = np.zeros(len(STAGES), np.float32)
        self.ctx.check(lib().lsdb_batch_stage_ms(self.h, _p(ms)), "lsdb_batch_stage_ms")
        return dict(zip(STAGES, (float(v) for v in ms)))

    def stats(self):
        st = _Stats()
        self.ctx.check(lib().lsdb_batch_stats(self.h, C.byref(st)), "lsdb_batch_stats")
        return {f: getattr(st, f) for f in STAT_FIELDS}

    def map_stats(self, i):
        st = _Stats()
        self.ctx.check(lib().lsdb_batch_map_stats(self.h, int(i), C.byref(st)), "lsdb_batch_map_stats")
        return {f: getattr(st, f) for f in STAT_FIELDS}

    def launches(self):
        return lib().lsdb_batch_launches(self.h)

    def close(self):
        if self.h:
            lib().lsdb_batch_destroy(self.h)
            self.h = C.c_void_p()


def _dev_grid(m):
    """(device pointer, (rows, cols), row pitch in bytes) of a 2-D uint8 CUDA tensor or __cuda_array_interface__ object whose
    last stride is 1"""
    import torch
    if isinstance(m, torch.Tensor):
        if not m.is_cuda or m.dtype != torch.uint8 or m.dim() != 2:
            raise ValueError(f"a 2-D uint8 CUDA tensor is required, got {m.dtype} {tuple(m.shape)} on {m.device}")
        shape, strides, ptr = tuple(m.shape), tuple(m.stride()), m.data_ptr()
    else:
        cai = getattr(m, "__cuda_array_interface__", None)
        if cai is None or len(cai["shape"]) != 2 or cai["typestr"] not in ("|u1", "<u1", ">u1"):
            raise ValueError("a 2-D uint8 CUDA tensor or __cuda_array_interface__ object is required")
        shape = tuple(int(v) for v in cai["shape"])
        strides = tuple(cai["strides"]) if cai.get("strides") else (shape[1], 1)
        ptr = int(cai["data"][0])
    rows, cols = shape
    if cols > 1 and strides[1] != 1:
        raise ValueError(f"the last stride must be 1, got {strides}")
    return ptr, (rows, cols), (int(strides[0]) if rows > 1 else cols)


def line_fields(lines):
    """zero-copy views of an (N, 80) uint8 tensor of lsdb_line records: ((N, 9) float64 k, b, dx, dy, x1, y1, x2, y2, len;
    (N,) int32 orient)"""
    import torch
    return lines.view(torch.float64)[:, :9], lines.view(torch.int32)[:, 18]


def lines_to_array(lines):
    """structured lsdb_line records -> (n,10) float array in oracle column order"""
    out = np.zeros((len(lines), 10))
    for j, f in enumerate(["k", "b", "dx", "dy", "x1", "y1", "x2", "y2", "len"]):
        out[:, j] = lines[f]
    out[:, 9] = lines["orient"]
    return out


def array_to_lines(arr):
    arr = np.asarray(arr, np.float64).reshape(-1, 10)
    out = np.zeros(len(arr), LINE_DTYPE)
    for j, f in enumerate(["k", "b", "dx", "dy", "x1", "y1", "x2", "y2", "len"]):
        out[f] = arr[:, j]
    out["orient"] = arr[:, 9].astype(np.int32)
    return out


class FaMap:
    """lsdb_fa_map: mapCache + the map's LSD lines resident on the device."""

    def __init__(self, ctx, map_cache, map_lines):
        self.ctx = ctx
        mc = np.ascontiguousarray(map_cache, np.float64)
        ml = map_lines if getattr(map_lines, "dtype", None) == LINE_DTYPE else array_to_lines(map_lines)
        ml = np.ascontiguousarray(ml)
        self.h = C.c_void_p()
        rows, cols = mc.shape
        ctx.check(lib().lsdb_fa_map_create(ctx.h, _p(mc), cols, rows, _p(ml), len(ml), C.byref(self.h)), "lsdb_fa_map_create")
        self.n_lines = len(ml)

    @classmethod
    def from_batch(cls, batch, i):
        """lsdb_fa_map_create_from_batch: map i of `batch` — its cache from Batch.map_caches, copied on the device, and its
        segment table as Batch.download returns it.  The FaMap owns its copies and outlives the batch."""
        self = cls.__new__(cls)
        self.ctx = batch.ctx
        self.h = C.c_void_p()
        batch.ctx.check(lib().lsdb_fa_map_create_from_batch(batch.h, int(i), C.byref(self.h)), "lsdb_fa_map_create_from_batch")
        self.n_lines = int(batch.counts()[i])
        return self

    def _marshal(self, frames):
        nf = len(frames)
        sl = [f["scan_lines"] if getattr(f["scan_lines"], "dtype", None) == LINE_DTYPE else array_to_lines(f["scan_lines"])
              for f in frames]
        loff = np.zeros(nf + 1, np.int32); poff = np.zeros(nf + 1, np.int32)
        for i, f in enumerate(frames):
            loff[i + 1] = loff[i] + len(sl[i]); poff[i + 1] = poff[i] + len(f["pts"])
        lines = np.ascontiguousarray(np.concatenate(sl)) if nf else np.zeros(0, LINE_DTYPE)
        pts = np.ascontiguousarray(np.concatenate([np.asarray(f["pts"], np.float64).reshape(-1, 2) for f in frames])) if nf else np.zeros((0, 2))
        lid = np.ascontiguousarray(np.array([f["lidar_pose"] for f in frames], np.float64).reshape(nf, 2))
        last = np.ascontiguousarray(np.array([f["last_pose"] for f in frames], np.float64).reshape(nf, 3))
        return nf, lines, loff, pts, poff, lid, last

    def score(self, frames, max_hyp=None):
        """frames: list of dicts(scan_lines=(n,10) or LINE_DTYPE, pts=(P,2), lidar_pose=(2,), last_pose=(3,))."""
        nf, lines, loff, pts, poff, lid, last = self._marshal(frames)
        if max_hyp is None:
            max_hyp = max(4 * int(loff[-1]) * max(self.n_lines, 1), 4)
        out = np.zeros(max_hyp, HYP_DTYPE); n = C.c_int(0)
        self.ctx.check(lib().lsdb_fa_score(self.ctx.h, self.h, nf, _p(lines), _p(loff), _p(pts), _p(poff), _p(lid), _p(last),
                                           _p(out), max_hyp, C.byref(n)), "lsdb_fa_score")
        return out[:n.value].copy()

    def legacy(self, scan_lines, map_resol, map_ori, lidar_pos, ranges, angles, max_cols=None):
        """lsdb_fa_legacy — the catkin snapshot's FeatureAssociation (ROS/lsd/src/FeatureAssociation.cpp:36-130) for one frame.
        Returns (pose_all (T,15): the columns of the reference's poseAll, estimate_pose (3,), estimate_pose_realworld (3,));
        the two estimates are None when no scan line pairs with any map line."""
        sl = scan_lines if getattr(scan_lines, "dtype", None) == LINE_DTYPE else array_to_lines(scan_lines)
        sl = np.ascontiguousarray(sl)
        r = np.ascontiguousarray(ranges, np.float64); a = np.ascontiguousarray(angles, np.float64)
        if len(r) != len(a):
            raise ValueError("ranges and angles differ in length")
        lp = np.ascontiguousarray(lidar_pos, np.int32)
        if max_cols is None:
            max_cols = max(4 * len(sl) * max(self.n_lines, 1), 4)
        out = np.zeros((max_cols, 15)); n = C.c_int(0); est = np.zeros(3); real = np.zeros(3)
        self.ctx.check(lib().lsdb_fa_legacy(self.ctx.h, self.h, _p(sl), len(sl), float(map_resol), float(map_ori[0]), float(map_ori[1]), _p(lp),
                                            _p(r), _p(a), len(r), _p(out), max_cols, C.byref(n), _p(est), _p(real)), "lsdb_fa_legacy")
        if n.value == 0:
            return out[:0].copy(), None, None
        return out[:n.value].copy(), est, real

    @staticmethod
    def pack_legacy(frames):
        """frames (dicts of scan_lines, lidar_pos, ranges, angles) as the flat arrays lsdb_fa_legacy_frames takes:
        (n_frames, scan lines, scan_line_off, lidar_pos (n,2) int32, ranges, angles, ray_off)."""
        nf = len(frames)
        sl = [f["scan_lines"] if getattr(f["scan_lines"], "dtype", None) == LINE_DTYPE else array_to_lines(f["scan_lines"]) for f in frames]
        loff = np.zeros(nf + 1, np.int32); roff = np.zeros(nf + 1, np.int32)
        loff[1:] = np.cumsum([len(x) for x in sl]); roff[1:] = np.cumsum([len(f["ranges"]) for f in frames])
        if any(len(f["ranges"]) != len(f["angles"]) for f in frames):
            raise ValueError("ranges and angles differ in length")
        lines = np.ascontiguousarray(np.concatenate(sl)) if nf else np.zeros(0, LINE_DTYPE)
        lp = np.ascontiguousarray(np.array([np.asarray(f["lidar_pos"]).reshape(2) for f in frames], np.int32).reshape(nf, 2))
        r = np.ascontiguousarray(np.concatenate([np.asarray(f["ranges"], np.float64).ravel() for f in frames])) if nf else np.zeros(0)
        a = np.ascontiguousarray(np.concatenate([np.asarray(f["angles"], np.float64).ravel() for f in frames])) if nf else np.zeros(0)
        return nf, lines, loff, lp, r, a, roff

    def legacy_frames(self, frames, map_resol, map_ori, want_pose_all=False, max_cols=None):
        """lsdb_fa_legacy_frames — lsdb_fa_legacy for many frames in one call.  `frames`: a list of dicts (scan_lines, lidar_pos,
        ranges, angles) or the tuple pack_legacy() returned.  Returns (est LEGACY_EST_DTYPE[n_frames], pose_all (T,15) or None,
        col_off int32[n_frames+1]); frame f's records are pose_all[col_off[f]:col_off[f+1]].  max_cols bounds pose_all (default:
        every pair the frames' scan lines could form)."""
        nf, lines, loff, lp, r, a, roff = frames if isinstance(frames, tuple) else self.pack_legacy(frames)
        est = np.zeros(nf, LEGACY_EST_DTYPE); coff = np.zeros(nf + 1, np.int32)
        out = None
        if want_pose_all:
            if max_cols is None:
                max_cols = min(4 * int(loff[-1]) * max(self.n_lines, 1), 2**31 - 1)
            out = np.empty((max(int(max_cols), 1), 15))   # only the T records written are touched
        self.ctx.check(lib().lsdb_fa_legacy_frames(self.ctx.h, self.h, nf, _p(lines), _p(loff), float(map_resol), float(map_ori[0]),
                                                   float(map_ori[1]), _p(lp), _p(r), _p(a), _p(roff), _p(est), _p(out),
                                                   int(max_cols or 0), _p(coff)), "lsdb_fa_legacy_frames")
        return est, (out[:coff[-1]] if want_pose_all else None), coff

    def pack(self, frames):
        """the frames as the flat arrays the C ABI takes (do this once when the same frames are scored repeatedly)"""
        return self._marshal(frames)

    def score_kept(self, frames, keep_below=3.0, max_kept=None, out=None):
        """lsdb_fa_score_kept: only the hypotheses with score < keep_below (what the reference keeps), compacted on the device.
        `frames` is a list of frame dicts or the tuple pack() returned.  Returns (kept HYP_DTYPE records, hypotheses scored).
        `out`: a caller-owned HYP_DTYPE array (pinned host memory, say) the records are written to; the result is then a view of it."""
        nf, lines, loff, pts, poff, lid, last = frames if isinstance(frames, tuple) else self._marshal(frames)
        own = out is None
        if own:
            if max_kept is None:
                max_kept = max(4 * int(loff[-1]) * max(self.n_lines, 1) // 8, 4096)
            out = np.empty(max_kept, HYP_DTYPE)
        else:
            if out.dtype != HYP_DTYPE or not out.flags.c_contiguous:
                raise ValueError("out must be a contiguous HYP_DTYPE array")
            max_kept = len(out) if max_kept is None else min(int(max_kept), len(out))
        nk = C.c_int(0); nh = C.c_int(0)
        self.ctx.check(lib().lsdb_fa_score_kept(self.ctx.h, self.h, nf, _p(lines), _p(loff), _p(pts), _p(poff), _p(lid), _p(last),
                                                float(keep_below), _p(out), max_kept, C.byref(nk), C.byref(nh)), "lsdb_fa_score_kept")
        return (out[:nk.value].copy() if own else out[:nk.value]), nh.value

    def estimate(self, frames):
        """Per-frame reduction on the device (lsdb_fa_estimate_frames): one EST_DTYPE record per frame."""
        nf, lines, loff, pts, poff, lid, last = self._marshal(frames)
        out = np.zeros(nf, EST_DTYPE)
        self.ctx.check(lib().lsdb_fa_estimate_frames(self.ctx.h, self.h, nf, _p(lines), _p(loff), _p(pts), _p(poff), _p(lid), _p(last),
                                                     _p(out)), "lsdb_fa_estimate_frames")
        return out

    def scan_estimate(self, map_res, map_ori_x, map_ori_y, sweeps, last_pose=None, **rdp):
        """lidar sweeps [(ranges, angles), ...] -> (SCAN_INFO_DTYPE, EST_DTYPE) records per frame in one call
        (lsdb_scan_estimate_frames: FeatureScan, scoring and reduction, raster samples device-resident)."""
        nf = len(sweeps)
        boff = np.zeros(nf + 1, np.int32)
        for i, (r, _a) in enumerate(sweeps):
            boff[i + 1] = boff[i] + len(r)
        rng = np.ascontiguousarray(np.concatenate([np.asarray(r, np.float64) for r, _ in sweeps])) if nf else np.zeros(0)
        ang = np.ascontiguousarray(np.concatenate([np.asarray(a, np.float64) for _, a in sweeps])) if nf else np.zeros(0)
        d = dict(RDP_DEFAULTS); d.update(rdp)
        prm = _RdpParams(int(d["least_point"]), float(d["thre_line"]), float(d["least_dist_m"]))
        last = np.tile(np.array([-1.0, -1.0, 0.0]), (nf, 1)) if last_pose is None else np.ascontiguousarray(last_pose, np.float64).reshape(nf, 3)
        info = np.zeros(nf, SCAN_INFO_DTYPE); est = np.zeros(nf, EST_DTYPE)
        self.ctx.check(lib().lsdb_scan_estimate_frames(self.ctx.h, self.h, float(map_res), float(map_ori_x), float(map_ori_y), C.byref(prm), nf,
                                                       _p(rng), _p(ang), _p(boff), _p(last), _p(info), _p(est)), "lsdb_scan_estimate_frames")
        return info, est

    def last_ms(self):
        return float(lib().lsdb_fa_last_ms(self.ctx.h))

    def close(self):
        if self.h:
            lib().lsdb_fa_map_destroy(self.h)
            self.h = C.c_void_p()
