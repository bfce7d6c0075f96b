"""lsdb_batch_map_caches (createMapCache, LSD/myLSD.cpp:11-127, for every map of an LSD batch in one chain of launches) and
lsdb_fa_map_create_from_batch (an association map straight from the batch): cell for cell what the oracle restatement and the
single-map call give, whatever the grouping, the order of the maps or the moment of the call."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np
import pytest

import oraclebind
import synth
from test_oracle import _extra_maps

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
BUNDLED = ["mapValue", "mapValue_aisle1", "mapValue_aisle2", "mapValue_aisle3", "mapValue_map1", "mapValue_map2"]
ANY_SIZE = dict(sca=1.0, sig=2.0)   # LSD parameters whose batch takes maps down to 1 x 1 (Gaussian half-width 8 as with 0.3 / 0.6)


_fill_lib = None


def map_cache_fill(map_u8, res, max_dist, unreached):
    """the reference's FIFO brush fire with z_occ_max_dis = max_dist and `unreached` in the cells it never reaches
    (tests/map_cache_fill.c, built with the oracle's flags into a temporary directory on first use)"""
    global _fill_lib
    if _fill_lib is None:
        so = os.path.join(tempfile.mkdtemp(prefix="lsdb_mc_fill_"), "libmcfill.so")
        subprocess.check_call(["gcc", "-O2", "-std=c99", "-fPIC", "-ffp-contract=off", "-shared", "-o", so,
                               os.path.join(os.path.dirname(os.path.abspath(__file__)), "map_cache_fill.c"), "-lm"])
        _fill_lib = C.CDLL(so)
        _fill_lib.map_cache_fill.restype = None
        _fill_lib.map_cache_fill.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, C.c_void_p]
    m = np.ascontiguousarray(map_u8, np.uint8)
    out = np.zeros(m.shape)
    _fill_lib.map_cache_fill(m.ctypes.data, m.shape[1], m.shape[0], float(res), float(max_dist), float(unreached), out.ctypes.data)
    return out


def _same(a, b):
    """same shape and the same bits in every cell"""
    a = np.ascontiguousarray(a, np.float64); b = np.ascontiguousarray(b, np.float64)
    return a.shape == b.shape and np.array_equal(a.view(np.int64), b.view(np.int64))


def _bundled():
    g = np.load(os.path.join(GOLD, "bundled_maps.npz"))
    out = [(n, g[n + "/map"], float(g[n + "/param"][2])) for n in BUNDLED]
    out += [(n, m, float(e[n + "/param"][2])) for n, m, e in _extra_maps()]
    return out


def _batch(lsdb, ctx, maps, **kw):
    b = lsdb.Batch(ctx, [(m.shape[1], m.shape[0]) for m in maps], **kw)
    b.upload(maps)
    return b


def _mixed_maps(seed=11):
    """~64 seeded maps: every degenerate shape, walls on row 0 / column 0, blank and fully occupied maps, synthetic grids"""
    rng = np.random.default_rng(seed)
    shapes = [(1, 1), (1, 2), (2, 1), (1, 57), (57, 1), (1, 1000), (700, 1), (3, 3), (97, 61), (61, 97), (128, 128), (300, 200),
              (511, 257), (1024, 768)]
    while len(shapes) < 64:
        shapes.append((int(rng.integers(1, 400)), int(rng.integers(1, 400))))
    maps = []
    for k, (rows, cols) in enumerate(shapes):
        kind = k % 6
        if kind == 0 and rows >= 40 and cols >= 40:
            m = synth.occupancy_grid(cols, rows, seed=100 + k)
        elif kind == 1:
            m = np.zeros((rows, cols), np.uint8)                              # blank: every cell stays `unreached`
        elif kind == 2:
            m = np.ones((rows, cols), np.uint8)                               # fully occupied: every cell 0
        else:
            m = rng.choice(np.array([0, 1, 255], np.uint8), (rows, cols), p=[0.93, 0.02, 0.05])
            if kind == 3:
                m[0, :] = 1                                                   # a wall on row 0
            if kind == 4:
                m[:, 0] = 1                                                   # a wall on column 0
        maps.append(np.ascontiguousarray(m))
    res = rng.choice([0.025, 0.05, 0.1, 0.3, 1.5, 3.0], len(maps))           # 1.5 and 3.0 > max_dist for some: cell radius 0
    res[:6] = [0.05, 3.0, 0.025, 1.5, 0.1, 0.3]
    return maps, [float(r) for r in res]


# ---- host only ----

def test_fill_restatement_generalises_the_oracle_map_cache():
    for name, m, res in _bundled():
        assert _same(map_cache_fill(m, res, 1.0, 1.0), oraclebind.map_cache(m, res)), name
    m = synth.occupancy_grid(300, 200, seed=5)
    std = map_cache_fill(m, 0.05, 2.0, 2.0)
    far = map_cache_fill(m, 0.05, 2.0, 7.0)
    assert (far == 7.0).any() and _same(np.where(far == 7.0, 2.0, far), std)


def test_new_entry_points_refuse_null_handles(lsdb):
    L = lsdb.lib()
    res = np.array([0.05])
    assert L.lsdb_batch_map_caches(None, res.ctypes.data_as(C.c_void_p), 1.0, 1.0, None) == 2
    h = C.c_void_p()
    assert L.lsdb_fa_map_create_from_batch(None, 0, C.byref(h)) == 2 and not h.value


# ---- on the device ----

@pytest.mark.gpu
def test_bundled_maps_in_one_ragged_batch(lsdb, ctx):
    items = _bundled()
    b = _batch(lsdb, ctx, [m for _, m, _ in items])
    got = b.map_caches([r for _, _, r in items])
    for (name, m, res), c in zip(items, got):
        want = oraclebind.map_cache(m, res)
        assert _same(c, want), name
        assert _same(c, ctx.map_cache(m, res)), name
    b.close()


@pytest.mark.gpu
def test_seeded_mixed_maps_against_the_oracle(lsdb, ctx):
    maps, res = _mixed_maps()
    b = _batch(lsdb, ctx, maps, **ANY_SIZE)
    for max_dist in (1.0, 2.0):
        for unreached in (max_dist, 2.0):
            got = b.map_caches(res, max_dist=max_dist, unreached=unreached)
            for k, (m, r, c) in enumerate(zip(maps, res, got)):
                assert _same(c, map_cache_fill(m, r, max_dist, unreached)), (k, m.shape, r, max_dist, unreached)
            assert np.all(got[1] == unreached) and np.all(got[2] == 0.0)                 # blank / fully occupied
    b.close()


@pytest.mark.gpu
def test_grouping_order_and_run_do_not_change_anything(lsdb, ctx, monkeypatch):
    items = _bundled()
    maps = [m for _, m, _ in items] + [synth.occupancy_grid(c, r, seed=300 + k) for k, (c, r) in enumerate([(640, 480), (97, 61), (1200, 333), (64, 900)])]
    res = [r for _, _, r in items] + [0.05, 0.025, 0.1, 0.05]
    b = _batch(lsdb, ctx, maps, max_lines=1024)
    base = b.map_caches(res)
    cells = [m.size for m in maps]
    for budget in (1, sum(cells) // 3 + 7, max(cells) + 1):              # one map per group; an uneven split; groups up to the largest map
        monkeypatch.setenv("LSDB_MC_GROUP_CELLS", str(budget))
        assert all(_same(a, c) for a, c in zip(b.map_caches(res), base)), budget
    monkeypatch.delenv("LSDB_MC_GROUP_CELLS")
    rb = _batch(lsdb, ctx, maps[::-1], max_lines=1024)                  # the order of the maps in the batch
    assert all(_same(a, c) for a, c in zip(rb.map_caches(res[::-1]), base[::-1]))
    rb.close()
    b.run()                                                              # before lsdb_batch_run (above) and after it
    t0 = b.download(want_rects=True)
    assert all(_same(a, c) for a, c in zip(b.map_caches(res), base))
    t1 = b.download(want_rects=True)                                     # the segment tables are untouched by the brush fire
    assert np.array_equal(t0["counts"], t1["counts"]) and t0["counts"].sum() > 0
    for i in range(len(maps)):
        assert t0["lines"][i].tobytes() == t1["lines"][i].tobytes() and t0["rects"][i].tobytes() == t1["rects"][i].tobytes()
    b.close()


@pytest.mark.gpu
def test_scan_rasters(lsdb, ctx):
    g = np.load(os.path.join(GOLD, "lidar_frames.npz"))
    mp = g["map_param"]
    sweeps = []
    for f in range(24):
        r, a = g[f"f{f}/ranges"], g[f"f{f}/angles"]
        keep = np.isfinite(r)
        sweeps.append((r[keep], a[keep]))
    info = ctx.feature_scan_info(mp[2], mp[3], mp[4], sweeps)
    b = lsdb.Batch(ctx, [(int(i["im_cols"]), int(i["im_rows"])) for i in info], max_lines=512)
    b.upload_scan_rasters(mp[2], mp[3], mp[4], sweeps)
    got = b.map_caches(float(mp[2]))
    host = ctx.feature_scan(mp[2], mp[3], mp[4], sweeps, want_rasters=True)
    for f, (o, c) in enumerate(zip(host, got)):
        occ = (o["line_im"] == 255).astype(np.uint8)
        assert occ.any() and _same(c, oraclebind.map_cache(occ, float(mp[2]))), f
    b.close()


def _fa_frames():
    g = np.load(os.path.join(GOLD, "fa_frames.npz"))
    return [dict(scan_lines=g[f"f{f}/scan_lines"], pts=g[f"f{f}/pts"], lidar_pose=g[f"f{f}/lidar_pose"], last_pose=g[f"f{f}/last_pose"])
            for f in range(int(g["n_frames"]))]


def _legacy_frames():
    g = np.load(os.path.join(GOLD, "fa_legacy.npz"))
    return g, [dict(scan_lines=g[f"f{f}/scan_lines"], lidar_pos=g[f"f{f}/lidar_pos"], ranges=g[f"f{f}/ranges"], angles=g[f"f{f}/angles"])
               for f in range(int(g["n_frames"]))]


@pytest.mark.gpu
def test_association_maps_from_the_batch(lsdb, ctx):
    items = _bundled()
    i = 0                                                                 # mapValue, the map of the association fixtures
    res = [r for _, _, r in items]
    b = _batch(lsdb, ctx, [m for _, m, _ in items])
    b.run()
    lines = b.download()["lines"]
    frames = _fa_frames()

    caches = b.map_caches(res)                                            # unreached = max_dist: the current source
    fb = lsdb.FaMap.from_batch(b, i)
    fh = lsdb.FaMap(ctx, caches[i], lines[i])
    assert fb.n_lines == fh.n_lines == len(lines[i]) > 0
    assert fb.estimate(frames).tobytes() == fh.estimate(frames).tobytes()
    assert fb.score(frames).tobytes() == fh.score(frames).tobytes()
    kb, nb = fb.score_kept(frames); kh, nh = fh.score_kept(frames)
    assert nb == nh and kb.tobytes() == kh.tobytes()

    gl, lf = _legacy_frames()                                             # unreached = 2: the catkin snapshot's three-argument flavour
    caches2 = b.map_caches(res, max_dist=1.0, unreached=2.0)
    assert _same(caches2[i], map_cache_fill(items[i][1], res[i], 1.0, 2.0))
    lb = lsdb.FaMap.from_batch(b, i)
    lh = lsdb.FaMap(ctx, caches2[i], lines[i])
    eb, pb, cb = lb.legacy_frames(lf, float(gl["resol"]), gl["ori"], want_pose_all=True)
    eh, ph, ch = lh.legacy_frames(lf, float(gl["resol"]), gl["ori"], want_pose_all=True)
    assert eb.tobytes() == eh.tobytes() and pb.tobytes() == ph.tobytes() and np.array_equal(cb, ch)
    for f in range(len(lf)):
        if eb[f]["n_cols"]:                                               # the goldens' estimates (their scores used a different cache)
            assert np.array_equal(eb[f]["estimate_pose"], gl[f"f{f}/est"], equal_nan=True)
            assert np.array_equal(eb[f]["estimate_pose_realworld"], gl[f"f{f}/est_real"], equal_nan=True)
        if not len(lf[f]["ranges"]):
            continue
        one = lb.legacy(lf[f]["scan_lines"], float(gl["resol"]), gl["ori"], lf[f]["lidar_pos"], lf[f]["ranges"], lf[f]["angles"])
        assert one[0].tobytes() == pb[cb[f]:cb[f + 1]].tobytes()

    b.close()                                                             # the FaMaps own their copies
    assert fb.estimate(frames).tobytes() == fh.estimate(frames).tobytes()
    assert lb.legacy_frames(lf, float(gl["resol"]), gl["ori"])[0].tobytes() == eb.tobytes()
    g = np.load(os.path.join(GOLD, "lidar_frames.npz"))
    mp = g["map_param"]
    sweeps = [(g[f"f{f}/ranges"][np.isfinite(g[f"f{f}/ranges"])], g[f"f{f}/angles"][np.isfinite(g[f"f{f}/ranges"])]) for f in range(6)]
    ib, sb = fb.scan_estimate(mp[2], mp[3], mp[4], sweeps)
    ih, sh = fh.scan_estimate(mp[2], mp[3], mp[4], sweeps)
    assert ib.tobytes() == ih.tobytes() and sb.tobytes() == sh.tobytes()
    for x in (fb, fh, lb, lh):
        x.close()


@pytest.mark.gpu
def test_argument_errors_write_nothing(lsdb, ctx):
    L = lsdb.lib()
    items = _bundled()[:3]
    maps = [m for _, m, _ in items]
    b = _batch(lsdb, ctx, maps)
    res = np.array([r for _, _, r in items])
    outs = [np.full(m.shape, -3.0) for m in maps]
    ptrs = (C.c_void_p * len(maps))(*[o.ctypes.data for o in outs])
    h = C.c_void_p()

    def valid():
        want = [oraclebind.map_cache(m, r) for m, r in zip(maps, res)]
        assert all(_same(c, w) for c, w in zip(b.map_caches(res), want))
        assert _same(ctx.map_cache(maps[0], res[0]), want[0])

    def rp(r):
        return np.ascontiguousarray(r, np.float64).ctypes.data_as(C.c_void_p)

    assert L.lsdb_fa_map_create_from_batch(b.h, 0, C.byref(h)) == 2 and not h.value          # before run, before map_caches
    b.run()
    assert L.lsdb_fa_map_create_from_batch(b.h, 0, C.byref(h)) == 2 and not h.value          # before map_caches
    bad_res = [None] + [rp(np.where(np.arange(len(maps)) == 1, v, res)) for v in (0.0, -0.05, np.nan, np.inf, -np.inf)]
    for r in bad_res:
        assert L.lsdb_batch_map_caches(b.h, r, 1.0, 1.0, ptrs) == 2
        assert all((o == -3.0).all() for o in outs)
        valid()
    for md in (-1.0, -1e-300, np.nan, -np.inf):
        assert L.lsdb_batch_map_caches(b.h, rp(res), md, 1.0, ptrs) == 2
        assert all((o == -3.0).all() for o in outs)
        valid()
    for i in (-1, len(maps), 1 << 30):
        assert L.lsdb_fa_map_create_from_batch(b.h, i, C.byref(h)) == 2 and not h.value
        valid()
    assert L.lsdb_fa_map_create_from_batch(b.h, 0, None) == 2
    assert L.lsdb_batch_map_caches(b.h, rp(res), 1.0, 1.0, ptrs) == 0                         # out pointers filled on success
    assert all(_same(o, oraclebind.map_cache(m, r)) for o, m, r in zip(outs, maps, res))
    fm = lsdb.FaMap.from_batch(b, 2)
    fm.close()
    b.close()
    wide = lsdb.Batch(ctx, [(65536, 4), (4, 4)], max_lines=16)                               # more than 65535 columns
    wide.upload([np.zeros((4, 65536), np.uint8), np.ones((4, 4), np.uint8)])
    with pytest.raises(lsdb.LsdbError, match="65535"):
        wide.map_caches(0.05)
    wide.close()
    tall = lsdb.Batch(ctx, [(4, 65536)], max_lines=16)
    tall.upload([np.zeros((65536, 4), np.uint8)])
    with pytest.raises(lsdb.LsdbError, match="65535"):
        tall.map_caches(0.05)
    tall.close()
    valid_b = _batch(lsdb, ctx, [np.ones((4, 4), np.uint8)])
    assert _same(valid_b.map_caches(0.05)[0], np.zeros((4, 4)))
    valid_b.close()


@pytest.mark.gpu
def test_scale(lsdb, ctx):
    n, size = 16, 4096
    maps = [synth.occupancy_grid(size, size, seed=1000 + k) for k in range(n)]
    b = _batch(lsdb, ctx, maps, max_lines=4096)
    res = np.full(n, 0.05)
    sample = sorted(np.random.default_rng(3).choice(n, 4, replace=False).tolist())
    outs = {k: np.empty((size, size)) for k in sample}
    ptrs = (C.c_void_p * n)(*[outs[k].ctypes.data if k in outs else None for k in range(n)])
    ctx.check(lsdb.lib().lsdb_batch_map_caches(b.h, res.ctypes.data_as(C.c_void_p), 1.0, 1.0, ptrs), "lsdb_batch_map_caches")
    for k in sample:
        assert _same(outs[k], oraclebind.map_cache(maps[k], 0.05)), k
    b.close()
    del maps, outs
    big = synth.occupancy_grid(8192, 8192, seed=5000)
    b = _batch(lsdb, ctx, [big], max_lines=16384)
    assert _same(b.map_caches(0.025)[0], ctx.map_cache(big, 0.025))
    b.close()
