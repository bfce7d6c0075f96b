"""Parity of the CUDA scan front-end (lsdb_feature_scan_frames = myrdp::FeatureScan, LSD/myRDP.cpp:9-185) with the
reference's golden outputs and the oracle: everything bit-exact (NaN == NaN for the intercept of vertical pieces)."""
import os

import numpy as np
import pytest

import oraclebind
import synth

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
MP = [1377, 428, 0.05, -41.4, -9.8]


def _lines10(rec):
    return np.stack([rec[k].astype(np.float64) for k in ("k", "b", "dx", "dy", "x1", "y1", "x2", "y2", "len", "orient")], 1)


def _check(got, want, tag):
    assert tuple(got["size"]) == tuple(want["size"]), tag
    assert np.array_equal(_lines10(got["lines"]), want["lines"], equal_nan=True), tag
    assert np.array_equal(got["pts"], np.asarray(want["pts"], np.float64)), tag
    assert np.array_equal(got["lidar_pos"], want["lidar_pos"]), tag
    if "line_im" in got and "line_im" in want:
        assert np.array_equal(got["line_im"], want["line_im"]), tag


def _finite(r, a):
    keep = np.isfinite(r)
    return r[keep], a[keep]


def test_golden_lidar_frames_one_batch(lsdb, ctx):
    """87 frames of the bundled Lidar.txt files in ONE call against the reference's own FeatureScan output"""
    g = np.load(os.path.join(GOLD, "lidar_frames.npz"))
    nf = int(g["n_frames"])
    mp = g["map_param"]
    frames = [_finite(g[f"f{f}/ranges"], g[f"f{f}/angles"]) for f in range(nf)]
    out = ctx.feature_scan(mp[2], mp[3], mp[4], frames, want_rasters=True)
    assert len(out) == nf
    for f in range(nf):
        want = dict(lines=g[f"f{f}/lines"], pts=g[f"f{f}/pts"], lidar_pos=g[f"f{f}/lidar_pos"], size=g[f"f{f}/size"])
        _check(out[f], want, f)
        im = np.zeros(out[f]["line_im"].shape, np.uint8)               # FS.lineIm = 255 exactly at scanImPoint
        im[g[f"f{f}/pts"][:, 1], g[f"f{f}/pts"][:, 0]] = 255
        assert np.array_equal(out[f]["line_im"], im), f
    # the golden association fixture starts from the same frames: its scan lines / points are reproduced too
    ga = np.load(os.path.join(GOLD, "fa_frames.npz"))
    for f in range(int(ga["n_frames"])):
        assert np.array_equal(_lines10(out[f]["lines"]), ga[f"f{f}/scan_lines"], equal_nan=True)
        assert np.array_equal(out[f]["pts"], ga[f"f{f}/pts"])


@pytest.mark.parametrize("n_beams", [360, 720, 97])
def test_synthetic_frames_vs_oracle(lsdb, ctx, n_beams):
    frames = [synth.lidar_frame(4000 + s, n_beams=n_beams) for s in range(64)]
    frames = [f for f in frames if len(f[0])]
    out = ctx.feature_scan(MP[2], MP[3], MP[4], frames, want_rasters=True)
    nl = 0
    for f, (r, a) in enumerate(frames):
        _check(out[f], oraclebind.feature_scan(MP, r, a), (n_beams, f))
        nl += len(out[f]["lines"])
    assert nl > len(frames)


def test_ragged_and_tiny_frames(lsdb, ctx):
    """frames of 1, 2, 3, 5 beams next to full sweeps; a sweep whose last beam joins the first (cluster 0 wraps)"""
    rng = np.random.default_rng(7)
    full = synth.lidar_frame(11)
    frames = [(np.array([2.0]), np.array([0.1])), (np.array([2.0, 2.01]), np.array([0.1, 0.12])), full,
              (np.array([1.0, 1.0, 1.0]), np.array([0.0, 0.01, 0.02])),
              (rng.uniform(0.5, 3, 5), np.sort(rng.uniform(-3, 3, 5))), synth.lidar_frame(12, dropout=0.0),
              (np.full(360, 3.0), -3.12414 + np.arange(360) * 0.0174532)]            # a circle: one cluster, never broken
    out = ctx.feature_scan(MP[2], MP[3], MP[4], frames, want_rasters=True)
    for f, (r, a) in enumerate(frames):
        _check(out[f], oraclebind.feature_scan(MP, r, a), f)
    # a batch in which no frame yields a line: empty outputs, no launch of the lines kernel
    none = ctx.feature_scan(MP[2], MP[3], MP[4], [frames[-1], frames[0]], want_rasters=True)
    assert [len(o["lines"]) for o in none] == [0, 0] and [len(o["pts"]) for o in none] == [0, 0]
    _check(none[0], oraclebind.feature_scan(MP, *frames[-1]), "circle")


def test_randomised_sweeps_vs_oracle(lsdb, ctx):
    """1 500 sweeps of random length (1..1500 beams), room, noise and dropout in one ragged call; degenerate beams mixed in
    (repeated points -> 0/0 slopes, exactly axis-aligned pieces, far returns beyond 9 m where the split threshold scales)"""
    rng = np.random.default_rng(99)
    frames = []
    for s in range(1500):
        nb = int(rng.integers(1, 1500)) if s % 3 else int(rng.integers(1, 40))
        r, a = synth.lidar_frame(7000 + s, n_beams=nb, dropout=float(rng.uniform(0, 0.4)), noise=float(rng.choice([0.0, 0.002, 0.02])))
        if len(r) == 0:
            r, a = np.array([1.0]), np.array([0.0])
        if s % 7 == 0 and len(r) > 8:                       # repeated returns
            r[3:6] = r[3]; a[3:6] = a[3]
        if s % 11 == 0:                                     # a far wall
            r = r * 3.0
        frames.append((r, a))
    # exactly axis-aligned walls in grid coordinates: x = const / y = const
    t = np.linspace(-1.0, 1.0, 120)
    frames.append((np.hypot(2.0, t * 2), np.arctan2(t * 2, 2.0)))
    frames.append((np.hypot(t * 2, 1.5), np.arctan2(1.5, t * 2)))
    out = ctx.feature_scan(0.05, -30.0, -12.0, frames, want_rasters=True)
    nl = 0
    for f, (r, a) in enumerate(frames):
        _check(out[f], oraclebind.feature_scan([0, 0, 0.05, -30.0, -12.0], r, a), f)
        nl += len(out[f]["lines"])
    assert nl > 3000


def test_non_default_parameters(lsdb, ctx):
    frames = [synth.lidar_frame(900 + s) for s in range(16)]
    for prm in (dict(least_point=1, thre_line=0.03, least_dist_m=0.2), dict(least_point=8, thre_line=0.2, least_dist_m=1.0),
                dict(least_point=3, thre_line=0.08, least_dist_m=0.0)):
        out = ctx.feature_scan(0.03, -20.0, -7.5, frames, want_rasters=True, **prm)
        for f, (r, a) in enumerate(frames):
            _check(out[f], oraclebind.feature_scan([0, 0, 0.03, -20.0, -7.5], r, a, **prm), (prm, f))


def test_error_paths(lsdb, ctx):
    r, a = synth.lidar_frame(1)
    with pytest.raises(lsdb.LsdbError, match="ARG"):
        ctx.feature_scan(MP[2], MP[3], MP[4], [(r, a), (np.zeros(0), np.zeros(0))])        # a frame without beams
    r2 = r.copy(); r2[3] = np.inf
    with pytest.raises(lsdb.LsdbError, match="not finite"):
        ctx.feature_scan(MP[2], MP[3], MP[4], [(r2, a)])
    with pytest.raises(lsdb.LsdbError, match="ARG"):
        ctx.feature_scan(0.0, MP[3], MP[4], [(r, a)])
    assert ctx.feature_scan(MP[2], MP[3], MP[4], []) == []
    # capacity: the sizing query fills the offsets, the real call refuses short buffers
    import ctypes as C
    L = lsdb.lib()
    boff = np.array([0, len(r)], np.int32); info = np.zeros(1, lsdb.SCAN_INFO_DTYPE)
    loff = np.zeros(2, np.int32); poff = np.zeros(2, np.int32); ioff = np.zeros(2, np.int64)
    prm = lsdb._RdpParams(3, 0.08, 0.5)
    p = lambda x: x.ctypes.data_as(C.c_void_p)  # noqa: E731
    args = (ctx.h, MP[2], MP[3], MP[4], C.byref(prm), 1, p(r), p(a), p(boff), p(info))
    assert L.lsdb_feature_scan_frames(*args, None, 0, p(loff), None, 0, p(poff), None, 0, p(ioff)) == 0
    assert loff[1] == info[0]["n_lines"] > 0 and poff[1] == info[0]["n_pts"] > 0 and ioff[1] == info[0]["im_cols"] * info[0]["im_rows"]
    lines = np.zeros(1, lsdb.LINE_DTYPE); pts = np.zeros((int(poff[1]), 2))
    assert L.lsdb_feature_scan_frames(*args, p(lines), 1, p(loff), p(pts), len(pts), p(poff), None, 0, p(ioff)) == 3   # LSDB_ERR_CAPACITY
    assert b"max_lines" in L.lsdb_last_error(ctx.h)


def test_angles_beyond_2_19_are_rejected_before_any_launch(lsdb, ctx):
    """A finite angle the device's sin / cos cannot reduce (|a| > LSDB_MAX_ANGLE = 2^19) is LSDB_ERR_ARG, found on the host
    before anything is launched or written; +-2^19 itself is accepted, and the context keeps working."""
    import ctypes as C
    L = lsdb.lib()
    r, a = synth.lidar_frame(1)
    base = ctx.feature_scan(MP[2], MP[3], MP[4], [(r, a)])
    boff = np.array([0, len(r)], np.int32); prm = lsdb._RdpParams(3, 0.08, 0.5)
    p = lambda x: x.ctypes.data_as(C.c_void_p)  # noqa: E731
    for bad in (1e22, -1e22, 2.0 ** 19 + 2.0 ** -33, 1.7976931348623157e308):
        a2 = a.copy(); a2[7] = bad
        info = np.frombuffer(b"\xab" * lsdb.SCAN_INFO_DTYPE.itemsize, lsdb.SCAN_INFO_DTYPE).copy()
        loff = np.zeros(2, np.int32); poff = np.zeros(2, np.int32); ioff = np.zeros(2, np.int64)
        assert L.lsdb_feature_scan_frames(ctx.h, MP[2], MP[3], MP[4], C.byref(prm), 1, p(r), p(a2), p(boff), p(info),
                                          None, 0, p(loff), None, 0, p(poff), None, 0, p(ioff)) == 2
        assert b"angle of beam 7" in L.lsdb_last_error(ctx.h)
        assert (info.view(np.uint8) == 0xAB).all()                        # nothing ran: the sizing query's output is untouched
        with pytest.raises(lsdb.LsdbError, match="ARG"):
            ctx.feature_scan(MP[2], MP[3], MP[4], [(r, a2)])
    for edge in (2.0 ** 19, -(2.0 ** 19)):
        a3 = a.copy(); a3[7] = edge
        assert len(ctx.feature_scan(MP[2], MP[3], MP[4], [(r, a3)])) == 1
    again = ctx.feature_scan(MP[2], MP[3], MP[4], [(r, a)])
    assert np.array_equal(lsdb.lines_to_array(again[0]["lines"]), lsdb.lines_to_array(base[0]["lines"]), equal_nan=True)
    assert np.array_equal(again[0]["pts"], base[0]["pts"])


def test_scan_to_estimate_chain(lsdb, ctx):
    """lidar frames -> device FeatureScan -> device scoring + reduction: the same estimates as from the reference's
    scan lines / points of the golden association fixture"""
    g = np.load(os.path.join(GOLD, "lidar_frames.npz"))
    ga = np.load(os.path.join(GOLD, "fa_frames.npz"))
    gm = np.load(os.path.join(GOLD, "bundled_maps.npz"))
    mp = g["map_param"]
    nf = int(ga["n_frames"])
    out = ctx.feature_scan(mp[2], mp[3], mp[4], [_finite(g[f"f{f}/ranges"], g[f"f{f}/angles"]) for f in range(nf)])
    mc = ctx.map_cache(gm["mapValue/map"], float(gm["mapValue/param"][2]))
    fm = lsdb.FaMap(ctx, mc, ga["map_lines"])
    mine = fm.estimate([dict(scan_lines=o["lines"], pts=o["pts"], lidar_pose=np.rint(o["lidar_pos"]), last_pose=ga[f"f{f}/last_pose"])
                        for f, o in enumerate(out)])
    ref = fm.estimate([dict(scan_lines=ga[f"f{f}/scan_lines"], pts=ga[f"f{f}/pts"], lidar_pose=ga[f"f{f}/lidar_pose"],
                            last_pose=ga[f"f{f}/last_pose"]) for f in range(nf)])
    assert mine.tobytes() == ref.tobytes()
    assert int((mine["n_kept"] > 0).sum()) >= 6
    # the same in ONE call with the raster samples resident on the device; gated frames included
    sweeps = [_finite(g[f"f{f}/ranges"], g[f"f{f}/angles"]) for f in range(nf)]
    last = np.stack([ga[f"f{f}/last_pose"] for f in range(nf)])
    info, est = fm.scan_estimate(mp[2], mp[3], mp[4], sweeps, last_pose=last)
    assert est.tobytes() == ref.tobytes()
    assert np.array_equal(info["n_lines"], [len(o["lines"]) for o in out]) and np.array_equal(info["n_pts"], [len(o["pts"]) for o in out])
    # frames without any line (a circle) and a large batch
    many = sweeps * 40 + [(np.full(360, 3.0), -3.12414 + np.arange(360) * 0.0174532)]
    info2, est2 = fm.scan_estimate(mp[2], mp[3], mp[4], many)
    one = fm.estimate([dict(scan_lines=o["lines"], pts=o["pts"], lidar_pose=np.rint(o["lidar_pos"]), last_pose=[-1.0, -1.0, 0.0]) for o in out])
    assert est2[:-1].tobytes() == np.tile(one, 40).tobytes()
    assert info2[-1]["n_lines"] == 0 and est2[-1]["n_kept"] == 0
    info3, est3 = fm.scan_estimate(mp[2], mp[3], mp[4], [many[-1]])             # nothing to score at all
    assert info3[0]["n_lines"] == 0 and est3[0]["n_hyp"] == 0 and est3[0]["n_kept"] == 0
    fm.close()


def test_scan_rasters_straight_into_a_batch(lsdb, ctx):
    """lsdb_batch_upload_scan_rasters: sweeps -> rasters on the device -> LSD, equal to rasterising on the host (FeatureScan
    lineIm > 0 as an occupancy grid) and uploading; the golden LSD-of-scan segment tables of the reference on top"""
    g = np.load(os.path.join(GOLD, "lidar_frames.npz"))
    ga = np.load(os.path.join(GOLD, "fa_frames.npz"))
    mp = g["map_param"]
    nf = 24
    sweeps = [_finite(g[f"f{f}/ranges"], g[f"f{f}/angles"]) for f in range(nf)]
    info = ctx.feature_scan_info(mp[2], mp[3], mp[4], sweeps)
    sizes = [(int(i["im_cols"]), int(i["im_rows"])) for i in info]
    b = lsdb.Batch(ctx, sizes, max_lines=512)
    info2 = b.upload_scan_rasters(mp[2], mp[3], mp[4], sweeps)
    assert info2.tobytes() == info.tobytes()
    b.run(); dev = b.download()
    host = ctx.feature_scan(mp[2], mp[3], mp[4], sweeps, want_rasters=True)
    b2 = lsdb.Batch(ctx, sizes, max_lines=512)
    b2.upload([np.ascontiguousarray((o["line_im"] > 0).astype(np.uint8)) for o in host]); b2.run(); ref = b2.download()
    assert np.array_equal(dev["counts"], ref["counts"]) and dev["counts"].sum() > nf
    for f in range(nf):
        n = int(dev["counts"][f])
        assert dev["lines"][f][:n].tobytes() == ref["lines"][f][:n].tobytes()
    for f in range(int(ga["n_frames"])):                    # frames 0..11 of the association fixture are the first golden sweeps
        want = ga[f"f{f}/scan_lsd_lines"]
        got = lsdb.lines_to_array(dev["lines"][f][:int(dev["counts"][f])])
        assert got.shape == want.shape and np.allclose(got, want, rtol=1e-9, atol=1e-9, equal_nan=True)
    # a batch of the wrong shape is refused
    bad = lsdb.Batch(ctx, [(s[0] + 1, s[1]) for s in sizes], max_lines=64)
    with pytest.raises(lsdb.LsdbError, match="does not have the size"):
        bad.upload_scan_rasters(mp[2], mp[3], mp[4], sweeps)
    for x in (b, b2, bad):
        x.close()
