"""Parity of the CUDA association scoring (lsdb_fa_score) with the reference's golden scores and the oracle:
poses bit-exact against the oracle, scores within the 1e-6 contract."""
import os

import numpy as np
import pytest

import oraclebind
import synth

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_fa_golden_frames_batched(lsdb, ctx):
    g = np.load(os.path.join(GOLD, "fa_frames.npz"))
    gm = np.load(os.path.join(GOLD, "bundled_maps.npz"))
    mc = oraclebind.map_cache(gm["mapValue/map"], float(gm["mapValue/param"][2]))
    nf = int(g["n_frames"])
    frames = [dict(scan_lines=g[f"f{f}/scan_lines"], pts=g[f"f{f}/pts"], lidar_pose=g[f"f{f}/lidar_pose"],
                   last_pose=g[f"f{f}/last_pose"]) for f in range(nf)]
    fm = lsdb.FaMap(ctx, mc, g["map_lines"])
    hyp = fm.score(frames)                     # all frames in ONE launch
    pos = 0
    for f in range(nf):
        idx, want = g[f"f{f}/idx"], g[f"f{f}/val"]
        h = hyp[pos:pos + len(idx)]; pos += len(idx)
        assert np.all(h["frame"] == f)
        assert np.array_equal(np.stack([h["i_scan"], h["i_map"], h["i_pair"]], 1), idx)
        fin = np.isfinite(want[:, 3])
        assert np.array_equal(np.isfinite(h["score"]), fin)
        assert np.allclose(h["score"][fin], want[fin, 3], rtol=1e-6, atol=0)          # vs unmodified reference
        for j, k in enumerate(("x", "y", "ang")):
            assert np.allclose(h[k], want[:, j], rtol=1e-9, atol=1e-9)
        oi, ov = oraclebind.fa_scores(frames[f]["scan_lines"], g["map_lines"], frames[f]["pts"], mc,
                                      frames[f]["lidar_pose"], frames[f]["last_pose"])
        assert np.array_equal(oi, idx)
        for j, k in enumerate(("x", "y", "ang")):
            assert np.array_equal(h[k], ov[:, j])                                      # poses: same bits as the oracle
        assert np.allclose(h["score"][fin], ov[fin, 3], rtol=1e-12, atol=0)            # sums differ only by reassociation
    assert pos == len(hyp)
    assert fm.last_ms() > 0
    fm.close()


def test_fa_edge_cases(lsdb, ctx):
    m = synth.occupancy_grid(500, 400, seed=31)
    o = oraclebind.lsd(m)
    mc = oraclebind.map_cache(m, 0.05)
    fm = lsdb.FaMap(ctx, mc, o["lines"])
    fr = synth.fake_scan_frame(m, o["lines"], seed=4)
    empty = dict(scan_lines=np.zeros((0, 10)), pts=np.zeros((0, 2)), lidar_pose=[0, 0], last_pose=[-1, -1, 0])
    short = dict(fr); short["scan_lines"] = fr["scan_lines"].copy(); short["scan_lines"][:, 8] = 10.0  # all < ignoreScanLength
    nopts = dict(fr); nopts["pts"] = np.zeros((0, 2))
    gated = dict(fr); gated["last_pose"] = np.array([1e6, 1e6, 0.0])
    hyp = fm.score([empty, short, fr, nopts, gated])
    assert not np.any(hyp["frame"] <= 1)
    for f, frame in [(2, fr), (3, nopts), (4, gated)]:
        h = hyp[hyp["frame"] == f]
        oi, ov = oraclebind.fa_scores(frame["scan_lines"], o["lines"], frame["pts"], mc, frame["lidar_pose"], frame["last_pose"])
        assert len(h) == len(oi) and len(h) > 0
        fin = np.isfinite(ov[:, 3])
        assert np.array_equal(np.isfinite(h["score"]), fin)
        assert np.allclose(h["score"][fin], ov[fin, 3], rtol=1e-9)
        if f != 2:
            assert not fin.any()
    assert fm.score([]).shape == (0,)
    fm.close()


def test_map_cache_device_matches_reference(lsdb, ctx):
    """lsdb_map_cache == mylsd::createMapCache cell for cell (FIFO tie-breaking between sources included): bundled maps
    against the oracle restatement, which tests/test_oracle.py pins to the unmodified reference."""
    gm = np.load(os.path.join(GOLD, "bundled_maps.npz"))
    for name in ("mapValue", "mapValue_map1"):
        m = gm[name + "/map"]; res = float(gm[name + "/param"][2])
        got = ctx.map_cache(m, res)
        assert np.array_equal(got, oraclebind.map_cache(m, res)), name
    for shape, seed, res in (((300, 200), 5, 0.05), ((97, 61), 6, 0.025), ((64, 64), 8, 0.3)):
        m = synth.occupancy_grid(shape[0], shape[1], seed=seed)
        assert np.array_equal(ctx.map_cache(m, res), oraclebind.map_cache(m, res))
    blank = np.zeros((40, 50), np.uint8)                       # no source: every cell keeps z_occ_max_dis
    assert np.all(ctx.map_cache(blank, 0.05) == 1.0)
    full = np.ones((30, 30), np.uint8)
    assert np.all(ctx.map_cache(full, 0.05) == 0.0)


def test_fa_estimate_matches_host_reduction(lsdb, ctx):
    """lsdb_fa_estimate_frames (device reduction, LSD/myFA.cpp:65-171 minus ukf) == the same reduction done on the host
    from lsdb_fa_score's hypotheses, bit for bit: keep score < 3, stable ascending sort, best, 1/score^2 weighted mean
    accumulated in that order."""
    g = np.load(os.path.join(GOLD, "fa_frames.npz"))
    gm = np.load(os.path.join(GOLD, "bundled_maps.npz"))
    mc = oraclebind.map_cache(gm["mapValue/map"], float(gm["mapValue/param"][2]))
    nf = int(g["n_frames"])
    frames = [dict(scan_lines=g[f"f{f}/scan_lines"], pts=g[f"f{f}/pts"], lidar_pose=g[f"f{f}/lidar_pose"],
                   last_pose=[-1.0, -1.0, 0.0]) for f in range(nf)]
    frames.append(dict(scan_lines=np.zeros((0, 10)), pts=np.zeros((0, 2)), lidar_pose=[0, 0], last_pose=[-1, -1, 0]))   # no hypotheses
    frames.append(dict(frames[0], last_pose=[1e6, 1e6, 0.0]))                                                            # everything gated out
    # a frame that keeps more hypotheses than the device sort holds (2048): its scan lines repeated — the reduction of that
    # frame then runs on the host from the device's scores (api.cu: est.n_kept < 0), and must give the same numbers
    big = max(range(nf), key=lambda f: int((g[f"f{f}/val"][:, 3] < 3).sum()))
    reps = 2048 // max(int((g[f"f{big}/val"][:, 3] < 3).sum()), 1) + 2
    frames.append(dict(frames[big], scan_lines=np.tile(frames[big]["scan_lines"], (reps, 1))))
    fm = lsdb.FaMap(ctx, mc, g["map_lines"])
    hyp = fm.score(frames)
    est = fm.estimate(frames)
    assert len(est) == len(frames)
    assert int((hyp[hyp["frame"] == len(frames) - 1]["score"] < 3).sum()) > 2048
    some = 0
    for f in range(len(frames)):
        h = hyp[hyp["frame"] == f]
        assert est["n_hyp"][f] == len(h)
        kept = h[h["score"] < 3]
        assert est["n_kept"][f] == len(kept)
        if len(kept) == 0:
            continue
        kept = kept[np.argsort(kept["score"], kind="stable")]
        assert (est["best_x"][f], est["best_y"][f], est["best_ang"][f], est["best_score"][f]) == \
            (kept["x"][0], kept["y"][0], kept["ang"][0], kept["score"][0])
        sx = sy = sa = sw = 0.0
        for k in range(len(kept)):                       # sequential, like the reference's loop
            w = 1.0 / (kept["score"][k] * kept["score"][k])
            sx += kept["x"][k] * w; sy += kept["y"][k] * w; sa += kept["ang"][k] * w; sw += w
        assert est["mean_x"][f] == sx / sw and est["mean_y"][f] == sy / sw and est["mean_ang"][f] == sa / sw
        assert est["mean_score"][f] == 1.0 / np.sqrt(sw / len(kept))
        some += 1
    assert some >= 6
    fm.close()


def test_kept_hypotheses_equal_the_filtered_full_table(lsdb, ctx):
    """lsdb_fa_score_kept (device pair filter + ordered compaction of score < 3, LSD/myFA.cpp:261-265) returns exactly the rows of
    lsdb_fa_score with score < 3, in the same order, and reports how many hypotheses were scored; a table that is too small is
    an error, not a truncation."""
    gold_fa = np.load(os.path.join(GOLD, "fa_frames.npz"))
    gold_maps = np.load(os.path.join(GOLD, "bundled_maps.npz"))
    mc = ctx.map_cache(gold_maps["mapValue/map"], float(gold_maps["mapValue/param"][2]))
    frames = [dict(scan_lines=gold_fa[f"f{f}/scan_lines"], pts=gold_fa[f"f{f}/pts"], lidar_pose=gold_fa[f"f{f}/lidar_pose"],
                   last_pose=[-1.0, -1.0, 0.0]) for f in range(int(gold_fa["n_frames"]))] * 3
    frames.insert(5, dict(scan_lines=np.zeros((0, 10)), pts=np.zeros((0, 2)), lidar_pose=[0.0, 0.0], last_pose=[-1.0, -1.0, 0.0]))   # an empty frame
    fm = lsdb.FaMap(ctx, mc, gold_fa["map_lines"])
    full = fm.score(frames)
    kept, n_hyp = fm.score_kept(fm.pack(frames))
    want = full[full["score"] < 3.0]
    assert n_hyp == len(full) and len(kept) == len(want) > 0
    for k in ("frame", "i_scan", "i_map", "i_pair", "x", "y", "ang", "score"):
        assert np.array_equal(kept[k], want[k]), k
    table = np.zeros(len(want) + 7, lsdb.HYP_DTYPE)                      # a caller-owned table: the result is a view of it
    mine, _ = fm.score_kept(frames, out=table)
    assert mine.base is table and len(mine) == len(want) and np.array_equal(mine, want)
    with pytest.raises(lsdb.LsdbError, match="CAPACITY"):
        fm.score_kept(frames, out=table[:len(want) - 1])
    kept5, _ = fm.score_kept(frames, keep_below=5.0)
    assert len(kept5) == int((full["score"] < 5.0).sum())
    with pytest.raises(lsdb.LsdbError, match="CAPACITY"):
        fm.score_kept(frames, max_kept=max(len(want) - 1, 1))
    none, nh0 = fm.score_kept([frames[5]])
    assert len(none) == 0 and nh0 == 0
    fm.close()


def _bits_equal(a, b):
    """same shape and the same bits, a NaN on both sides counting as equal (so -0 differs from +0)"""
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return a.shape == b.shape and np.array_equal(np.isnan(a), np.isnan(b)) and \
        np.array_equal(a[~np.isnan(a)].view(np.int64), b[~np.isnan(b)].view(np.int64))


def _degenerate(lines):
    """copies of line records (the lengths kept, so the length filters still pair them) with degenerate end points: vertical with
    dx = +-0, dx = +-5e-324 / 1e-310 / 1e-300 under dy = 1 (|dy/dx| overflows or reaches 1e300, where atan used to overflow on the
    host), horizontal (dy = 0), zero length"""
    out = []
    for ln in lines:
        for x1, x2, dy in [(0.0, 0.0, 1.0), (0.0, -0.0, 1.0), (-0.0, 0.0, -1.0), (3.0, 3.0, -2.0)] + \
                          [(0.0, s * d, 1.0) for d in (5e-324, 1e-310, 1e-300) for s in (1.0, -1.0)] + \
                          [(12.0, 15.0, 0.0), (15.0, 12.0, 0.0), (7.0, 7.0, 0.0)]:
            r = np.array(ln, np.float64)
            r[4], r[6], r[7] = x1, x2, r[5] + dy
            out.append(r)
    return np.array(out)


def test_degenerate_line_geometry(lsdb, ctx):
    """Vertical, horizontal, nearly vertical (|dy/dx| up to 2^1074) and zero-length scan and map lines through both association
    paths: lsdb_fa_score's poses and lsdb_fa_legacy_frames' records have the oracle's bits."""
    m = synth.occupancy_grid(500, 400, seed=31)
    o = oraclebind.lsd(m)
    mc = oraclebind.map_cache(m, 0.05)
    fr = synth.fake_scan_frame(m, o["lines"], seed=4)
    ml = np.concatenate([o["lines"], _degenerate(o["lines"][:3])])
    sl = np.concatenate([fr["scan_lines"][:2], _degenerate(fr["scan_lines"][:3])])
    fm = lsdb.FaMap(ctx, mc, ml)
    frames = [dict(fr, scan_lines=sl), dict(fr, scan_lines=sl, last_pose=np.array([-1.0, -1.0, 0.0]))]
    hyp = fm.score(frames)
    n_deg = 0
    for f, frame in enumerate(frames):
        h = hyp[hyp["frame"] == f]
        oi, ov = oraclebind.fa_scores(frame["scan_lines"], ml, frame["pts"], mc, frame["lidar_pose"], frame["last_pose"])
        assert np.array_equal(np.stack([h["i_scan"], h["i_map"], h["i_pair"]], 1), oi)
        for j, k in enumerate(("x", "y", "ang")):
            assert _bits_equal(h[k], ov[:, j]), k
        fin = np.isfinite(ov[:, 3])
        assert np.array_equal(np.isfinite(h["score"]), fin)
        assert np.allclose(h["score"][fin], ov[fin, 3], rtol=1e-9)
        n_deg += int(((oi[:, 0] >= 2) | (oi[:, 1] >= len(o["lines"]))).sum())
    assert n_deg > 100                                                   # the degenerate lines do get paired
    r, a = synth.lidar_frame(5)
    lp = np.rint(np.asarray(fr["lidar_pose"], np.float64)).astype(np.int32)
    res, ori = 0.05, (1.5, -2.0)
    est, pose, coff = fm.legacy_frames([dict(scan_lines=sl, lidar_pos=lp, ranges=r, angles=a)], res, ori, want_pose_all=True)
    want, we, wr = oraclebind.fa_legacy(sl, ml, res, ori, lp, mc, r, a)
    assert len(pose) > 100 and _bits_equal(pose, want)
    assert _bits_equal(est[0]["estimate_pose"], we) and _bits_equal(est[0]["estimate_pose_realworld"], wr)
    fm.close()
