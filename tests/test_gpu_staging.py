"""One context's staging buffers, reused across entry points.

A context grows its staging buffers on demand and keeps them between calls: the association, the catkin snapshot's association
and the scan front-end share some of them, and each grows on its own.  The same context runs every entry point that stages
through them, interleaved, on inputs that grow, shrink and grow again past their first peak; every result must have the bits
of the same call on a fresh context.  Then the batch entry points must leave the launch count and the stage events as they
always did: lsdb_batch_run, and the staged pair lsdb_batch_run_stencil_rows + lsdb_batch_run_regions that giant.py drives."""
import os

import numpy as np
import pytest

import oraclebind
import synth

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ROUNDS = (2, 6, 1, 12)   # input size per round: up, down, then up past the first peak


@pytest.fixture(scope="module")
def inputs():
    """golden and seeded inputs, and the two association maps' cache and lines (both on the bundled mapValue)"""
    gm = np.load(os.path.join(GOLD, "bundled_maps.npz"))
    fa = np.load(os.path.join(GOLD, "fa_frames.npz"))
    lg = np.load(os.path.join(GOLD, "fa_legacy.npz"))
    lf = np.load(os.path.join(GOLD, "lidar_frames.npz"))
    m = gm["mapValue/map"]
    cache = oraclebind.map_cache(m, float(gm["mapValue/param"][2]))
    legacy_cache = cache.copy()
    legacy_cache[legacy_cache == 1.0] = 2.0   # the snapshot's three-argument createMapCache
    fa_gold = [dict(scan_lines=fa[f"f{f}/scan_lines"], pts=fa[f"f{f}/pts"], lidar_pose=fa[f"f{f}/lidar_pose"], last_pose=fa[f"f{f}/last_pose"])
               for f in range(int(fa["n_frames"]))]
    lg_gold = [dict(scan_lines=lg[f"f{f}/scan_lines"], lidar_pos=lg[f"f{f}/lidar_pos"], ranges=lg[f"f{f}/ranges"], angles=lg[f"f{f}/angles"])
               for f in range(int(lg["n_frames"]))]
    sweeps_gold = []
    for f in range(int(lf["n_frames"])):
        r = lf[f"f{f}/ranges"]
        keep = np.isfinite(r)
        sweeps_gold.append((r[keep], lf[f"f{f}/angles"][keep]))
    return dict(map=m, cache=cache, lines=fa["map_lines"], legacy_cache=legacy_cache, legacy_lines=lg["map_lines"],
                resol=float(lg["resol"]), ori=lg["ori"], scan_param=lf["map_param"], fa_gold=fa_gold, lg_gold=lg_gold, sweeps_gold=sweeps_gold)


def _fa_maps(lsdb, ctx, inp):
    return dict(fa=lsdb.FaMap(ctx, inp["cache"], inp["lines"]), legacy=lsdb.FaMap(ctx, inp["legacy_cache"], inp["legacy_lines"]))


@pytest.fixture(scope="module")
def shared(lsdb, inputs):
    """the one context every call of the interleaving runs on, with its association maps"""
    ctx = lsdb.Context(0)
    maps = _fa_maps(lsdb, ctx, inputs)
    yield ctx, maps
    for fm in maps.values():
        fm.close()
    ctx.close()


# ---- the inputs of round r at size n: golden and seeded items alternate ----

def _fa_frames(inp, r, n):
    return [inp["fa_gold"][(r + i) % len(inp["fa_gold"])] if i % 2 == 0 else synth.fake_scan_frame(inp["map"], inp["lines"], seed=1000 * r + i)
            for i in range(n)]


def _sweeps(inp, r, n):
    out = []
    for i in range(n):
        if i % 2 == 0:
            out.append(inp["sweeps_gold"][(7 * r + i) % len(inp["sweeps_gold"])])
        else:
            out.append(synth.lidar_frame(2000 * r + i, n_beams=(200, 360, 1081)[i % 3]))
    return out


def _legacy_frames(inp, r, n):
    out = []
    for i in range(n):
        g = inp["lg_gold"][(r + i) % len(inp["lg_gold"])]
        if i % 2 == 0:
            out.append(g)
        else:   # the golden frame's scan lines with a seeded sweep
            rng, ang = synth.lidar_frame(3000 * r + i, n_beams=(360, 1081)[(i // 2) % 2])
            out.append(dict(scan_lines=g["scan_lines"], lidar_pos=g["lidar_pos"], ranges=rng, angles=ang))
    return out


# ---- every entry point: (ctx, association maps, inputs, round, size) -> the arrays it returns ----

def _score(lsdb, ctx, maps, inp, r, n):
    return [maps["fa"].score(_fa_frames(inp, r, n))]


def _estimate(lsdb, ctx, maps, inp, r, n):
    return [maps["fa"].estimate(_fa_frames(inp, r, n))]


def _score_kept(lsdb, ctx, maps, inp, r, n):
    kept, scored = maps["fa"].score_kept(_fa_frames(inp, r, n))
    return [kept, np.array([scored])]


def _scan_estimate(lsdb, ctx, maps, inp, r, n):
    mp = inp["scan_param"]
    return list(maps["fa"].scan_estimate(mp[2], mp[3], mp[4], _sweeps(inp, r, 4 * n)))


def _legacy_frames_call(lsdb, ctx, maps, inp, r, n):
    est, pose_all, col_off = maps["legacy"].legacy_frames(_legacy_frames(inp, r, 2 * n), inp["resol"], inp["ori"], want_pose_all=True)
    return [est, pose_all, col_off]


def _feature_scan(lsdb, ctx, maps, inp, r, n):
    mp = inp["scan_param"]
    out = []
    for o in ctx.feature_scan(mp[2], mp[3], mp[4], _sweeps(inp, r + 1, 4 * n), want_rasters=True):
        out += [o["lines"], o["pts"], o["lidar_pos"], np.array(o["size"]), o["line_im"]]
    return out


def _scan_rasters(lsdb, ctx, maps, inp, r, n):
    """the rasters a batch receives, through what is computed from them: mapCache and the LSD segment tables"""
    mp = inp["scan_param"]
    sweeps = _sweeps(inp, r + 2, 2 * n)
    info = ctx.feature_scan_info(mp[2], mp[3], mp[4], sweeps)
    b = lsdb.Batch(ctx, [(int(i["im_cols"]), int(i["im_rows"])) for i in info], max_lines=512)
    try:
        out = [b.upload_scan_rasters(mp[2], mp[3], mp[4], sweeps)]
        out += b.map_caches(float(mp[2]))
        b.run()
        got = b.download(want_rects=True)
        return out + [got["counts"]] + got["lines"] + got["rects"]
    finally:
        b.close()


def _map_cache(lsdb, ctx, maps, inp, r, n):
    m = synth.occupancy_grid(120 * n + 7, 90 * n + 3, seed=4000 + r)
    return [ctx.map_cache(m, 0.05), ctx.map_cache(m, 0.05, max_dist=1.0, unreached=2.0)]


CALLS = [_score, _scan_estimate, _estimate, _feature_scan, _score_kept, _map_cache, _legacy_frames_call, _scan_rasters]


def _on_fresh_context(lsdb, call, inp, r, n):
    ctx = lsdb.Context(0)
    maps = _fa_maps(lsdb, ctx, inp)
    try:
        return call(lsdb, ctx, maps, inp, r, n)
    finally:
        for fm in maps.values():
            fm.close()
        ctx.close()


def test_staging_reused_across_entry_points_matches_fresh_contexts(lsdb, inputs, shared):
    ctx, maps = shared
    for r, n in enumerate(ROUNDS):
        order = CALLS[r:] + CALLS[:r]   # each round starts at another entry point
        for call in order:
            got = call(lsdb, ctx, maps, inputs, r, n)
            want = _on_fresh_context(lsdb, call, inputs, r, n)
            what = f"{call.__name__} in round {r} (size {n})"
            assert len(got) == len(want), what
            for k, (a, b) in enumerate(zip(got, want)):
                a, b = np.asarray(a), np.asarray(b)
                assert a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes(), f"{what}: array {k}"
            assert sum(np.asarray(a).size for a in got) > 0, what


def _stages_ok(b):
    ms = b.stage_ms()
    assert len(ms) == 3 and all(np.isfinite(v) and v >= 0 for v in ms.values()), ms


def test_batch_entry_points_keep_launches_and_stage_events(lsdb, inputs, shared):
    from lsdb200 import giant
    ctx, _maps = shared
    n_stencil = 2
    maps = [inputs["map"], synth.occupancy_grid(700, 500, seed=5)]
    b = lsdb.Batch(ctx, [(m.shape[1], m.shape[0]) for m in maps])
    b.upload(maps)
    b.run()
    assert b.launches() == 4 + n_stencil
    _stages_ok(b)
    assert b.download()["counts"].min() > 0
    b.close()

    m = inputs["map"]
    s = lsdb.Batch(ctx, [(m.shape[1], m.shape[0])])
    s.upload([m])
    s.run()
    whole = s.download(want_rects=True)
    tile_rows = giant.band_planes(s)[1]
    giant.run_stencil_rows(s, 0, tile_rows)
    assert s.launches() == n_stencil
    with pytest.raises(lsdb.LsdbError):   # the stencil stage alone is not a run: no stage times, no download
        s.stage_ms()
    with pytest.raises(lsdb.LsdbError):
        s.download()
    giant.run_regions(s)
    assert s.launches() == 4 + n_stencil
    _stages_ok(s)
    staged = s.download(want_rects=True)
    assert np.array_equal(whole["counts"], staged["counts"]) and whole["counts"][0] > 0
    assert whole["lines"][0].tobytes() == staged["lines"][0].tobytes() and whole["rects"][0].tobytes() == staged["rects"][0].tobytes()
    s.run()
    assert s.launches() == 4 + n_stencil
    _stages_ok(s)
    s.close()
