"""Parity of the CUDA LSD path (through the C ABI) with the oracle and with the reference's golden outputs.
Bit-exact: mag, deg (vs the oracle on the same arithmetic), seed order, used-map, labels, segment table, lineIm."""
import contextlib
import os

import numpy as np
import pytest

import oraclebind
import synth

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
NAMES = ["mapValue", "mapValue_aisle1", "mapValue_aisle2", "mapValue_aisle3", "mapValue_map1", "mapValue_map2"]


def _compare_with_oracle(lsdb, b, i, m, got, check_planes=True, **params):
    """map i of batch b against the oracle at the batch's LSD parameters `params` (default: the reference's constants)"""
    o = oraclebind.lsd(m, **params)
    W = o["used"].shape[1]
    assert got["counts"][i] == o["n"]
    pl = b.planes(i)
    if check_planes:
        assert np.array_equal(pl["mag"], o["mag"])
        assert np.array_equal(pl["deg"], o["deg"])
    assert np.array_equal(pl["seeds"], o["seeds"][:, 2] * W + o["seeds"][:, 1])
    assert np.array_equal(pl["used"], o["used"])
    assert np.array_equal(pl["labels"], o["labels"])
    assert np.array_equal(lsdb.lines_to_array(got["lines"][i]), o["lines"], equal_nan=True)
    assert np.array_equal(got["rects"][i], o["rects"], equal_nan=True)      # rectangles and log-NFA, bit for bit
    assert np.array_equal(b.line_image(i), o["line_im"])
    return o


@contextlib.contextmanager
def lsdb_env(env):
    """`env` set in os.environ for the block, the previous values back afterwards.  The library reads its switches when a
    batch is created (team size, ban plane, the stencil stage's deferred-list cap) and when it runs (LSDB_GROW_WIDE picks the grower's build at
    launch), so the block covers both."""
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


@pytest.fixture(scope="module")
def gold():
    return np.load(os.path.join(GOLD, "bundled_maps.npz"))


def test_bundled_maps_batched_bit_exact(lsdb, ctx, gold):
    """BASELINE config 2: all bundled maps in one batch; golden = unmodified reference (stock glibc)."""
    maps = [gold[n + "/map"] for n in NAMES]
    b = lsdb.Batch(ctx, [(m.shape[1], m.shape[0]) for m in maps])
    b.upload(maps); b.run()
    got = b.download(want_rects=True)
    for i, n in enumerate(NAMES):
        o = _compare_with_oracle(lsdb, b, i, maps[i], got)
        pl = b.planes(i)
        assert got["counts"][i] == len(gold[n + "/lines"])
        assert np.array_equal(lsdb.lines_to_array(got["lines"][i]), gold[n + "/lines"], equal_nan=True)
        assert np.array_equal(pl["used"], gold[n + "/used"])
        assert np.array_equal((pl["labels"] & 0xFF).astype(np.uint8), gold[n + "/reg_idx"])
        assert np.array_equal(pl["seeds"], gold[n + "/seeds"])
        assert np.array_equal(np.packbits(b.line_image(i) > 0), gold[n + "/line_im_bits"])
    st = b.stats()
    assert st["accepts"] == sum(len(gold[n + "/lines"]) for n in NAMES)
    b.close()


def test_line_images_on_the_device_equal_the_host_epilogue(lsdb, ctx, gold):
    """lsdb_batch_line_images (csrc/lineim.cu: every map's lineIm rasterised on the device, LSD/myLSD.cpp:296-355) == the host
    epilogue lsdb_batch_line_image == the reference's lineIm (goldens), for the bundled maps and two synthetic ones."""
    maps = [gold[n + "/map"] for n in NAMES] + [synth.occupancy_grid(900, 700, seed=3), synth.occupancy_grid(333, 901, seed=22, border_walls=True)]
    b = lsdb.Batch(ctx, [(m.shape[1], m.shape[0]) for m in maps])
    b.upload(maps); b.run()
    ims = b.line_images()
    for i, m in enumerate(maps):
        assert ims[i].shape == m.shape and set(np.unique(ims[i])) <= {0, 255}
        assert np.array_equal(ims[i], b.line_image(i)), i
        if i < len(NAMES):
            assert np.array_equal(np.packbits(ims[i] > 0), gold[NAMES[i] + "/line_im_bits"])
        else:
            assert np.array_equal(ims[i], oraclebind.lsd(m)["line_im"])
    b.run(); again = b.line_images()                 # the plane is cleared on every call
    assert all(np.array_equal(x, y) for x, y in zip(ims, again))
    b.close()


def test_the_two_further_bundled_maps(lsdb, ctx):
    """BASELINE configs[1] 'all bundled maps': the distinct maps of data_20190513 / data_20190514 against the reference's goldens"""
    from test_oracle import _extra_maps
    items = list(_extra_maps())
    b = lsdb.Batch(ctx, [(m.shape[1], m.shape[0]) for _, m, _ in items])
    b.upload([m for _, m, _ in items]); b.run()
    got = b.download()
    for i, (name, m, g) in enumerate(items):
        pl = b.planes(i)
        assert got["counts"][i] == len(g[name + "/lines"])
        assert np.array_equal(lsdb.lines_to_array(got["lines"][i]), g[name + "/lines"], equal_nan=True)
        assert np.array_equal(pl["used"], g[name + "/used"]) and np.array_equal((pl["labels"] & 0xFF).astype(np.uint8), g[name + "/reg_idx"])
        assert np.array_equal(pl["seeds"], g[name + "/seeds"])
    b.close()


def test_single_map_call_matches_reference_entry_point(lsdb, ctx, gold):
    """lsdb_lsd = the body behind mylsd::myLineSegmentDetector (config 1)."""
    m = gold["mapValue/map"]
    r = ctx.lsd(m, want_remap=True)
    o = oraclebind.lsd(m)
    assert r["n"] == 41
    assert np.array_equal(lsdb.lines_to_array(r["lines"]), gold["mapValue/lines"], equal_nan=True)
    assert np.array_equal(r["line_im"], o["line_im"]) and np.array_equal(r["map_out"], o["map_out"])
    r2 = ctx.lsd(m)   # cached batch, second call identical
    assert np.array_equal(lsdb.lines_to_array(r2["lines"]), lsdb.lines_to_array(r["lines"]), equal_nan=True)


@pytest.mark.parametrize("shape,seed", [((600, 400), 7), ((333, 901), 22), ((64, 50), 23), ((1377, 428), 11),
                                         ((40, 34), 3), ((2048, 2048), 1000)])
def test_synthetic_maps_vs_oracle(lsdb, ctx, shape, seed):
    m = synth.occupancy_grid(shape[0], shape[1], seed=seed)
    b = lsdb.Batch(ctx, [shape])
    b.upload([m]); b.run()
    got = b.download(want_rects=True)
    _compare_with_oracle(lsdb, b, 0, m, got)
    b.close()


def test_ragged_batch_and_determinism(lsdb, ctx):
    shapes = [(500, 300), (34, 40), (777, 555), (128, 128), (1000, 90), (90, 1000), (600, 400)]
    maps = [synth.occupancy_grid(c, r, seed=100 + i) for i, (c, r) in enumerate(shapes)]
    b = lsdb.Batch(ctx, shapes)
    b.upload(maps); b.run()
    got = b.download(want_rects=True)
    for i, m in enumerate(maps):
        _compare_with_oracle(lsdb, b, i, m, got)
    b.run()   # same resident inputs again: identical output (the commit order is deterministic)
    got2 = b.download(want_rects=True)
    assert np.array_equal(got["counts"], got2["counts"])
    for i in range(len(maps)):
        assert np.array_equal(got["rects"][i], got2["rects"][i], equal_nan=True)
    b.close()


def test_edge_cases(lsdb, ctx):
    blank = np.zeros((120, 160), np.uint8)                      # maxGrad == 0: no seeds, no segments
    full = np.ones((120, 160), np.uint8)                        # everything occupied: flat interior
    unknown = np.full((100, 100), 255, np.uint8)               # row 0 / col 0 keep 255 (not remapped): a border edge
    one = np.zeros((90, 90), np.uint8); one[45, 10:80] = 1      # a single 1-px wall
    border = np.zeros((90, 120), np.uint8); border[0, :] = 1; border[:, 0] = 1; border[30, :] = 1
    tiny = np.zeros((7, 9), np.uint8); tiny[3, :] = 1           # scaled image 2x2
    maps = [blank, full, unknown, one, border, tiny]
    b = lsdb.Batch(ctx, [(m.shape[1], m.shape[0]) for m in maps])
    b.upload(maps); b.run()
    got = b.download(want_rects=True)
    assert got["counts"][0] == 0
    for i, m in enumerate(maps):
        _compare_with_oracle(lsdb, b, i, m, got)
    b.close()


def test_full_size_map_vs_oracle(lsdb, ctx):
    """BASELINE config 3 shape (4096x4096): one map compared in full with the oracle, plus size-independent
    properties: every accepted pixel is banned, labels are 1..n, seed list sorted by (bin desc, raster asc)."""
    m = synth.occupancy_grid(4096, 4096, seed=1000)
    b = lsdb.Batch(ctx, [(4096, 4096)])
    b.upload([m]); b.run()
    got = b.download(want_rects=True)
    _compare_with_oracle(lsdb, b, 0, m, got)
    pl = b.planes(0)
    n = got["counts"][0]
    assert n > 100
    assert set(np.unique(pl["labels"])) == set(range(0, n + 1))
    assert np.all(pl["used"][pl["labels"] > 0] == 1)
    zoom = 1024.0 / pl["max_grad"]
    bins = np.minimum(np.floor(pl["mag"].ravel()[pl["seeds"]] * zoom), 1024)
    key = bins * 2.0 ** 32 - pl["seeds"]
    assert np.all(np.diff(key) < 0)
    b.close()


def test_sixteen_full_size_maps_vs_oracle(lsdb, ctx):
    """Parity at the benchmark configuration (BASELINE configs[2] shape): 16 distinct 4096x4096 maps in ONE batch — the
    team shape bench.py runs — four of them with walls along row 0 / column 0.  Segment count, rectangles, log-NFA and
    line tables bit for bit against the oracle, and the work counters (accepts, rejects, live seeds) per map: the
    angle decisions on the running sums and the NFA tail break rest on wide differential coverage at this size."""
    seeds = [1001 + 7 * k for k in range(12)] + [2001, 2002, 2003, 2004]
    maps = [synth.occupancy_grid(4096, 4096, seed=s_, border_walls=(s_ >= 2001)) for s_ in seeds]
    b = lsdb.Batch(ctx, [(4096, 4096)] * len(maps))
    b.upload(maps); b.run()
    got = b.download(want_rects=True)
    for i, m in enumerate(maps):
        o = oraclebind.lsd(m, want_maps=False, want_line_im=False)
        assert got["counts"][i] == o["n"], (seeds[i], got["counts"][i], o["n"])
        assert np.array_equal(got["rects"][i], o["rects"], equal_nan=True), seeds[i]
        assert np.array_equal(lsdb.lines_to_array(got["lines"][i]), o["lines"], equal_nan=True), seeds[i]
        st = b.map_stats(i)
        assert (st["accepts"], st["rejects"], st["live_seeds"]) == (o["stats"]["accepts"], o["stats"]["rejects"], o["stats"]["live_seeds"]), seeds[i]
    b.close()


def test_scan_rasters_batched_then_associated(lsdb, ctx):
    """BASELINE config 4 at test scale: rasterised lidar scans (myrdp::FeatureScan lineIm of data/Lidar.txt frames, golden
    fixture) go through LSD as one ragged batch — segment tables equal to the unmodified reference's (1e-9) and the oracle's (bit-exact) — and the frames are
    then associated against LSD(data/mapValue.txt) in one launch."""
    g = np.load(os.path.join(GOLD, "fa_frames.npz"))
    gm = np.load(os.path.join(GOLD, "bundled_maps.npz"))
    nf = int(g["n_frames"])
    rasters = []
    for f in range(nf):
        h, w = (int(v) for v in g[f"f{f}/scan_im_shape"])
        rasters.append(np.unpackbits(g[f"f{f}/scan_im_bits"])[:h * w].reshape(h, w).astype(np.uint8))   # occupied = 1
    b = lsdb.Batch(ctx, [(r.shape[1], r.shape[0]) for r in rasters])
    b.upload(rasters); b.run()
    got = b.download()
    for f in range(nf):
        want = g[f"f{f}/scan_lsd_lines"]            # unmodified reference, stock glibc
        mine = lsdb.lines_to_array(got["lines"][f])
        assert got["counts"][f] == len(want)
        # contract: 1e-9 relative on segment geometry.  (glibc's sin/cos are 1 ulp off the correctly rounded value in two of
        # the twelve frames' dx/dy; against the oracle on the shared correctly-rounded math the table is bit-exact.)
        assert np.allclose(mine, want, rtol=1e-9, atol=0, equal_nan=True)
        assert np.array_equal(mine, oraclebind.lsd(rasters[f], want_maps=False)["lines"], equal_nan=True)
    b.close()
    mc = oraclebind.map_cache(gm["mapValue/map"], float(gm["mapValue/param"][2]))
    fm = lsdb.FaMap(ctx, mc, g["map_lines"])
    frames = [dict(scan_lines=lsdb.lines_to_array(got["lines"][f]), pts=g[f"f{f}/pts"], lidar_pose=g[f"f{f}/lidar_pose"],
                   last_pose=[-1.0, -1.0, 0.0]) for f in range(nf)]
    hyp = fm.score(frames)
    pos = 0
    for f in range(nf):
        oi, ov = oraclebind.fa_scores(frames[f]["scan_lines"], g["map_lines"], frames[f]["pts"], mc, frames[f]["lidar_pose"],
                                      frames[f]["last_pose"])
        h = hyp[pos:pos + len(oi)]; pos += len(oi)
        assert np.array_equal(np.stack([h["i_scan"], h["i_map"], h["i_pair"]], 1).reshape(-1, 3), oi.reshape(-1, 3))
        fin = np.isfinite(ov[:, 3]) if len(ov) else np.zeros(0, bool)
        assert np.array_equal(np.isfinite(h["score"]), fin)
        assert np.allclose(h["score"][fin], ov[fin, 3], rtol=1e-9, atol=0)
    assert pos == len(hyp)
    fm.close()


@pytest.mark.parametrize("env", [dict(LSDB_GROW_WARPS="1"), dict(LSDB_GROW_WARPS="3"), dict(LSDB_GROW_WARPS="8", LSDB_STEAL="1"),
                                 dict(LSDB_GROW_WARPS="16", LSDB_RUNAHEAD="16"), dict(LSDB_NO_SMEM_BAN="1"),
                                 dict(LSDB_SMEM_BAN_KB="200", LSDB_GROW_WARPS="16"), dict(LSDB_GROW_WIDE="0"), dict(LSDB_GROW_WIDE="1", LSDB_GROW_WARPS="8"), dict(LSDB_SUPER_SHIFT="0"), dict(LSDB_SUPER_SHIFT="3", LSDB_GROW_WARPS="16")])
def test_result_is_independent_of_team_shape(lsdb, ctx, gold, env):
    """The ordered-commit pipeline must give the sequential result whatever the speculation looks like: team size,
    run-ahead window, team-wide queue for large seeds, ban plane in shared memory or not."""
    maps = [gold["mapValue_aisle2/map"], synth.occupancy_grid(1500, 1100, seed=77), synth.occupancy_grid(900, 1300, seed=78, border_walls=True)]
    with lsdb_env(env):
        b = lsdb.Batch(ctx, [(m.shape[1], m.shape[0]) for m in maps])
        b.upload(maps); b.run()
    got = b.download(want_rects=True)
    for i, m in enumerate(maps):
        _compare_with_oracle(lsdb, b, i, m, got, check_planes=False)
    b.close()


@pytest.mark.parametrize("cap", [0, 2, 5, 64, 512], ids=lambda c: f"{c}_records" if c else "whole_plane")
def test_stencil_planes_with_the_deferred_list_full_and_not(lsdb, ctx, gold, cap):
    """The stencil stage queues the pixels whose phase-1 rounding test fails in a deferred list that a second kernel
    evaluates.  At its default size (the scratch plane) the tiles' reservations fit; capped at 2, 5, 64 and 512 records the
    list fills after fewer or more tiles, and a tile whose reservation does not fit evaluates its own (the part inside the
    list becomes no-ops).  Same planes, seed lists and segments as the oracle either way — borders with reflected taps, a
    ragged 33rd column and row 0 / column 0 walls included."""
    maps = [gold["mapValue/map"], synth.occupancy_grid(1057, 771, seed=91), synth.occupancy_grid(400, 1300, seed=92, border_walls=True),
            synth.occupancy_grid(97, 45, seed=12), synth.occupancy_grid(2048, 2048, seed=93)]
    with lsdb_env(dict(LSDB_STENCIL_DEFER=str(cap)) if cap else {}):
        b = lsdb.Batch(ctx, [(m.shape[1], m.shape[0]) for m in maps])
        b.upload(maps); b.run()
    got = b.download(want_rects=True)
    assert b.launches() == 6
    for i, m in enumerate(maps):
        _compare_with_oracle(lsdb, b, i, m, got, check_planes=True)
    b.close()


@pytest.mark.parametrize("warps", [1, 4, 16])
def test_team_size_set_through_the_abi(lsdb, warps):
    """lsdb_set_team_warps: the caller's team size (several small batches in flight want 4 where one alone gets 8) — same result."""
    c = lsdb.Context(0)
    try:
        c.set_team_warps(warps)
        maps = [synth.occupancy_grid(1200, 900, seed=91), synth.occupancy_grid(700, 1000, seed=92, border_walls=True)]
        b = lsdb.Batch(c, [(m.shape[1], m.shape[0]) for m in maps])
        b.upload(maps); b.run()
        got = b.download(want_rects=True)
        for i, m in enumerate(maps):
            _compare_with_oracle(lsdb, b, i, m, got, check_planes=False)
        b.close()
        with pytest.raises(lsdb.LsdbError, match="ARG"):
            c.set_team_warps(17)
        c.set_team_warps(0)
    finally:
        c.close()


def test_giant_map_on_one_gpu(lsdb, ctx):
    """BASELINE config 5 shape (one 16384x16384 map, seed 5000) on a single GPU: segment table and rectangles bit-exact
    against the oracle.  (Tiling it across GPUs is not built; this pins the single-GPU result the tiled version must keep.)"""
    m = synth.occupancy_grid(16384, 16384, seed=5000)
    b = lsdb.Batch(ctx, [(16384, 16384)], max_lines=65536)
    b.upload([m]); b.run()
    got = b.download(want_rects=True)
    o = oraclebind.lsd(m, want_maps=False, want_line_im=False, max_lines=65536)
    assert got["counts"][0] == o["n"] and o["n"] > 5000
    assert np.array_equal(got["rects"][0], o["rects"], equal_nan=True)
    assert np.array_equal(lsdb.lines_to_array(got["lines"][0]), o["lines"], equal_nan=True)
    st = b.stats()
    assert st["accepts"] == o["stats"]["accepts"] and st["rejects"] == o["stats"]["rejects"] and st["live_seeds"] == o["stats"]["live_seeds"]
    b.close()


def test_error_paths_fail_loudly_and_leave_the_context_usable(lsdb, ctx, gold):
    """No silent truncation: a segment table that is too small is an LSDB_ERR_CAPACITY error, bad parameters are
    LSDB_ERR_ARG, and the context keeps working afterwards."""
    m = gold["mapValue/map"]
    b = lsdb.Batch(ctx, [(m.shape[1], m.shape[0])], max_lines=5)        # the map has 41 segments
    b.upload([m]); b.run()
    with pytest.raises(lsdb.LsdbError, match="CAPACITY"):
        b.download()
    b.close()
    with pytest.raises(lsdb.LsdbError, match="ARG"):
        lsdb.Batch(ctx, [(m.shape[1], m.shape[0])], pseBin=5000)
    with pytest.raises(lsdb.LsdbError, match="ARG"):
        lsdb.Batch(ctx, [(m.shape[1], m.shape[0])], sca=0.5)             # Gaussian half-width != 8: only sig/sca = 2 is built
    with pytest.raises(lsdb.LsdbError, match="ARG"):
        lsdb.Batch(ctx, [(0, 10)])
    with pytest.raises(lsdb.LsdbError, match="ARG"):                     # half-width 8, but a tile's source window would not fit
        lsdb.Batch(ctx, [(m.shape[1], m.shape[0])], sca=0.2, sig=0.4)    # the stencil's shared-memory staging (ADVICE r1)
    r = ctx.lsd(m)                                                       # still fine
    assert r["n"] == 41


def test_two_devices_in_one_process(lsdb, gold):
    """One context per GPU inside one process (SURVEY §8e: 'one host thread/stream per GPU'): a batch split across two
    devices by shard_range gives the same tables as the whole batch on one."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from lsdb200 import shard
    names = NAMES[:4]
    maps = [gold[n + "/map"] for n in names]
    outs = []
    for dev in range(2):
        first, cnt = shard.shard_range(len(maps), dev, 2)
        c = lsdb.Context(dev)
        b = lsdb.Batch(c, [(m.shape[1], m.shape[0]) for m in maps[first:first + cnt]])
        b.upload(maps[first:first + cnt]); b.run()
        outs.extend(lsdb.lines_to_array(x) for x in b.download()["lines"])
        b.close(); c.close()
    for n, got in zip(names, outs):
        assert np.array_equal(got, gold[n + "/lines"], equal_nan=True), n


def test_staged_single_map_path_on_one_gpu(lsdb, ctx, gold):
    """The pieces of the tiled single-map path (SURVEY §8e, configs[4]) without NCCL: two batches on one GPU play two ranks —
    each runs the stencil stage on its band of tile rows, the bands are copied into rank 0's planes (what giant.py does with
    NCCL broadcasts), maxGrad becomes the max of the two, the region stages run on the assembled planes.  Equal to the goldens."""
    import torch
    from lsdb200 import giant
    for name in ("mapValue_aisle1", "mapValue"):
        m = gold[name + "/map"]
        bs = [lsdb.Batch(ctx, [(m.shape[1], m.shape[0])]) for _ in range(2)]
        for b in bs:
            b.upload([m])
        planes = [giant.band_planes(b) for b in bs]
        tile_rows, rpt = planes[0][1], planes[0][2]
        H = bs[0].scaled(0)[1]
        bands = [giant.band_rows(tile_rows, rpt, H, r, 2) for r in range(2)]
        assert bands[0][1] > 0 and bands[1][1] > 0 and bands[0][3] == bands[1][2] and bands[1][3] == H
        for r, b in enumerate(bs):
            giant.run_stencil_rows(b, bands[r][0], bands[r][0] + bands[r][1])
        g = [giant.max_grad(b) for b in bs]
        giant.max_grad(bs[0], max(g))
        y0, y1 = bands[1][2], bands[1][3]
        for (p0, rb), (p1, _rb) in zip(planes[0][0], planes[1][0]):
            dst = torch.as_tensor(giant._DevView(p0, rb * H), device="cuda"); src = torch.as_tensor(giant._DevView(p1, rb * H), device="cuda")
            dst[y0 * rb:y1 * rb].copy_(src[y0 * rb:y1 * rb])
        torch.cuda.synchronize()
        giant.run_regions(bs[0])
        got = bs[0].download(want_rects=True)
        assert got["counts"][0] == len(gold[name + "/lines"])
        assert np.array_equal(lsdb.lines_to_array(got["lines"][0]), gold[name + "/lines"], equal_nan=True)
        pl = bs[0].planes(0)
        assert np.array_equal(pl["used"], gold[name + "/used"]) and np.array_equal(pl["seeds"], gold[name + "/seeds"])
        assert pl["max_grad"] == max(g) and min(g) > 0
        for b in bs:
            b.close()


def test_one_process_several_devices_entry_point(lsdb, gold):
    """lsdb_multi_lsd (SURVEY §8b/§8e): one process drives several devices, one host thread and stream per device, the batch
    split contiguously.  On a one-GPU box device 0 is listed three times (three contexts, three threads, uneven shards of
    2/2/1 maps); with more GPUs the first three devices are used.  Tables must equal the goldens in batch order."""
    import torch
    nd = torch.cuda.device_count()
    devs = [0, 0, 0] if nd < 2 else [d % nd for d in range(3)]
    names = NAMES[:5]
    mc = lsdb.MultiContext(devs)
    out = mc.lsd([gold[n + "/map"] for n in names], want_rects=True)
    for i, n in enumerate(names):
        assert out["counts"][i] == len(gold[n + "/lines"]), n
        assert np.array_equal(lsdb.lines_to_array(out["lines"][i]), gold[n + "/lines"], equal_nan=True), n
    out2 = mc.lsd([gold[NAMES[0] + "/map"]])                     # fewer maps than devices: two empty shards
    assert out2["counts"][0] == len(gold[NAMES[0] + "/lines"])
    with pytest.raises(lsdb.LsdbError, match="device 0"):
        mc.lsd([gold[NAMES[0] + "/map"]], max_lines=3)          # errors carry the device and the library's message
    mc.close()
    with pytest.raises(lsdb.LsdbError):
        lsdb.MultiContext([99])


@pytest.mark.parametrize("params", [dict(angThre=30.0), dict(denThre=0.55), dict(pseBin=512), dict(angThre=15.0, denThre=0.8, pseBin=256)])
def test_non_default_parameters_vs_oracle(lsdb, ctx, gold, params):
    """arguments 6-8 of myLineSegmentDetector (angThre, denThre, pseBin) other than the constants of LSD/baseFunc.h:64-68"""
    maps = [gold["mapValue_aisle1/map"], synth.occupancy_grid(700, 500, seed=41)]
    b = lsdb.Batch(ctx, [(m.shape[1], m.shape[0]) for m in maps], **params)
    b.upload(maps); b.run()
    got = b.download(want_rects=True)
    for i, m in enumerate(maps):
        o = oraclebind.lsd(m, **params)
        pl = b.planes(i)
        assert got["counts"][i] == o["n"]
        assert np.array_equal(pl["used"], o["used"]) and np.array_equal(pl["labels"], o["labels"])
        assert np.array_equal(got["rects"][i], o["rects"], equal_nan=True)
        assert np.array_equal(lsdb.lines_to_array(got["lines"][i]), o["lines"], equal_nan=True)
    b.close()
