"""LSD batches fed from device memory and exported into it (lsdb_batch_upload_device, lsdb_batch_lines_device,
lsdb_batch_line_images_device, lsdb_batch_map_caches_device): byte for byte what the host path gives for the same maps, ordered
on the context stream without a host synchronise, and every refused argument refused before anything is enqueued."""
import ctypes as C
import os

import numpy as np
import pytest

import oraclebind
import synth

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
BUNDLED = ["mapValue", "mapValue_aisle1", "mapValue_aisle2", "mapValue_aisle3", "mapValue_map1", "mapValue_map2"]
ERR_ARG, ERR_CAPACITY = 2, 3
SLEEP_CYCLES = 200_000_000   # torch.cuda._sleep: about 0.1 s at the B200's ~2 GHz SM clock

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch():
    import torch
    return torch


@pytest.fixture(scope="module")
def dctx(lsdb):
    c = lsdb.Context(0)
    yield c
    c.close()


def _bundled():
    g = np.load(os.path.join(GOLD, "bundled_maps.npz"))
    return [g[n + "/map"] for n in BUNDLED]


def _ragged(seed=5):
    """seeded synthetic maps of mixed shapes"""
    shapes = [(900, 700), (333, 901), (1500, 400), (257, 1024), (640, 480), (1201, 799)]
    return [synth.occupancy_grid(c, r, seed=seed + k, border_walls=bool(k & 1)) for k, (c, r) in enumerate(shapes)]


def _host_path(lsdb, ctx, maps, res=0.05, **kw):
    """the tables, line images and map caches of the maps uploaded from host memory"""
    b = lsdb.Batch(ctx, [(m.shape[1], m.shape[0]) for m in maps], **kw)
    b.upload(maps); b.run()
    out = b.download(want_rects=True)
    out["line_ims"] = b.line_images()
    out["caches"] = b.map_caches(res)
    b.close()
    return out


def _to_device(torch, m, kind):
    """map m in device memory: 0 contiguous, 1 a column slice of a wider tensor (row pitch > cols, odd byte offset), 2 a view of
    a flat buffer at an odd byte offset"""
    rows, cols = m.shape
    t = torch.from_numpy(np.ascontiguousarray(m)).cuda()
    if kind == 0:
        return t
    if kind == 1:
        wide = torch.full((rows, cols + 37), 77, dtype=torch.uint8, device="cuda")
        wide[:, 5:5 + cols] = t
        return wide[:, 5:5 + cols]
    flat = torch.full((rows * cols + 3,), 77, dtype=torch.uint8, device="cuda")
    v = flat[3:].view(rows, cols)
    v.copy_(t)
    return v


def _tables_equal(got, want, n, check_status=True):
    """lines_device tensors (after a synchronise) == lsdb_batch_download records, map by map, byte for byte"""
    counts = got["counts"].cpu().numpy(); offs = got["offsets"].cpu().numpy(); st = got["status"].cpu().numpy()
    lines = got["lines"].cpu().numpy(); rects = got["rects"].cpu().numpy() if "rects" in got else None
    assert offs[0] == 0 and np.array_equal(np.diff(offs), counts)
    for i in range(n):
        assert counts[i] == want["counts"][i], i
        if check_status:
            assert st[i] == 0, i
        o, c = offs[i], counts[i]
        assert lines[o:o + c].tobytes() == np.ascontiguousarray(want["lines"][i]).tobytes(), i
        if rects is not None:
            assert rects[o:o + c].tobytes() == np.ascontiguousarray(want["rects"][i]).tobytes(), i


def _device_path(lsdb, ctx, maps, torch, kinds=None, res=0.05, **kw):
    b = lsdb.Batch(ctx, [(m.shape[1], m.shape[0]) for m in maps], **kw)
    grids = [_to_device(torch, m, (kinds or [0] * len(maps))[i]) for i, m in enumerate(maps)]
    b.upload_device(grids); b.run()
    got = b.lines_device(want_rects=True)
    ims, im_views = b.line_images_device()
    host_caches = b.map_caches(res)
    caches, cache_views = b.map_caches_device()
    torch.cuda.synchronize()
    return b, got, im_views, host_caches, cache_views


def test_bundled_and_ragged_maps_from_device_memory(lsdb, dctx, torch):
    maps = _bundled() + _ragged()
    want = _host_path(lsdb, dctx, maps)
    kinds = [k % 3 for k in range(len(maps))]
    b, got, ims, host_caches, caches = _device_path(lsdb, dctx, maps, torch, kinds)
    _tables_equal(got, want, len(maps))
    fields, orient = lsdb.line_fields(got["lines"])
    assert fields.shape == (got["lines"].shape[0], 9) and orient.shape == (got["lines"].shape[0],)
    assert fields.data_ptr() == got["lines"].data_ptr()
    offs = got["offsets"].cpu().numpy()
    for i, m in enumerate(maps):
        assert ims[i].shape == m.shape and np.array_equal(ims[i].cpu().numpy(), want["line_ims"][i]), i
        c = caches[i].cpu().numpy()
        assert c.tobytes() == want["caches"][i].tobytes() and c.tobytes() == host_caches[i].tobytes(), i
        f = fields[offs[i]:offs[i + 1]].cpu().numpy(); o = orient[offs[i]:offs[i + 1]].cpu().numpy()
        arr = lsdb.lines_to_array(want["lines"][i])
        assert np.array_equal(f, arr[:, :9], equal_nan=True) and np.array_equal(o, arr[:, 9].astype(np.int32)), i
    for i in (len(BUNDLED), len(BUNDLED) + 1):   # two synthetic maps against the oracle
        ref = oraclebind.lsd(maps[i])
        f = np.concatenate([fields[offs[i]:offs[i + 1]].cpu().numpy(), orient[offs[i]:offs[i + 1]].cpu().numpy()[:, None]], axis=1)
        assert np.array_equal(f, ref["lines"], equal_nan=True), i
        assert np.array_equal(ims[i].cpu().numpy(), ref["line_im"]), i
    # the host exits still work after the device ones, and agree
    again = b.download(want_rects=True)
    assert all(x.tobytes() == y.tobytes() for x, y in zip(again["lines"], want["lines"]))
    b.close()


def test_results_are_ordered_after_a_torch_producer(lsdb, torch):
    """grids written by a torch op on torch's current stream (a side stream, behind a sleep); the context has its own stream"""
    maps = _ragged(seed=31)[:4]
    ctx = lsdb.Context(0)
    want = _host_path(lsdb, ctx, maps)
    src = [torch.from_numpy(m).cuda() for m in maps]
    b = lsdb.Batch(ctx, [(m.shape[1], m.shape[0]) for m in maps])
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        grids = [torch.zeros_like(s) for s in src]
        torch.cuda._sleep(SLEEP_CYCLES)
        for g, s in zip(grids, src):
            g.copy_(s)                       # the producer: only after the sleep do the grids hold the maps
        b.upload_device(grids); b.run()
        got = b.lines_device(want_rects=True)
        ims, views = b.line_images_device()
        # consumers on the same (current) stream see the results: .cpu() orders on it
        _tables_equal(got, want, len(maps))
        for i in range(len(maps)):
            assert np.array_equal(views[i].cpu().numpy(), want["line_ims"][i]), i
    b.close(); ctx.close()


def test_calls_return_before_the_stream_gets_to_them(lsdb, torch):
    maps = _ragged(seed=41)[:3]
    host_ctx = lsdb.Context(0)
    want = _host_path(lsdb, host_ctx, maps)
    host_ctx.close()
    s = torch.cuda.Stream()
    ctx = lsdb.Context(0, stream=s.cuda_stream)
    b = lsdb.Batch(ctx, [(m.shape[1], m.shape[0]) for m in maps])
    with torch.cuda.stream(s):
        grids = [torch.from_numpy(m).cuda() for m in maps]
        b.upload_device(grids); b.run(); b.map_caches(0.05, download=False)   # warm every kernel; map_caches synchronises
        b.lines_device(); b.line_images_device(); b.map_caches_device()
        torch.cuda.synchronize()
        torch.cuda._sleep(SLEEP_CYCLES)
        ev = torch.cuda.Event()
        ev.record(s)
        b.upload_device(grids)
        assert not ev.query()
        b.run()
        got = b.lines_device(want_rects=True)
        assert not ev.query()
        ims, views = b.line_images_device()
        assert not ev.query()
        caches, cviews = b.map_caches_device()
        assert not ev.query()
    torch.cuda.synchronize()
    _tables_equal(got, want, len(maps))
    for i in range(len(maps)):
        assert np.array_equal(views[i].cpu().numpy(), want["line_ims"][i]), i
        assert cviews[i].cpu().numpy().tobytes() == want["caches"][i].tobytes(), i
    b.close(); ctx.close()


def test_a_map_over_max_lines_is_flagged_and_the_others_are_exact(lsdb, dctx, torch):
    maps = _bundled()
    want = _host_path(lsdb, dctx, maps)
    counts = np.asarray(want["counts"])
    big = int(np.argmax(counts))
    cap = int(np.sort(counts)[-2])            # enough for every map but the largest
    assert counts[big] > cap
    b = lsdb.Batch(dctx, [(m.shape[1], m.shape[0]) for m in maps], max_lines=cap)
    b.upload_device([_to_device(torch, m, 0) for m in maps]); b.run()
    got = b.lines_device(want_rects=True)
    torch.cuda.synchronize()
    st = got["status"].cpu().numpy(); cn = got["counts"].cpu().numpy(); offs = got["offsets"].cpu().numpy()
    lines = got["lines"].cpu().numpy()
    assert st[big] == ERR_CAPACITY and cn[big] == 0
    for i in range(len(maps)):
        if i != big:
            assert st[i] == 0 and cn[i] == counts[i]
            assert lines[offs[i]:offs[i + 1]].tobytes() == want["lines"][i].tobytes(), i
    with pytest.raises(lsdb.LsdbError, match="CAPACITY"):
        b.sync()
    b.close()


def test_max_total_too_small(lsdb, dctx, torch):
    maps = _bundled()
    want = _host_path(lsdb, dctx, maps)
    counts = np.asarray(want["counts"], np.int64)
    offs = np.concatenate([[0], np.cumsum(counts)])
    k = 3
    max_total = int(offs[k] + counts[k] - 1)   # map k and everything after it does not fit
    b = lsdb.Batch(dctx, [(m.shape[1], m.shape[0]) for m in maps])
    b.upload_device([_to_device(torch, m, 0) for m in maps]); b.run()
    guard = 64
    d_counts = torch.full((len(maps),), -1, dtype=torch.int32, device="cuda")
    d_offs = torch.full((len(maps) + 1,), -1, dtype=torch.int32, device="cuda")
    d_st = torch.full((len(maps),), -1, dtype=torch.int32, device="cuda")
    d_lines = torch.full(((max_total + guard) * 80,), 0xAB, dtype=torch.uint8, device="cuda")
    d_rects = torch.full(((max_total + guard) * 13 * 8,), 0xCD, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    rc = lsdb.lib().lsdb_batch_lines_device(b.h, d_counts.data_ptr(), d_offs.data_ptr(), d_st.data_ptr(), d_lines.data_ptr(),
                                            d_rects.data_ptr(), max_total)
    assert rc == 0
    torch.cuda.synchronize()
    assert np.array_equal(d_counts.cpu().numpy(), counts) and np.array_equal(d_offs.cpu().numpy(), offs)
    st = d_st.cpu().numpy()
    assert np.all(st[:k] == 0) and np.all(st[k:] == ERR_CAPACITY)
    lines = d_lines.cpu().numpy(); rects = d_rects.cpu().numpy()
    for i in range(k):
        assert lines[offs[i] * 80:offs[i + 1] * 80].tobytes() == want["lines"][i].tobytes(), i
        assert rects[offs[i] * 104:offs[i + 1] * 104].tobytes() == want["rects"][i].tobytes(), i
    assert np.all(lines[offs[k] * 80:] == 0xAB) and np.all(rects[offs[k] * 104:] == 0xCD)
    # the sizing query: counts and offsets only
    d_offs.fill_(-1)
    assert lsdb.lib().lsdb_batch_lines_device(b.h, d_counts.data_ptr(), d_offs.data_ptr(), None, None, None, 0) == 0
    torch.cuda.synchronize()
    assert np.array_equal(d_offs.cpu().numpy(), offs)
    b.close()


def test_argument_errors_leave_the_context_usable(lsdb, torch):
    L = lsdb.lib()
    maps = _ragged(seed=51)[:2]
    ctx = lsdb.Context(0)
    want = _host_path(lsdb, ctx, maps)
    n = len(maps)
    b = lsdb.Batch(ctx, [(m.shape[1], m.shape[0]) for m in maps])
    grids = [_to_device(torch, m, 0) for m in maps]
    dev_ptrs = [g.data_ptr() for g in grids]

    def upload(ptrs, pitches=None):
        arr = (C.c_void_p * n)(*ptrs)
        pa = None if pitches is None else np.asarray(pitches, np.int64)
        return L.lsdb_batch_upload_device(b.h, C.cast(arr, C.c_void_p), None if pa is None else pa.ctypes.data)
    host = [np.ascontiguousarray(m) for m in maps]
    pinned = [torch.from_numpy(m).pin_memory() for m in maps]
    assert upload([host[0].ctypes.data, dev_ptrs[1]]) == ERR_ARG                  # a numpy (pageable host) pointer
    assert upload([dev_ptrs[0], pinned[1].data_ptr()]) == ERR_ARG                 # pinned host memory
    assert upload([dev_ptrs[0], None]) == ERR_ARG                                 # a null map
    assert L.lsdb_batch_upload_device(b.h, None, None) == ERR_ARG
    assert upload(dev_ptrs, [maps[0].shape[1] - 1, maps[1].shape[1]]) == ERR_ARG  # pitch below cols
    assert "pitch" in L.lsdb_last_error(ctx.h).decode()
    with pytest.raises(ValueError):
        b.upload_device([torch.from_numpy(m) for m in maps])                      # CPU tensors never reach the library
    # before lsdb_batch_run / lsdb_batch_map_caches
    cnt = torch.zeros(n, dtype=torch.int32, device="cuda"); off = torch.zeros(n + 1, dtype=torch.int32, device="cuda")
    out = torch.zeros(sum(m.size for m in maps), dtype=torch.uint8, device="cuda")
    cache = torch.zeros(sum(m.size for m in maps), dtype=torch.float64, device="cuda")
    assert L.lsdb_batch_lines_device(b.h, cnt.data_ptr(), off.data_ptr(), None, None, None, 0) == ERR_ARG
    assert L.lsdb_batch_line_images_device(b.h, out.data_ptr()) == ERR_ARG
    assert L.lsdb_batch_map_caches_device(b.h, cache.data_ptr()) == ERR_ARG
    assert upload(dev_ptrs) == 0
    b.run()
    assert L.lsdb_batch_map_caches_device(b.h, cache.data_ptr()) == ERR_ARG
    # host outputs
    hc = np.zeros(n, np.int32); ho = np.zeros(n + 1, np.int32)
    assert L.lsdb_batch_lines_device(b.h, hc.ctypes.data, off.data_ptr(), None, None, None, 0) == ERR_ARG
    assert L.lsdb_batch_lines_device(b.h, cnt.data_ptr(), ho.ctypes.data, None, None, None, 0) == ERR_ARG
    assert L.lsdb_batch_lines_device(b.h, cnt.data_ptr(), off.data_ptr(), None, None, None, -1) == ERR_ARG
    hl = torch.zeros((100, 80), dtype=torch.uint8).pin_memory()
    assert L.lsdb_batch_lines_device(b.h, cnt.data_ptr(), off.data_ptr(), None, hl.data_ptr(), None, 100) == ERR_ARG
    host_out = np.zeros(out.numel(), np.uint8); host_cache = np.zeros(out.numel())
    assert L.lsdb_batch_line_images_device(b.h, host_out.ctypes.data) == ERR_ARG
    assert L.lsdb_batch_line_images_device(b.h, None) == ERR_ARG
    assert L.lsdb_batch_lines_device(None, None, None, None, None, None, 0) == ERR_ARG
    assert L.lsdb_batch_line_images_device(None, None) == ERR_ARG and L.lsdb_batch_map_caches_device(None, None) == ERR_ARG
    sp = C.c_void_p()
    assert L.lsdb_stream(None, C.byref(sp)) == ERR_ARG and L.lsdb_stream(ctx.h, None) == ERR_ARG
    # the context and the batch still work
    b.map_caches(0.05, download=False)
    assert L.lsdb_batch_map_caches_device(b.h, host_cache.ctypes.data) == ERR_ARG
    got = b.lines_device(want_rects=True)
    ims, views = b.line_images_device()
    cs, cviews = b.map_caches_device()
    torch.cuda.synchronize()
    _tables_equal(got, want, n)
    for i in range(n):
        assert np.array_equal(views[i].cpu().numpy(), want["line_ims"][i])
        assert cviews[i].cpu().numpy().tobytes() == want["caches"][i].tobytes()
    b.close(); ctx.close()


def test_another_gpus_memory_is_refused(lsdb, torch):
    if torch.cuda.device_count() < 2:
        pytest.skip("one device")
    m = _ragged(seed=61)[0]
    ctx = lsdb.Context(0)
    b = lsdb.Batch(ctx, [(m.shape[1], m.shape[0])])
    other = torch.from_numpy(m).to("cuda:1")
    arr = (C.c_void_p * 1)(other.data_ptr())
    assert lsdb.lib().lsdb_batch_upload_device(b.h, C.cast(arr, C.c_void_p), None) == ERR_ARG
    b.upload_device([torch.from_numpy(m).cuda()]); b.run()
    cnt = torch.zeros(1, dtype=torch.int32, device="cuda:1"); off = torch.zeros(2, dtype=torch.int32, device="cuda:1")
    assert lsdb.lib().lsdb_batch_lines_device(b.h, cnt.data_ptr(), off.data_ptr(), None, None, None, 0) == ERR_ARG
    got = b.lines_device()
    torch.cuda.synchronize()
    assert int(got["counts"][0]) == int(b.counts()[0])
    b.close(); ctx.close()


def test_context_stream_handle(lsdb, torch):
    s = torch.cuda.Stream()
    ctx = lsdb.Context(0, stream=s.cuda_stream)
    assert ctx.stream == s.cuda_stream
    own = lsdb.Context(0)
    assert own.stream not in (0, s.cuda_stream)
    ctx.close(); own.close()


def test_scan_raster_batch(lsdb, dctx, torch):
    g = np.load(os.path.join(GOLD, "lidar_frames.npz"))
    mp = g["map_param"]
    sweeps = []
    for f in range(24):
        r, a = g[f"f{f}/ranges"], g[f"f{f}/angles"]
        keep = np.isfinite(r)
        sweeps.append((r[keep], a[keep]))
    info = dctx.feature_scan_info(mp[2], mp[3], mp[4], sweeps)
    b = lsdb.Batch(dctx, [(int(i["im_cols"]), int(i["im_rows"])) for i in info], max_lines=512)
    b.upload_scan_rasters(mp[2], mp[3], mp[4], sweeps)
    b.run()
    got = b.lines_device(want_rects=True)
    ims, views = b.line_images_device()
    torch.cuda.synchronize()
    want = b.download(want_rects=True)
    assert sum(want["counts"]) > 0
    _tables_equal(got, want, b.n)
    host_ims = b.line_images()
    for i in range(b.n):
        assert np.array_equal(views[i].cpu().numpy(), host_ims[i]), i
    b.close()


def test_sixteen_4096_maps(lsdb, dctx, torch):
    import bench
    maps = [bench.make_map(4096, k) for k in range(16)]
    want = _host_path(lsdb, dctx, maps)
    b, got, ims, _host_caches, caches = _device_path(lsdb, dctx, maps, torch, [k % 3 for k in range(16)])
    _tables_equal(got, want, len(maps))
    for i in range(len(maps)):
        assert np.array_equal(ims[i].cpu().numpy(), want["line_ims"][i]), i
        assert caches[i].cpu().numpy().tobytes() == want["caches"][i].tobytes(), i
    b.close()
