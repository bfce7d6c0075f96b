"""lsdb_fa_legacy_frames: the catkin snapshot's association (ROS/lsd/src/FeatureAssociation.cpp:36-299) for many sweeps in one
call, with the strict-minimum selection of :117-119 and the estimates of :120-127 on the device.

not gpu : LEGACY_EST_DTYPE against the C struct; the selection rule the header states (and the lane-strided merge the reduction
          kernel does) against a literal transcription of the reference's loop; no CPU fallback;
gpu     : the goldens in one call; a batch of seeded frames (beam counts at the warp boundaries of the ray loop, Inf / NaN ranges,
          lidar positions off the map, 0-12 scan lines, three resolutions) against lsdb_fa_legacy frame by frame and the C
          restatement; results independent of how frames are grouped; the output modes, capacity and argument errors; 10 000 frames."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

import oraclebind
import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
PI = 3.14159265358979323846
BEAMS = (0, 1, 31, 32, 33, 360, 1081)


# ---- the selection rule ----

def ref_loop(s):
    """:117-119 as written: t = 0; for i: if (s[i] < s[t]) t = i"""
    t = 0
    for i in range(len(s)):
        if s[i] < s[t]:
            t = i
    return t


def header_rule(s):
    """the rule include/lsdb200.h states: 0 if s[0] is NaN, else the first column whose score == min of the non-NaN scores"""
    s = np.asarray(s, np.float64)
    if np.isnan(s[0]):
        return 0
    return int(np.flatnonzero(s == s[~np.isnan(s)].min())[0])


def _before(a, ca, b, cb):   # fal_before of csrc/fa_legacy.cu
    if a != a:
        return b != b and ca < cb
    return b != b or a < b or (a == b and ca < cb)


def kernel_rule(s):
    """the reduction kernel's selection: 32 lanes strided over the columns, then a butterfly merge with the same order"""
    s = [float(v) for v in s]
    best = [(float("nan"), 2**31 - 1)] * 32
    for c, v in enumerate(s):
        ln = c % 32
        if _before(v, c, *best[ln]):
            best[ln] = (v, c)
    d = 16
    while d:
        best = [best[ln] if not _before(*best[ln ^ d], *best[ln]) else best[ln ^ d] for ln in range(32)]
        d //= 2
    return 0 if s[0] != s[0] else best[0][1]


def _seeded_score_vectors():
    rng = np.random.default_rng(17)
    pool = np.array([np.nan, np.inf, -np.inf, 0.0, -0.0, 1.5, 2.0, 2.0, 3.25])
    out = [np.array([v]) for v in pool]                                   # length 1
    out += [np.full(n, np.inf) for n in (1, 2, 33, 100)]                  # all +inf
    out += [np.full(n, np.nan) for n in (1, 4, 65)]
    out += [np.array([np.nan, 1.0, 0.5]), np.array([1.0, np.nan, 0.5, 0.5]), np.array([0.0, -0.0, -0.0]),
            np.array([-0.0, 0.0]), np.array([np.inf, np.nan, np.inf]), np.array([2.0, np.nan, np.nan, 2.0])]
    for _ in range(400):
        n = int(rng.integers(1, 300))
        v = np.where(rng.random(n) < 0.6, rng.choice(pool, n), np.round(rng.uniform(0, 4, n), int(rng.integers(0, 3))))
        if rng.random() < 0.3:
            v[0] = np.nan
        out.append(v)
    return out


def test_legacy_est_dtype_matches_the_c_struct(lsdb, tmp_path):
    dt = lsdb.LEGACY_EST_DTYPE
    assert dt.itemsize == 64
    assert [dt.fields[f][1] for f in ("n_cols", "best_col", "best_score", "estimate_pose", "estimate_pose_realworld")] == [0, 4, 8, 16, 40]
    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        pytest.skip("no C compiler")
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "lsdb200.h"\n'
                   "#define O(f) (int)offsetof(lsdb_fa_legacy_estimate, f)\n"
                   'int main(void) { printf("%d %d %d %d %d %d\\n", (int)sizeof(lsdb_fa_legacy_estimate), O(n_cols), O(best_col), '
                   "O(best_score), O(estimate_pose), O(estimate_pose_realworld)); return 0; }\n")
    exe = tmp_path / "layout"
    subprocess.check_call([cc, "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    assert got == [64, 0, 4, 8, 16, 40]


def test_selection_rule_equals_the_reference_loop():
    gold = np.load(os.path.join(GOLD, "fa_legacy.npz"))
    vecs = [gold[f"f{f}/pose_all"][:, 3] for f in range(int(gold["n_frames"])) if len(gold[f"f{f}/pose_all"])]
    assert len(vecs) == 7
    for f in range(int(gold["n_frames"])):                              # the goldens' estimates are the record the rule picks
        pose = gold[f"f{f}/pose_all"]
        if len(pose):
            t = header_rule(pose[:, 3])
            assert np.array_equal(gold[f"f{f}/est"], [pose[t, 0], pose[t, 1], pose[t, 2] / 180 * PI])
    vecs += _seeded_score_vectors()
    for s in vecs:
        t = ref_loop(s)
        assert header_rule(s) == t, s
        assert kernel_rule(s) == t, s


def test_no_cpu_fallback_for_the_frames_call(lsdb):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    L = lsdb.lib()
    assert L.lsdb_fa_legacy_frames(None, None, 0, None, None, 0.05, 0.0, 0.0, None, None, None, None, None, None, 0, None) == 2


# ---- on the device ----

@pytest.fixture(scope="module")
def gold():
    return np.load(os.path.join(GOLD, "fa_legacy.npz"))


@pytest.fixture(scope="module")
def cache():
    g = np.load(os.path.join(GOLD, "bundled_maps.npz"))
    mc = oraclebind.map_cache(g["mapValue/map"], float(g["mapValue/param"][2]))
    mc[mc == 1.0] = 2.0        # unreached cells as the snapshot's three-argument createMapCache leaves them (z_occ_max_dis = 2)
    return mc


@pytest.fixture(scope="module")
def fm(lsdb, ctx, gold, cache):
    m = lsdb.FaMap(ctx, cache, gold["map_lines"])
    yield m
    m.close()


def make_frames(n, seed, map_lines, pool=48):
    """n seeded frames composed from a pool of synthetic scans and sweeps: 0-12 scan lines, beam counts cycling through BEAMS,
    Inf / NaN ranges in some, lidar positions off the map in some"""
    g = np.load(os.path.join(GOLD, "bundled_maps.npz"))
    m = g["mapValue/map"]
    rng = np.random.default_rng(seed)
    scans = [synth.fake_scan_frame(m, map_lines, seed=seed * 1000 + i) for i in range(pool)]
    sweeps = [synth.lidar_frame(seed * 1000 + 500 + i, n_beams=1200, dropout=0.0) for i in range(pool)]
    frames = []
    for i in range(n):
        sc = scans[int(rng.integers(pool))]
        sl = sc["scan_lines"]
        sl = sl[rng.permutation(len(sl))[:int(rng.integers(0, 13))]]
        r, a = sweeps[int(rng.integers(pool))]
        nb = BEAMS[i % len(BEAMS)]
        r = np.resize(r, nb).copy(); a = np.resize(a, nb).copy()
        if nb and rng.random() < 0.25:
            k = rng.choice(nb, int(rng.integers(1, max(2, nb // 8))), replace=False)
            r[k] = rng.choice([np.inf, -np.inf, np.nan], len(k))
        lp = np.asarray(sc["lidar_pose"], np.int32)
        if rng.random() < 0.05:
            lp = np.array([-100000, 70000], np.int32)
        frames.append(dict(scan_lines=sl, lidar_pos=lp, ranges=r, angles=a))
    return frames


def _same(a, b):
    """same shape, NaN where the other is NaN, and the same bits everywhere else (so -0 differs from +0)"""
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    if a.shape != b.shape or not np.array_equal(np.isnan(a), np.isnan(b)):
        return False
    k = ~np.isnan(a)
    return np.array_equal(a[k].view(np.int64), b[k].view(np.int64))


def _check_frame(e, pose, want_pose, want_est, want_real):
    """one frame of lsdb_fa_legacy_frames (est record e, pose_all slice) against what the one-frame call / oracle returned"""
    assert _same(pose, want_pose)
    assert e["n_cols"] == len(pose)
    if len(pose) == 0:
        assert e["best_col"] == -1 and np.isnan(e["best_score"])
        assert np.isnan(e["estimate_pose"]).all() and np.isnan(e["estimate_pose_realworld"]).all()
        return
    t = int(e["best_col"])
    assert t == ref_loop(pose[:, 3])
    assert _same(e["best_score"], pose[t, 3])
    assert _same(e["estimate_pose"], want_est) and _same(e["estimate_pose_realworld"], want_real)


@pytest.mark.gpu
def test_goldens_in_one_call(fm, gold):
    n = int(gold["n_frames"])
    frames = [dict(scan_lines=gold[f"f{f}/scan_lines"], lidar_pos=gold[f"f{f}/lidar_pos"], ranges=gold[f"f{f}/ranges"],
                   angles=gold[f"f{f}/angles"]) for f in range(n)]
    est, pose, coff = fm.legacy_frames(frames, float(gold["resol"]), gold["ori"], want_pose_all=True)
    assert len(est) == n and len(coff) == n + 1 and coff[0] == 0 and len(pose) == coff[-1]
    for f in range(n):
        p = pose[coff[f]:coff[f + 1]]
        want = gold[f"f{f}/pose_all"]
        assert np.array_equal(p, want, equal_nan=True)                  # every column, scores included: the unmodified source's bits
        _check_frame(est[f], p, want, gold[f"f{f}/est"], gold[f"f{f}/est_real"])
    assert est[6]["n_cols"] == 0 and est[6]["best_col"] == -1 and np.isnan(est[6]["estimate_pose"]).all()
    s5 = pose[coff[5]:coff[6], 3]
    assert len(s5) and np.isnan(s5).any() and not np.isfinite(s5).any() and est[5]["best_col"] == 0
    assert fm.last_ms() > 0


@pytest.mark.gpu
def test_batch_equals_the_one_frame_call_and_the_oracle(fm, gold, cache):
    ml = gold["map_lines"]
    frames = make_frames(2100, 7, ml)
    n_cols = n_fin = n_off = 0
    for part, (res, ori) in enumerate([(0.025, (-3.5, 2.25)), (0.05, (1.5, -2.0)), (0.1, (0.0, 0.0))]):
        fs = frames[part::3]
        est, pose, coff = fm.legacy_frames(fs, res, ori, want_pose_all=True)
        for f, fr in enumerate(fs):
            p = pose[coff[f]:coff[f + 1]]
            one, oe, orl = fm.legacy(fr["scan_lines"], res, ori, fr["lidar_pos"], fr["ranges"], fr["angles"])
            o = oraclebind.fa_legacy(fr["scan_lines"], ml, res, ori, fr["lidar_pos"], cache, fr["ranges"], fr["angles"])
            assert _same(one, o[0])
            if len(p):
                assert _same(oe, o[1]) and _same(orl, o[2])
            _check_frame(est[f], p, one, o[1], o[2])
            n_cols += len(p); n_fin += int(np.isfinite(p[:, 3]).sum())
            n_off += int(len(p) > 0 and fr["lidar_pos"][0] == -100000)
    assert n_cols > 100000 and n_fin > 10000 and n_off > 10           # the batch is not degenerate


@pytest.mark.gpu
def test_results_do_not_depend_on_grouping(fm, gold):
    frames = make_frames(1000, 11, gold["map_lines"])
    res, ori = 0.05, (1.5, -2.0)

    def per_frame(fs):
        est, pose, coff = fm.legacy_frames(fs, res, ori, want_pose_all=True)
        return [(est[f].tobytes(), pose[coff[f]:coff[f + 1]].tobytes()) for f in range(len(fs))]

    base = per_frame(frames)
    assert per_frame(frames[::-1])[::-1] == base
    perm = np.random.default_rng(3).permutation(len(frames))
    shuffled = per_frame([frames[i] for i in perm])
    assert [shuffled[j] for j in np.argsort(perm)] == base
    for chunk in (1, 7, 500):
        got = []
        for i in range(0, len(frames), chunk):
            got += per_frame(frames[i:i + chunk])
        assert got == base, chunk


@pytest.mark.gpu
def test_modes_capacity_and_argument_errors(lsdb, ctx, fm, gold):
    frames = make_frames(300, 13, gold["map_lines"])
    res, ori = 0.05, (1.5, -2.0)
    est, pose, coff = fm.legacy_frames(frames, res, ori, want_pose_all=True)
    est2, none, coff2 = fm.legacy_frames(frames, res, ori)
    assert none is None and est2.tobytes() == est.tobytes() and np.array_equal(coff2, coff)
    T = int(coff[-1])
    assert T > 0
    with pytest.raises(lsdb.LsdbError, match="CAPACITY"):
        fm.legacy_frames(frames, res, ori, want_pose_all=True, max_cols=T - 1)
    # the same through the C ABI: est / col_off filled, the records buffer untouched
    L = lsdb.lib()
    nf, lines, loff, lp, r, a, roff = fm.pack_legacy(frames)
    p = lsdb._p
    e3 = np.zeros(nf, lsdb.LEGACY_EST_DTYPE); c3 = np.full(nf + 1, -7, np.int32); buf = np.full((T - 1, 15), 1234.5)

    def call(n=nf, lines=lines, loff=loff, lp=lp, r=r, a=a, roff=roff, est=e3, out=buf, max_cols=T - 1, coff=c3, resol=res):
        return L.lsdb_fa_legacy_frames(ctx.h, fm.h, n, p(lines), p(loff), float(resol), float(ori[0]), float(ori[1]), p(lp), p(r), p(a),
                                       p(roff), p(est), p(out), max_cols, p(coff))

    assert call() == 3
    assert e3.tobytes() == est.tobytes() and np.array_equal(c3, coff) and (buf == 1234.5).all()
    full = np.full((T, 15), 1234.5)
    assert call(out=full, max_cols=T) == 0 and _same(full, pose)
    # no frames
    e0, p0, c0 = fm.legacy_frames([], res, ori, want_pose_all=True)
    assert len(e0) == 0 and len(p0) == 0 and list(c0) == [0]
    c1 = np.full(1, -7, np.int32)
    assert L.lsdb_fa_legacy_frames(ctx.h, fm.h, 0, None, None, res, 0.0, 0.0, None, None, None, None, None, None, 0, p(c1)) == 0 and c1[0] == 0
    # argument errors
    bad_l = loff.copy(); bad_l[0] = 1
    dec_r = roff.copy(); dec_r[5] = dec_r[4] - 1
    dec_l = loff.copy(); k = int(np.argmax(np.diff(loff) > 0)); dec_l[k + 1] = dec_l[k] - 1
    bad_r = roff.copy(); bad_r[0] = 2
    cases = dict(offsets_not_at_0=dict(loff=bad_l), ray_offsets_not_at_0=dict(roff=bad_r), lines_decrease=dict(loff=dec_l),
                 rays_decrease=dict(roff=dec_r), null_lines=dict(lines=None), null_ranges=dict(r=None), null_angles=dict(a=None),
                 null_line_off=dict(loff=None), null_ray_off=dict(roff=None), null_est=dict(est=None), null_lidar=dict(lp=None),
                 resol_0=dict(resol=0.0), resol_neg=dict(resol=-0.05), resol_nan=dict(resol=float("nan")), max_cols_neg=dict(max_cols=-1),
                 neg_frames=dict(n=-1))
    for name, kw in cases.items():
        assert call(**kw) == 2, name
        assert "lsdb_fa_legacy_frames" in L.lsdb_last_error(ctx.h).decode(), name
    assert L.lsdb_fa_legacy_frames(None, fm.h, nf, p(lines), p(loff), res, 0.0, 0.0, p(lp), p(r), p(a), p(roff), p(e3), None, 0, None) == 2
    assert L.lsdb_fa_legacy_frames(ctx.h, None, nf, p(lines), p(loff), res, 0.0, 0.0, p(lp), p(r), p(a), p(roff), p(e3), None, 0, None) == 2


@pytest.mark.gpu
def test_angles_beyond_2_19_are_rejected_before_any_launch(lsdb, ctx, fm, gold):
    """A ray angle the device's sin / cos cannot reduce (|a| > LSDB_MAX_ANGLE = 2^19; the kernel adds up to 3 pi) is LSDB_ERR_ARG
    in both entry points, found before any launch: the estimates stay untouched.  +-2^19 itself is accepted, NaN angles keep
    their meaning (the ray falls outside the map), and the context keeps working."""
    frames = make_frames(40, 17, gold["map_lines"])
    res, ori = 0.05, (1.5, -2.0)
    est, pose, coff = fm.legacy_frames(frames, res, ori, want_pose_all=True)
    L = lsdb.lib()
    p = lsdb._p
    nf, lines, loff, lp, r, a, roff = fm.pack_legacy(frames)
    k = int(roff[nf // 2]) + 1                                            # a ray of a frame in the middle of the batch
    fr = next(f for f in frames if len(f["angles"]) > 1 and len(f["scan_lines"]) > 0)
    for bad in (1e22, -1e22, np.nextafter(2.0 ** 19, np.inf), np.inf, -1.7976931348623157e308):
        a2 = a.copy(); a2[k] = bad
        e = np.frombuffer(b"\xab" * est.nbytes, lsdb.LEGACY_EST_DTYPE).copy(); c = np.full(nf + 1, -7, np.int32)
        assert L.lsdb_fa_legacy_frames(ctx.h, fm.h, nf, p(lines), p(loff), res, ori[0], ori[1], p(lp), p(r), p(a2), p(roff), p(e),
                                       None, 0, p(c)) == 2
        assert "lsdb_fa_legacy_frames: the angle of ray %d" % k in L.lsdb_last_error(ctx.h).decode()
        assert (e.view(np.uint8) == 0xAB).all() and (c == -7).all()
        one = np.asarray(fr["angles"], np.float64).copy(); one[1] = bad
        with pytest.raises(lsdb.LsdbError, match="ARG"):
            fm.legacy(fr["scan_lines"], res, ori, fr["lidar_pos"], fr["ranges"], one)
        assert "lsdb_fa_legacy: the angle of ray 1" in L.lsdb_last_error(ctx.h).decode()
    for edge in (2.0 ** 19, -(2.0 ** 19), np.nan):
        one = np.asarray(fr["angles"], np.float64).copy(); one[1] = edge
        fm.legacy(fr["scan_lines"], res, ori, fr["lidar_pos"], fr["ranges"], one)
    est2, pose2, coff2 = fm.legacy_frames(frames, res, ori, want_pose_all=True)
    assert est2.tobytes() == est.tobytes() and _same(pose2, pose) and np.array_equal(coff2, coff)


@pytest.mark.gpu
def test_ten_thousand_frames_in_one_call(fm, gold):
    frames = make_frames(10000, 19, gold["map_lines"])
    res, ori = 0.05, (1.5, -2.0)
    est, pose, coff = fm.legacy_frames(frames, res, ori, want_pose_all=True)
    assert len(est) == 10000 and fm.last_ms() > 0 and len(pose) == coff[-1]
    assert np.array_equal(est["n_cols"], np.diff(coff))
    for f in np.random.default_rng(5).choice(10000, 200, replace=False):
        fr = frames[f]
        one, oe, orl = fm.legacy(fr["scan_lines"], res, ori, fr["lidar_pos"], fr["ranges"], fr["angles"])
        _check_frame(est[f], pose[coff[f]:coff[f + 1]], one, oe, orl)
