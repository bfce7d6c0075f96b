"""The LSD path at LSD parameters other than the reference's constants: angThre, denThre and pseBin (arguments 6-8 of
myLineSegmentDetector) against the oracle, bit for bit, plus the argument domain.

The region stage picks its code from these parameters (csrc/grow.cu): the lane-per-seed grower (small_grow) decides the
seeds whose region stays below T = ceil(regThre) pixels when T <= 32 and the tolerance is <= pi/2; every other seed goes
through the warp grower, whose build on the squares serves tolerances <= pi/2 and whose wide build (float pre-test, the
reference's un-wrapped band (pi, 3pi/2], tolerances above pi) serves the rest, including the Refiner's re-grows at
2 sigma.  test_the_sweep_reaches_every_region_path checks on the oracle alone that the sweep below reaches each of them."""
import functools
import math
import os

import numpy as np
import pytest

import oraclebind
import synth
from test_gpu_lsd import _compare_with_oracle, lsdb_env

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "bundled_maps.npz")
ANGLES = [1, 5, 10, 45, 60, 75, 89.9, 90, 90.1, 95, 100, 120, 135, 170, 179]
SG_CAP = 32   # grow.cu: the lane-per-seed grower handles T <= SG_CAP


@functools.lru_cache(maxsize=1)
def sweep_maps():
    """(name, map): small maps (T <= 32 above 90 degrees), medium ones, a bundled map and one 2048^2 map"""
    g = np.load(GOLD)
    return (("60x50", synth.occupancy_grid(60, 50, seed=301)), ("120x100", synth.occupancy_grid(120, 100, seed=3)),
            ("140x110", synth.occupancy_grid(140, 110, seed=5)), ("200x150", synth.occupancy_grid(200, 150, seed=304)),
            ("260x200", synth.occupancy_grid(260, 200, seed=305)), ("700x500", synth.occupancy_grid(700, 500, seed=41)),
            ("1057x771", synth.occupancy_grid(1057, 771, seed=91)),
            ("400x1300_walls", synth.occupancy_grid(400, 1300, seed=92, border_walls=True)),
            ("mapValue_aisle1", g["mapValue_aisle1/map"]), ("2048x2048", synth.occupancy_grid(2048, 2048, seed=93)))


def seed_threshold(m, angThre, sca=0.3):
    """T = ceil(regThre) as lsdb_batch_create and the region stage compute it (api.cu, grow.cu)"""
    W, H = math.floor(m.shape[1] * sca), math.floor(m.shape[0] * sca)
    logNT = 5 * (math.log10(H) + math.log10(W)) / 2.0
    return math.ceil(-logNT / math.log10(angThre / 180.0))


def _run_and_compare(lsdb, ctx, maps, params, check_planes=True):
    b = lsdb.Batch(ctx, [(m.shape[1], m.shape[0]) for _, m in maps], **params)
    b.upload([m for _, m in maps]); b.run()
    got = b.download(want_rects=True)
    try:
        for i, (name, m) in enumerate(maps):
            o = _compare_with_oracle(lsdb, b, i, m, got, check_planes=check_planes, **params)
            st = b.map_stats(i)
            assert (st["accepts"], st["rejects"], st["live_seeds"]) == \
                (o["stats"]["accepts"], o["stats"]["rejects"], o["stats"]["live_seeds"]), name
    finally:
        b.close()


def test_the_sweep_reaches_every_region_path():
    """Host-only, on the oracle: the angThre sweep below grows, at T computed as the product does,
    - with the main tolerance <= pi/2 and > pi/2, each with T <= 32 (lane-per-seed grower or, above pi/2, the warp path)
      and T > 32 (warp path only), seeds whose region stays small and seeds whose region reaches T;
    - Refiner re-grows with a tolerance <= pi/2, in (pi/2, pi] and above pi (the wide grower and its tauGtPi branch)."""
    seen = {}
    tols = []
    for ang in ANGLES:
        for name, m in sweep_maps():
            o = oraclebind.lsd_regrow_tols(m, angThre=ang, want_maps=False, want_line_im=False)
            key = (ang * math.pi / 180 <= math.pi / 2, seed_threshold(m, ang) <= SG_CAP)
            st = o["stats"]   # small: live seeds whose first region stays below regThre, i.e. below T
            s = seen.setdefault(key, [0, 0])
            s[0] += st["small"]; s[1] += st["live_seeds"] - st["small"]
            tols.extend(o["regrow_tols"])
    for key in [(True, True), (True, False), (False, True), (False, False)]:
        assert key in seen and seen[key][0] > 0 and seen[key][1] > 0, (key, seen.get(key))
    tols = np.array(tols)
    assert (tols <= math.pi / 2).sum() > 0
    assert ((tols > math.pi / 2) & (tols <= math.pi)).sum() > 0
    assert (tols > math.pi).sum() > 0


@pytest.mark.gpu
@pytest.mark.parametrize("angThre", ANGLES)
def test_angle_threshold_sweep_vs_oracle(lsdb, ctx, angThre):
    """one batch per tolerance: planes, seeds, used map, labels, rectangles with log-NFA, lines, lineIm and the per-map
    accept / reject / live-seed counters bit for bit.  89.9 / 90 / 90.1 degrees put axis-aligned gradients on the knife edge
    of the angle test (cos 90 degrees = 6e-17); 1 and 179 degrees ban nearly every pixel (gradThre = 114.6)."""
    _run_and_compare(lsdb, ctx, sweep_maps(), dict(angThre=angThre))


def _param_maps():
    keep = ("120x100", "700x500", "400x1300_walls", "mapValue_aisle1", "2048x2048")
    return [(n, m) for n, m in sweep_maps() if n in keep]


@pytest.mark.gpu
@pytest.mark.parametrize("params", [dict(denThre=0.0), dict(denThre=0.3), dict(denThre=1.0), dict(denThre=1.5),
                                    dict(pseBin=1), dict(pseBin=2), dict(pseBin=3), dict(pseBin=7), dict(pseBin=1023),
                                    dict(angThre=100.0, pseBin=1, denThre=1.0)],
                         ids=lambda p: "-".join(f"{k}={v}" for k, v in p.items()))
def test_density_threshold_and_bin_count_vs_oracle(lsdb, ctx, params):
    """denThre from 0 (no Refiner) to 1.5 (Refiner and RegionRadiusReducer on nearly every region); pseBin down to 1, where
    almost every pixel lands in bin 0, which is not a seed"""
    _run_and_compare(lsdb, ctx, _param_maps(), params)


@pytest.mark.gpu
@pytest.mark.parametrize("angThre", [60.0, 100.0])
@pytest.mark.parametrize("env", [dict(LSDB_GROW_WARPS="1"), dict(LSDB_GROW_WARPS="16"), dict(LSDB_GROW_WIDE="0"),
                                 dict(LSDB_GROW_WIDE="1", LSDB_GROW_WARPS="8"), dict(LSDB_NO_SMEM_BAN="1")],
                         ids=lambda e: "-".join(f"{k}={v}" for k, v in e.items()))
def test_wide_tolerance_result_is_independent_of_team_shape(lsdb, ctx, angThre, env):
    """at wide tolerances (T > 32 at 60 degrees on the larger maps; above pi/2 at 100 degrees, where every seed takes the warp
    path) the ordered commit must still give the sequential result whatever the team looks like"""
    maps = [(n, m) for n, m in sweep_maps() if n in ("120x100", "1057x771", "400x1300_walls", "mapValue_aisle1")]
    with lsdb_env(env):
        _run_and_compare(lsdb, ctx, maps, dict(angThre=angThre), check_planes=False)


@pytest.mark.gpu
@pytest.mark.parametrize("angThre", [1.0, 170.0])
@pytest.mark.parametrize("env", [dict(), dict(LSDB_STENCIL_DEFER="5")], ids=["whole_plane", "5_records"])
def test_extreme_gradient_threshold_through_the_stencil_stage(lsdb, ctx, gold_maps_for_stencil, angThre, env):
    """gradThre = 2/sin(angThre): 114.6 at 1 degree (nearly every pixel goes to the banned queue) and 11.5 at 170 degrees;
    the planes, seed lists and segments of the stencil stage against the oracle, with the deferred list at its default size
    and capped at five records (the tiles that do not fit it evaluate their own, banned pixels included)"""
    with lsdb_env(env):
        _run_and_compare(lsdb, ctx, gold_maps_for_stencil, dict(angThre=angThre))


@pytest.fixture(scope="module")
def gold_maps_for_stencil():
    g = np.load(GOLD)
    return [("mapValue", g["mapValue/map"]), ("1057x771", synth.occupancy_grid(1057, 771, seed=91)),
            ("400x1300_walls", synth.occupancy_grid(400, 1300, seed=92, border_walls=True)),
            ("97x45", synth.occupancy_grid(97, 45, seed=12)), ("2048x2048", synth.occupancy_grid(2048, 2048, seed=93))]


@pytest.mark.gpu
def test_parameters_outside_the_domain_are_refused(lsdb, ctx):
    """angThre outside the open interval (0, 180) degrees and a non-finite denThre are LSDB_ERR_ARG from lsdb_batch_create and
    lsdb_lsd alike; the context keeps working"""
    g = np.load(GOLD)
    m = g["mapValue/map"]
    bad = [dict(angThre=a) for a in (0.0, -5.0, 180.0, 200.0, float("nan"), float("inf"))] + \
          [dict(denThre=d) for d in (float("nan"), float("inf"), float("-inf"))]
    for p in bad:
        with pytest.raises(lsdb.LsdbError, match="ARG"):
            lsdb.Batch(ctx, [(m.shape[1], m.shape[0])], **p)
        with pytest.raises(lsdb.LsdbError, match="ARG"):
            ctx.lsd(m, **p)
    assert ctx.lsd(m)["n"] == 41
    edge = dict(angThre=179.9, denThre=-1.0)                   # inside the domain, however far out
    assert ctx.lsd(m, **edge)["n"] == oraclebind.lsd(m, **edge)["n"]
