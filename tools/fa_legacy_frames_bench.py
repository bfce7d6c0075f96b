#!/usr/bin/env python3
"""The catkin snapshot's association over many sweeps: one lsdb_fa_legacy call per frame against one lsdb_fa_legacy_frames call.

Map: the bundled mapValue map, its golden LSD lines and its mapCache with unreached cells at 2.0 (as tests/test_fa_legacy.py
builds them), resolution and origin of tests/golden/fa_legacy.npz.  Frames: N seeded frames, scan lines from synth.fake_scan_frame
(a pool of --pool scans, drawn per frame) and a sweep of its own from synth.lidar_frame, 360 and 1081 beams alternating.

Timings (host clock around work that ends in a synchronise; every mode warmed up first):
  (a) a Python loop of FaMap.legacy, one frame per call;
  (b) one FaMap.legacy_frames call, estimates only;
  (c) the same call with pose_all;
plus the device time of (b)'s and (c)'s kernels (lsdb_fa_last_ms) and the host part of (b) (length filter, staging, copies,
launches).  (b) and (c) start from the packed arrays; packing the frame list
(FaMap.pack_legacy) is timed apart.  (a), (b) and (c) must agree bit for bit.
Writes DIR/fa_legacy_frames_bench.json with the card's name, power limit and maximum SM clock read in the same run.
    python tools/fa_legacy_frames_bench.py --frames 10000 --out DIR"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import oraclebind  # noqa: E402
import synth  # noqa: E402
from __graft_entry__ import load_package  # noqa: E402


def same(a, b):
    """same shape, NaN where the other is NaN, the same bits elsewhere"""
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    if a.shape != b.shape or not np.array_equal(np.isnan(a), np.isnan(b)):
        return False
    k = ~np.isnan(a)
    return bool(np.array_equal(a[k].view(np.int64), b[k].view(np.int64)))


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                             text=True, timeout=60)
        return out.stdout.strip() if out.returncode == 0 else f"nvidia-smi failed: {out.stderr.strip()}"
    except (OSError, subprocess.TimeoutExpired) as e:
        return f"nvidia-smi unavailable: {e}"


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--frames", type=int, default=10000)
    ap.add_argument("--pool", type=int, default=512, help="synthetic scans the frames draw their scan lines from")
    ap.add_argument("--reps", type=int, default=5, help="timed repetitions of (b) and (c)")
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    lsdb = load_package()

    gold = np.load(os.path.join(ROOT, "tests", "golden", "fa_legacy.npz"))
    g = np.load(os.path.join(ROOT, "tests", "golden", "bundled_maps.npz"))
    m = g["mapValue/map"]
    mc = oraclebind.map_cache(m, float(g["mapValue/param"][2]))
    mc[mc == 1.0] = 2.0
    ml = gold["map_lines"]
    res, ori = float(gold["resol"]), gold["ori"]

    rng = np.random.default_rng(a.seed)
    scans = [synth.fake_scan_frame(m, ml, seed=a.seed * 100000 + i) for i in range(a.pool)]
    frames = []
    for i in range(a.frames):
        sc = scans[int(rng.integers(a.pool))]
        r, an = synth.lidar_frame(a.seed * 1000000 + i, n_beams=(360, 1081)[i % 2])
        frames.append(dict(scan_lines=lsdb.array_to_lines(sc["scan_lines"]), lidar_pos=np.asarray(sc["lidar_pose"], np.int32),
                           ranges=r, angles=an))

    ctx = lsdb.Context(0)
    fm = lsdb.FaMap(ctx, mc, ml)

    def loop():
        return [fm.legacy(f["scan_lines"], res, ori, f["lidar_pos"], f["ranges"], f["angles"]) for f in frames]

    # warm-up of every mode
    for f in frames[:64]:
        fm.legacy(f["scan_lines"], res, ori, f["lidar_pos"], f["ranges"], f["angles"])
    fm.legacy_frames(frames, res, ori)
    fm.legacy_frames(frames, res, ori, want_pose_all=True)

    t0 = time.perf_counter(); ra = loop(); ta = time.perf_counter() - t0
    tb, kb, tc, kc, tp = [], [], [], [], []
    for _ in range(a.reps):
        t0 = time.perf_counter(); packed = fm.pack_legacy(frames); tp.append(time.perf_counter() - t0)
        t0 = time.perf_counter(); eb, _, cb = fm.legacy_frames(packed, res, ori); tb.append(time.perf_counter() - t0); kb.append(fm.last_ms())
        t0 = time.perf_counter(); ec, pc, cc = fm.legacy_frames(packed, res, ori, want_pose_all=True); tc.append(time.perf_counter() - t0)
        kc.append(fm.last_ms())

    # (a) = (b) = (c), bit for bit
    ok = eb.tobytes() == ec.tobytes() and np.array_equal(cb, cc)
    T = int(cc[-1])
    for f, (pose, est, real) in enumerate(ra):
        p = pc[cc[f]:cc[f + 1]]
        e = ec[f]
        ok &= same(p, pose) and int(e["n_cols"]) == len(pose)
        if len(pose):
            ok &= same(e["estimate_pose"], est) and same(e["estimate_pose_realworld"], real)
        else:
            ok &= int(e["best_col"]) == -1
    fm.close(); ctx.close()

    med = lambda v: float(np.median(v))  # noqa: E731
    out = dict(
        card=card(),
        frames=a.frames, pool=a.pool, beams=[360, 1081], hypotheses=T, map_lines=int(len(ml)), resol=res,
        bit_exact_a_b_c=bool(ok),
        a_loop_s=ta, a_frames_per_s=a.frames / ta, a_hyp_per_s=T / ta,
        b_estimates_s=med(tb), b_estimates_s_min=float(min(tb)), b_frames_per_s=a.frames / med(tb), b_hyp_per_s=T / med(tb),
        b_kernel_ms=med(kb), b_kernel_hyp_per_s=T / (med(kb) / 1e3),
        b_host_ms=med(tb) * 1e3 - med(kb), b_host_share=(med(tb) * 1e3 - med(kb)) / (med(tb) * 1e3),
        pack_ms=med(tp) * 1e3,
        c_pose_all_s=med(tc), c_pose_all_s_min=float(min(tc)), c_frames_per_s=a.frames / med(tc), c_hyp_per_s=T / med(tc),
        c_kernel_ms=med(kc), c_pose_all_mb=T * 120 / 1e6,
        speedup_b_over_a=ta / med(tb), speedup_c_over_a=ta / med(tc),
    )
    with open(os.path.join(a.out, "fa_legacy_frames_bench.json"), "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps(out))
    if not ok:
        sys.exit("(a), (b) and (c) differ")


if __name__ == "__main__":
    main()
