#!/usr/bin/env python3
"""createMapCache for a whole LSD batch: a loop of single-map calls against one lsdb_batch_map_caches call.

Maps: N synthetic occupancy grids of SIZE^2 (synth.occupancy_grid, seeds 1000 + i as bench.py), resolution 0.05, max_dist 1.

Timings (host clock around work that ends in a synchronise; every arm warmed up first):
  (a) a loop of lsdb_map_cache, one map per call, from host buffers into host buffers;
  (b) one lsdb_batch_map_caches call on the uploaded batch, every cache copied to the host;
  (c) the same call, caches kept on the device;
plus lsdb_fa_map_create_from_batch against lsdb_fa_map_create from a host cache and host lines, per association map.
The host copies of (a) and (b) go to one buffer per sampled map and to one shared scratch buffer for the others (a caller
keeping every cache of 256 4096^2 maps on the host would hold 34 GB); the copies are the same either way.
(a), (b) and the oracle agree bit for bit on a seeded sample of maps, and the two kinds of association map score a synthetic
frame with the same bits.  The peak device memory of a (c) call is the largest drop of free device memory (cudaMemGetInfo,
polled every millisecond) below the free memory before the call; the cache plane is already allocated then.
Writes DIR/map_cache_batch_bench.json with the card's name, power limit and maximum SM clock read in the same run.
    python tools/map_cache_batch_bench.py --maps 256 --size 4096 --out DIR"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import oraclebind  # noqa: E402
import synth  # noqa: E402
from __graft_entry__ import load_package  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                             text=True, timeout=60)
        return out.stdout.strip() if out.returncode == 0 else f"nvidia-smi failed: {out.stderr.strip()}"
    except (OSError, subprocess.TimeoutExpired) as e:
        return f"nvidia-smi unavailable: {e}"


def same(a, b):
    a = np.ascontiguousarray(a, np.float64); b = np.ascontiguousarray(b, np.float64)
    return a.shape == b.shape and bool(np.array_equal(a.view(np.int64), b.view(np.int64)))


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--maps", type=int, default=256)
    ap.add_argument("--size", type=int, default=4096)
    ap.add_argument("--res", type=float, default=0.05)
    ap.add_argument("--sample", type=int, default=4, help="maps checked against the oracle")
    ap.add_argument("--reps", type=int, default=3, help="timed repetitions of (b) and (c)")
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    import torch
    lsdb = load_package()
    L = lsdb.lib()
    n, size = a.maps, a.size
    maps = [synth.occupancy_grid(size, size, seed=1000 + i) for i in range(n)]
    sample = sorted(np.random.default_rng(a.seed).choice(n, min(a.sample, n), replace=False).tolist())
    scratch = np.empty((size, size))
    own_a = {k: np.empty((size, size)) for k in sample}
    own_b = {k: np.empty((size, size)) for k in sample}
    ptr = lambda x: x.ctypes.data_as(C.c_void_p)  # noqa: E731

    ctx = lsdb.Context(0)
    b = lsdb.Batch(ctx, [(size, size)] * n)
    b.upload(maps)
    res = np.full(n, a.res)
    outs_b = (C.c_void_p * n)(*[own_b[k].ctypes.data if k in own_b else scratch.ctypes.data for k in range(n)])

    def arm_a():
        for i in range(n):
            ctx.check(L.lsdb_map_cache(ctx.h, ptr(maps[i]), size, size, a.res, 1.0, ptr(own_a.get(i, scratch))), "lsdb_map_cache")

    def arm(out):
        ctx.check(L.lsdb_batch_map_caches(b.h, ptr(res), 1.0, 1.0, out), "lsdb_batch_map_caches")

    # warm-up of every arm
    ctx.check(L.lsdb_map_cache(ctx.h, ptr(maps[0]), size, size, a.res, 1.0, ptr(scratch)), "lsdb_map_cache")
    arm(outs_b); arm(None)

    t0 = time.perf_counter(); arm_a(); ta = time.perf_counter() - t0
    tb, tc = [], []
    for _ in range(a.reps):
        t0 = time.perf_counter(); arm(outs_b); tb.append(time.perf_counter() - t0)
        t0 = time.perf_counter(); arm(None); tc.append(time.perf_counter() - t0)

    # peak device memory of one (c) call
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info(0)[0]
    low = [free0]
    done = threading.Event()

    def poll():
        while not done.is_set():
            low[0] = min(low[0], torch.cuda.mem_get_info(0)[0])
            time.sleep(0.001)
    th = threading.Thread(target=poll); th.start()
    arm(None)
    done.set(); th.join()
    peak_gb = (free0 - low[0]) / 1e9

    ok = True
    for k in sample:
        want = oraclebind.map_cache(maps[k], a.res)
        ok &= same(own_a[k], want) and same(own_b[k], want)

    # association maps: straight from the batch against from host buffers
    b.run()
    lines = b.download()["lines"]
    arm(None)
    tf_b, tf_h = [], []
    for k in sample:
        h = C.c_void_p()
        lk = np.ascontiguousarray(lines[k])
        t0 = time.perf_counter(); ctx.check(L.lsdb_fa_map_create_from_batch(b.h, k, C.byref(h)), "from_batch"); tf_b.append(time.perf_counter() - t0)
        L.lsdb_fa_map_destroy(h)
        t0 = time.perf_counter(); ctx.check(L.lsdb_fa_map_create(ctx.h, ptr(own_b[k]), size, size, ptr(lk), len(lk), C.byref(h)), "create")
        tf_h.append(time.perf_counter() - t0)
        L.lsdb_fa_map_destroy(h)
        fb = lsdb.FaMap.from_batch(b, k)
        fh = lsdb.FaMap(ctx, own_b[k], lines[k])
        fr = synth.fake_scan_frame(maps[k], lsdb.lines_to_array(lines[k]), seed=7 + k)
        ok &= fb.score([fr]).tobytes() == fh.score([fr]).tobytes()
        fb.close(); fh.close()
    b.close(); ctx.close()

    med = lambda v: float(np.median(v))  # noqa: E731
    cells = n * size * size
    out = dict(
        card=card(),
        maps=n, size=size, res=a.res, max_dist=1.0, sample=sample,
        bit_exact_a_b_oracle_and_fa_maps=bool(ok),
        a_loop_s=ta, a_ms_per_map=ta / n * 1e3,
        b_batch_host_copies_s=med(tb), b_s_min=float(min(tb)), b_ms_per_map=med(tb) / n * 1e3,
        c_batch_device_only_s=med(tc), c_s_min=float(min(tc)), c_ms_per_map=med(tc) / n * 1e3, c_gcells_per_s=cells / med(tc) / 1e9,
        c_transient_peak_device_gb=peak_gb, cache_plane_gb=cells * 8 / 1e9,
        speedup_b_over_a=ta / med(tb), speedup_c_over_a=ta / med(tc),
        fa_map_from_batch_ms=med(tf_b) * 1e3, fa_map_from_host_ms=med(tf_h) * 1e3,
    )
    with open(os.path.join(a.out, "map_cache_batch_bench.json"), "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps(out))
    if not ok:
        sys.exit("(a), (b), the oracle or the association maps differ")


if __name__ == "__main__":
    main()
