#!/usr/bin/env python3
"""An LSD batch fed from host memory against one fed from device memory.

Maps: N synthetic occupancy grids of SIZE^2 (bench.make_map, seeds 1000 + i as bench.py).  Per step, one batch on one context:
  (a) host:   pinned host grids -> lsdb_batch_upload -> lsdb_batch_run -> lsdb_batch_download (segment tables, host epilogue)
              + lsdb_batch_line_images into pinned host memory (both synchronise);
  (b) device: the grids already in one CUDA tensor -> lsdb_batch_upload_device -> lsdb_batch_run -> lsdb_batch_lines_device
              (segment tables built on the device) + lsdb_batch_line_images_device into a CUDA tensor; nothing synchronises.
Each arm is warmed up, then timed over STEPS steps with CUDA events on the context stream around the steps and a synchronise
after them (and with the host clock around the same window).  Both arms must give identical segment tables (byte for byte,
rectangles too) and identical line images for every map.  Prints one JSON line with the card's name and power limit, read in
the same run, and writes it to DIR/device_io_bench.json when --out is given.
    python tools/device_io_bench.py --maps 256 --size 4096 --steps 5 [--out DIR]"""
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
import bench  # noqa: E402
from __graft_entry__ import load_package  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60)
        return out.stdout.strip().splitlines()[0] if out.returncode == 0 else f"nvidia-smi failed: {out.stderr.strip()}"
    except (OSError, subprocess.TimeoutExpired, IndexError) as e:
        return f"nvidia-smi unavailable: {e}"


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--maps", type=int, default=256)
    ap.add_argument("--size", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("device_io_bench: no CUDA device (nothing is measured on the CPU)")
    lsdb = load_package()
    n, size = a.maps, a.size
    host = torch.empty((n, size, size), dtype=torch.uint8).pin_memory()
    hnp = host.numpy()
    for i in range(n):
        hnp[i] = bench.make_map(size, i)
    ptrs = [int(hnp[i].ctypes.data) for i in range(n)]
    dev = host.cuda()
    grids = [dev[i] for i in range(n)]
    im_host = torch.empty((n, size, size), dtype=torch.uint8).pin_memory()
    im_views = [im_host.numpy()[i] for i in range(n)]
    im_dev = torch.empty(n * size * size, dtype=torch.uint8, device="cuda")

    ctx = lsdb.Context(0)
    b = lsdb.Batch(ctx, [(size, size)] * n)
    ext = ctx.torch_stream()
    res = {}

    def arm_host():
        b.upload(ptrs); b.run()
        res["a"] = b.download(want_rects=True)
        b.line_images(im_views)

    def arm_device():
        b.upload_device(grids); b.run()
        res["b"] = b.lines_device(want_rects=True)
        b.line_images_device(im_dev)

    def timed(arm):
        for _ in range(a.warmup):
            arm()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(ext)
        for _ in range(a.steps):
            arm()
        e1.record(ext)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / a.steps, (time.perf_counter() - t0) * 1e3 / a.steps

    ms_a, host_ms_a = timed(arm_host)
    ms_b, host_ms_b = timed(arm_device)

    # both arms computed the same maps: tables byte for byte, line images
    ta, tb = res["a"], res["b"]
    counts = tb["counts"].cpu().numpy(); offs = tb["offsets"].cpu().numpy(); st = tb["status"].cpu().numpy()
    lines = tb["lines"].cpu().numpy(); rects = tb["rects"].cpu().numpy()
    same_tables = bool(np.array_equal(counts, ta["counts"]) and not st.any())
    for i in range(n):
        o, c = offs[i], counts[i]
        same_tables &= lines[o:o + c].tobytes() == ta["lines"][i].tobytes() and rects[o:o + c].tobytes() == ta["rects"][i].tobytes()
    same_images = bool(torch.equal(im_host.view(-1).cuda(), im_dev))
    b.close(); ctx.close()

    px = n * size * size
    out = dict(card=card(), maps=n, size=size, steps=a.steps, warmup=a.warmup, segments=int(counts.sum()),
               host_arm_ms_per_step=ms_a, host_arm_gpixel_per_s=px / ms_a / 1e6, host_arm_host_clock_ms=host_ms_a,
               device_arm_ms_per_step=ms_b, device_arm_gpixel_per_s=px / ms_b / 1e6, device_arm_host_clock_ms=host_ms_b,
               speedup=ms_a / ms_b, identical_tables=same_tables, identical_line_images=same_images)
    print(json.dumps(out))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "device_io_bench.json"), "w") as fh:
            json.dump(out, fh, indent=1)
    assert same_tables and same_images, "the host and device arms differ"


if __name__ == "__main__":
    main()
