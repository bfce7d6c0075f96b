#!/usr/bin/env python3
"""Generates tests/golden/*.npz from the UNMODIFIED reference compiled into oracle/_ref (stock glibc variant).

Needs oracle/_ref, built from the checkout LSD_REFERENCE_DIR names:  LSD_REFERENCE_DIR=... python tools/make_golden.py
  bundled_maps.npz : the six bundled occupancy grids (inputs, u8) and the reference's outputs for each:
                     segment table, usedMap, regIdx, sorted seed list, lineIm (bit-packed)
  fa_frames.npz    : the first frames of data/Lidar.txt pushed through the reference's own RDP front-end
                     (myrdp::FeatureScan) and scored by the reference's NormalizedLineDirection /
                     rotateScanIm / CalcScore against LSD(data/mapValue.txt) and its mapCache."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import datautil  # noqa: E402
import refbind  # noqa: E402

REF_ROOT = os.environ["LSD_REFERENCE_DIR"]
D = os.path.join(REF_ROOT, "data") + "/"
MAPS = [("mapValue", "mapParam"), ("mapValue_aisle1", "mapParam_aisle1"), ("mapValue_aisle2", "mapParam_aisle2"),
        ("mapValue_aisle3", "mapParam_aisle3"), ("mapValue_map1", "mapParam_map1"), ("mapValue_map2", "mapParam_map1")]
out = {}
for name, par in MAPS:
    p = datautil.load_map_param(D + par + ".txt")
    m = datautil.load_map_value(D + name + ".txt", p["cols"], p["rows"])
    r = refbind.ref_lsd(m, variant="glibc")
    W = r["used"].shape[1]
    out[name + "/map"] = m
    out[name + "/param"] = np.array([p["cols"], p["rows"], p["res"], p["ori_x"], p["ori_y"]])
    out[name + "/lines"] = r["lines"]
    out[name + "/used"] = r["used"]
    out[name + "/reg_idx"] = r["reg_idx"]
    out[name + "/seeds"] = (r["seeds"][:, 2] * W + r["seeds"][:, 1]).astype(np.int32)
    out[name + "/seed_bins"] = r["seeds"][:, 0].astype(np.int16)
    out[name + "/line_im_bits"] = np.packbits(r["line_im"] > 0)
    print(name, m.shape, "segments", r["n"], "seeds", len(r["seeds"]))
np.savez_compressed(os.path.join(ROOT, "tests", "golden", "bundled_maps.npz"), **out)

# association fixture
p = datautil.load_map_param(D + "mapParam.txt")
m = datautil.load_map_value(D + "mapValue.txt", p["cols"], p["rows"])
mc = refbind.ref_map_cache(m, p["res"])
map_lines = refbind.ref_lsd(m)["lines"]
frames = datautil.load_lidar_frames(D + "Lidar.txt")
fa = {"map_lines": map_lines, "n_frames": np.array(12)}
mp = [p["cols"], p["rows"], p["res"], p["ori_x"], p["ori_y"]]
for f in range(12):
    rng_, ang_ = frames[f * 8]
    fs = refbind.ref_feature_scan(mp, rng_, ang_)
    lidar = np.rint(fs["lidar_pos"])  # (int)round, LSD/main_on_windows.cpp:229-230
    last = np.array([-1.0, -1.0, 0.0]) if f % 2 == 0 else np.array([lidar[0] + 700.0, lidar[1] + 150.0, 0.0])
    idx, val = refbind.ref_fa_scores(fs["lines"], map_lines, fs["pts"], mc, lidar, last)
    fa[f"f{f}/scan_lines"] = fs["lines"]; fa[f"f{f}/pts"] = fs["pts"]; fa[f"f{f}/lidar_pose"] = lidar
    fa[f"f{f}/last_pose"] = last; fa[f"f{f}/idx"] = idx; fa[f"f{f}/val"] = val
    # the frame's scan raster (myrdp::FeatureScan lineIm, 0/255), bit-packed: the LSD-on-scan workload of BASELINE configs[3]
    fa[f"f{f}/scan_im_bits"] = np.packbits(fs["line_im"] > 0); fa[f"f{f}/scan_im_shape"] = np.array(fs["line_im"].shape)
    occ = (fs["line_im"] > 0).astype(np.uint8)            # mapValue convention: occupied = 1
    fa[f"f{f}/scan_lsd_lines"] = refbind.ref_lsd(occ, want_maps=False)["lines"]
    print("frame", f * 8, "lines", len(fs["lines"]), "pts", len(fs["pts"]), "hyp", len(idx), "kept(<3)", int((val[:, 3] < 3).sum()))
np.savez_compressed(os.path.join(ROOT, "tests", "golden", "fa_frames.npz"), **fa)

# scan front-end fixture: raw lidar frames (Inf beams included, as in Lidar.txt) and what the reference's
# myrdp::FeatureScan makes of them.  Oracle (ii) build (portable math = the device's arithmetic); `glibc_same` records
# whether the stock-glibc build gives the identical result for that frame.
import glob  # noqa: E402
picks = [(D + "Lidar.txt", list(range(0, 96, 8)))]
for fn in sorted(glob.glob(os.path.join(REF_ROOT, "data_2019051*/data_f*key/data*/Lidar.txt"))):
    picks.append((fn, [5, 31, 35, 119]))
ls = {}
k = 0
for fn, idxs in picks:
    raw = np.loadtxt(fn).reshape(-1, 2)
    for i in idxs:
        if (i + 1) * 360 > len(raw):
            continue
        fr = raw[i * 360:(i + 1) * 360]
        keep = np.isfinite(fr[:, 0])
        a = refbind.ref_feature_scan(mp, fr[keep, 0], fr[keep, 1], variant="lsdm")
        g = refbind.ref_feature_scan(mp, fr[keep, 0], fr[keep, 1], variant="glibc")
        same = (a["size"] == g["size"] and np.array_equal(a["lines"], g["lines"], equal_nan=True) and np.array_equal(a["pts"], g["pts"]))
        ls[f"f{k}/ranges"] = fr[:, 0].copy(); ls[f"f{k}/angles"] = fr[:, 1].copy()
        ls[f"f{k}/lines"] = a["lines"]; ls[f"f{k}/pts"] = a["pts"].astype(np.int32)
        ls[f"f{k}/lidar_pos"] = a["lidar_pos"].copy(); ls[f"f{k}/size"] = np.array(a["size"]); ls[f"f{k}/glibc_same"] = np.array(same)
        k += 1
ls["n_frames"] = np.array(k); ls["map_param"] = np.array(mp, np.float64)
print("lidar frames", k, "glibc-identical", sum(bool(ls[f"f{i}/glibc_same"]) for i in range(k)))
np.savez_compressed(os.path.join(ROOT, "tests", "golden", "lidar_frames.npz"), **ls)
for f in ("bundled_maps.npz", "fa_frames.npz", "lidar_frames.npz"):
    print(f, os.path.getsize(os.path.join(ROOT, "tests", "golden", f)) // 1024, "KiB")
