#!/usr/bin/env python3
"""Golden vectors of the catkin snapshot's association (ROS/lsd/src/FeatureAssociation.cpp), made where LSD_REFERENCE_DIR names a checkout of the original
by the UNMODIFIED source behind oracle/ros_fa_harness.cpp (oracle/_ref/libref_rosfa.so, stock libm): tests/golden/fa_legacy.npz.
Inputs: the bundled map of configs[0] (its LSD lines from tests/golden/bundled_maps.npz, its mapCache with unreached cells at 2.0 as
the snapshot's three-argument createMapCache leaves them), seeded synthetic scan frames / lidar sweeps from the package's synth.py."""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import oraclebind  # noqa: E402
import synth  # noqa: E402

ref = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libref_rosfa.so"))
ref.ros_fa.restype = C.c_int
g = np.load(os.path.join(ROOT, "tests", "golden", "bundled_maps.npz"))
m = g["mapValue/map"]; lines = g["mapValue/lines"]; res = float(g["mapValue/param"][2]); ori = g["mapValue/param"][3:5]
mc = oraclebind.map_cache(m, res)
mc[mc == 1.0] = 2.0                       # cells the distance transform never reached (ROS/lsd/src/myLSD.cpp:11: z_occ_max_dis = 2)
out = dict(n_frames=8, resol=res, ori=np.asarray(ori, np.float64), map_lines=lines)
for f in range(8):
    fr = synth.fake_scan_frame(m, lines, seed=100 + f)
    r, a = synth.lidar_frame(200 + f, n_beams=360 if f % 2 == 0 else 1081)
    if f == 5:
        r = r[:0]; a = a[:0]              # a sweep without beams: 0/0 scores
    if f == 6:
        fr["scan_lines"] = fr["scan_lines"][:0]   # no scan line: no candidate pair, nothing estimated
    pose, est, real = oraclebind.fa_legacy(fr["scan_lines"], lines, res, ori, fr["lidar_pose"], mc, r, a, fn=ref.ros_fa)
    out[f"f{f}/scan_lines"] = fr["scan_lines"]; out[f"f{f}/lidar_pos"] = np.asarray(fr["lidar_pose"], np.int32)
    out[f"f{f}/ranges"] = r; out[f"f{f}/angles"] = a
    out[f"f{f}/pose_all"] = pose; out[f"f{f}/est"] = est; out[f"f{f}/est_real"] = real
    print(f, pose.shape, int(np.isfinite(pose[:, 3]).sum()) if len(pose) else 0, est)
np.savez_compressed(os.path.join(ROOT, "tests", "golden", "fa_legacy.npz"), **out)
