#!/usr/bin/env python3
"""tests/golden/extra_maps.npz: the two further distinct occupancy grids of the reference mount (data_20190513/data_f3key,
1440x979; data_20190514/data_f4key, 1404x707 — BASELINE configs[1] "all bundled maps") through the UNMODIFIED reference
(oracle/_ref, stock glibc): segment table, usedMap, regIdx, sorted seed list.  Needs LSD_REFERENCE_DIR (a checkout of the original)."""
import glob
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import datautil  # noqa: E402
import refbind  # noqa: E402

out = {}
REF_ROOT = os.environ["LSD_REFERENCE_DIR"]
for name, pat in (("f3key", os.path.join(REF_ROOT, "data_20190513/data_f3key/data*/")), ("f4key", os.path.join(REF_ROOT, "data_20190514/data_f4key/data*/"))):
    d = next(x for x in sorted(glob.glob(pat)) if os.path.exists(x + "mapValue.txt") and os.path.exists(x + "mapParam.txt"))
    p = datautil.load_map_param(d + "mapParam.txt")
    m = datautil.load_map_value(d + "mapValue.txt", p["cols"], p["rows"])
    r = refbind.ref_lsd(m, variant="glibc")
    W = r["used"].shape[1]
    out[name + "/map_bits2"] = np.packbits(np.stack([m == 1, m == 255]))   # values are 0 / 1 / 255: two bit planes
    out[name + "/shape"] = np.array(m.shape)
    out[name + "/param"] = np.array([p["cols"], p["rows"], p["res"], p["ori_x"], p["ori_y"]])
    out[name + "/lines"] = r["lines"]
    out[name + "/used"] = r["used"]
    out[name + "/reg_idx"] = r["reg_idx"]
    out[name + "/seeds"] = (r["seeds"][:, 2] * W + r["seeds"][:, 1]).astype(np.int32)
    assert set(np.unique(m)) <= {0, 1, 255}
    print(name, d, m.shape, "segments", r["n"])
np.savez_compressed(os.path.join(ROOT, "tests", "golden", "extra_maps.npz"), **out)
