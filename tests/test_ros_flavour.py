"""SURVEY.md §8 f4: the catkin snapshot's flavour of the entry points (ROS/lsd/include/myLSD.h:131-132, called by
LSD/main_on_linux.cpp:130,132): createMapCache(Mat, double res, double z_occ_max_dis) and myLineSegmentDetector(..., double pseBin).

not gpu : the UNMODIFIED ROS/lsd/src/myLSD.cpp (oracle/_ref/libref_ros.so) returns the segment tables of the current source
          except for the direction fields, which go through the snapshot's own (different) atand — so the goldens of the current
          source pin the snapshot's LSD as well;
gpu     : this repo's drop-in bodies built -DLSDB_ROS_FLAVOUR against the snapshot's header (oracle/_ref/libdropin_ros.so)."""
import ctypes as C
import os

import numpy as np
import pytest

import refbind

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_ROS = os.path.join(ROOT, "oracle", "_ref", "libref_ros.so")
DROPIN_ROS = os.path.join(ROOT, "oracle", "_ref", "libdropin_ros.so")
NAMES = ["mapValue", "mapValue_aisle1", "mapValue_map1"]


@pytest.fixture(scope="module")
def gold():
    return np.load(os.path.join(ROOT, "tests", "golden", "bundled_maps.npz"))


def _bind(path):
    L = C.CDLL(path)
    L.ros_lsd.restype = C.c_int
    L.ros_lsd.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, C.c_void_p, C.c_int,
                          C.c_void_p, C.c_void_p]
    return L


def _ros_lsd(L, m, pse_bin=1024.0):
    m = np.ascontiguousarray(m, np.uint8)
    rows, cols = m.shape
    lines = np.zeros((4096, 10)); im = np.zeros((rows, cols), np.uint8); mo = np.zeros((rows, cols), np.uint8)
    n = L.ros_lsd(m.ctypes.data, cols, rows, 0.3, 0.6, 22.5, 0.7, float(pse_bin), lines.ctypes.data, len(lines), im.ctypes.data, mo.ctypes.data)
    return lines[:n].copy(), im, mo


@pytest.mark.skipif(not os.path.exists(REF_ROS), reason="oracle/_ref/libref_ros.so not built")
@pytest.mark.parametrize("name", NAMES)
def test_snapshot_lsd_equals_current_source(gold, name):
    lines, im, mo = _ros_lsd(_bind(REF_ROS), gold[name + "/map"])
    g = gold[name + "/lines"]
    same = [0, 1, 4, 5, 6, 7, 8]                                                 # k b x1 y1 x2 y2 len
    assert lines.shape == g.shape and np.array_equal(lines[:, same], g[:, same], equal_nan=True)
    ang = np.arctan(g[:, 0] / 180.0 * np.pi)                                     # ROS/lsd/src/baseFunc.cpp:14-16
    orient = np.where(ang < 0, -1.0, 1.0); ang = np.where(ang < 0, ang + 180, ang)
    assert np.array_equal(lines[:, 9], orient)
    assert np.allclose(lines[:, 2], np.cos(ang / 180 * np.pi), rtol=1e-12) and np.allclose(lines[:, 3], np.sin(ang / 180 * np.pi), rtol=1e-12)
    assert np.array_equal(np.packbits(im > 0), gold[name + "/line_im_bits"])


@pytest.mark.gpu
@pytest.mark.skipif(not os.path.exists(DROPIN_ROS), reason="oracle/_ref/libdropin_ros.so not built")
def test_ros_flavour_dropin(lsdb, ctx, gold):
    L = _bind(DROPIN_ROS)
    R = _bind(REF_ROS)                                                        # the unmodified snapshot, prebuilt (travels with the repo)
    L.ros_map_cache.restype = None
    L.ros_map_cache.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_double, C.c_void_p]
    for name in NAMES:
        m = gold[name + "/map"]
        lines, im, mo = _ros_lsd(L, m, pse_bin=1024.0)                      # `double pseBin` overload
        rl, rim, rmo = _ros_lsd(R, m, pse_bin=1024.0)
        assert np.array_equal(lines, rl, equal_nan=True)                      # every field, incl. the snapshot's direction fields
        assert np.array_equal(im, rim) and np.array_equal(mo, rmo)
        assert np.array_equal(np.packbits(im > 0), gold[name + "/line_im_bits"])
        remap = m.copy(); sub = remap[1:, 1:]; one = sub == 1; sub[sub == 255] = 0; sub[one] = 255
        assert np.array_equal(mo, remap)                                     # the caller's Mat is remapped in place
        # createMapCache(Mat, res, z_occ_max_dis): the current source's brush fire (pinned to the reference elsewhere) with
        # the truncation distance as an argument and 2 in the cells it never reaches (ROS/lsd/src/myLSD.cpp:37)
        res = float(gold[name + "/param"][2])
        for zmax in (1.0, 0.6):
            out = np.zeros(m.shape, np.float64)
            mm = np.ascontiguousarray(m)
            L.ros_map_cache(mm.ctypes.data, m.shape[1], m.shape[0], res, zmax, out.ctypes.data)
            std = ctx.map_cache(m, res, zmax)
            if refbind.available("glibc") and zmax == 1.0:
                assert np.array_equal(std, refbind.ref_map_cache(m, res))
            unreached = ctx.map_cache(m, res, zmax, unreached=7.0) == 7.0
            assert unreached.any() and np.array_equal(out, np.where(unreached, 2.0, std))


@pytest.mark.gpu
@pytest.mark.skipif(not os.path.exists(DROPIN_ROS), reason="oracle/_ref/libdropin_ros.so not built")
@pytest.mark.parametrize("pse_bin", [512.0, 1.0])
def test_ros_flavour_dropin_other_pse_bins(lsdb, gold, pse_bin):
    """the snapshot takes pseBin as a double and bins with 1.0*pseBin/maxGrad: every integral value must give its segments"""
    L, R = _bind(DROPIN_ROS), _bind(REF_ROS)
    for name in NAMES:
        m = gold[name + "/map"]
        lines, im, mo = _ros_lsd(L, m, pse_bin=pse_bin)
        rl, rim, rmo = _ros_lsd(R, m, pse_bin=pse_bin)
        assert np.array_equal(lines, rl, equal_nan=True), name
        assert np.array_equal(im, rim) and np.array_equal(mo, rmo), name


@pytest.mark.gpu
@pytest.mark.skipif(not os.path.exists(DROPIN_ROS), reason="oracle/_ref/libdropin_ros.so not built")
@pytest.mark.parametrize("pse_bin", [512.5, 0.0, 1025.0, float("nan")])
def test_ros_flavour_dropin_refuses_a_pse_bin_it_cannot_honour(pse_bin):
    """a pseBin the library cannot take as it is (not an integer in [1,1024]) aborts with a message instead of being
    truncated to another seed order; the wrapper has no error channel, so the call runs in a child process"""
    import subprocess
    import sys
    code = ("import sys; sys.path.insert(0, %r); import numpy as np, test_ros_flavour as t\n"
            "g = np.load(%r)\n"
            "t._ros_lsd(t._bind(t.DROPIN_ROS), g['mapValue/map'], pse_bin=float('%s'))\n"
            "print('returned')\n") % (os.path.join(ROOT, "tests"), os.path.join(ROOT, "tests", "golden", "bundled_maps.npz"), pse_bin)
    p = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert p.returncode != 0 and "returned" not in p.stdout
    assert "pseBin" in p.stderr and "not an integer in [1,1024]" in p.stderr
