"""The reference's text formats through the product's own readers / writer (lsdb_read_map_param / _value / _cache,
lsdb_write_map_cache; SURVEY.md §8b, §8 f1 "also writer/reader").  Host only."""
import os

import numpy as np
import pytest

import datautil
import oraclebind

REF_ROOT = os.environ.get("LSD_REFERENCE_DIR")          # a checkout of the original LineSegmentDetector-SLAM
REF_DATA = os.path.join(REF_ROOT, "data") if REF_ROOT else None


def test_map_cache_file_round_trip(lsdb, tmp_path):
    rng = np.random.default_rng(5)
    m = np.zeros((37, 53), np.uint8); m[rng.integers(0, 37, 40), rng.integers(0, 53, 40)] = 1
    mc = oraclebind.map_cache(m, 0.025)                         # createMapCache (oracle): 0 on the walls, truncated at 1 m
    mc[3, 4] = 1.0 / 3.0; mc[5, 6] = 4.9406564584124654e-324    # values that need all 17 digits / a subnormal
    path = str(tmp_path / "mapCache.txt")
    lsdb.write_map_cache(path, mc)
    back = lsdb.read_map_cache(path, 53, 37)
    assert np.array_equal(back, mc)                             # bit for bit through the text file
    assert np.array_equal(np.loadtxt(path), mc)                 # and it is the rows x cols text the reference reads (LSD/test.cpp:11-17)
    with pytest.raises(lsdb.LsdbError):
        lsdb.read_map_cache(path, 53, 38)                       # short file
    with pytest.raises(lsdb.LsdbError):
        lsdb.read_map_cache(str(tmp_path / "missing.txt"), 53, 37)


def test_map_value_and_param_files(lsdb, tmp_path):
    (tmp_path / "mapParam.txt").write_text("5 3 0.025 -4.43187 -5.49357\n")
    (tmp_path / "mapValue.txt").write_text("-1 0 1 0 -1\n0 1 1 0 255\n-1 -1 0 0 1\n")
    p = lsdb.read_map_param(str(tmp_path / "mapParam.txt"))
    assert p == dict(cols=5, rows=3, res=0.025, ori_x=-4.43187, ori_y=-5.49357)
    v = lsdb.read_map_value(str(tmp_path / "mapValue.txt"), p["cols"], p["rows"])
    assert v.tolist() == [[255, 0, 1, 0, 255], [0, 1, 1, 0, 255], [255, 255, 0, 0, 1]]   # -1 -> 255 (`%d` into a uint8 slot)


@pytest.mark.skipif(not (REF_DATA and os.path.isdir(REF_DATA)), reason="reference data not present (set LSD_REFERENCE_DIR)")
def test_bundled_files_parse_like_the_reference(lsdb):
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "bundled_maps.npz"))
    p = lsdb.read_map_param(os.path.join(REF_DATA, "mapParam.txt"))
    assert (p["cols"], p["rows"], p["res"]) == (1377, 428, 0.025)
    v = lsdb.read_map_value(os.path.join(REF_DATA, "mapValue.txt"), p["cols"], p["rows"])
    assert np.array_equal(v, gold["mapValue/map"])
    assert np.array_equal(v, datautil.load_map_value(os.path.join(REF_DATA, "mapValue.txt"), p["cols"], p["rows"]))
