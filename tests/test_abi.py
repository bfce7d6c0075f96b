"""The C-ABI boundary: liblsdb200.so loads, exports every symbol include/lsdb200.h declares, and fails loudly
(no CPU fallback) when no B200 is present."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "lsdb200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(lsdb_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol(lsdb):
    L = lsdb.lib()
    names = _declared()
    assert len(names) >= 20
    for n in names:
        assert hasattr(L, n), n
    assert b"sm_100a" in L.lsdb_version()


def test_struct_layouts_match_reference(lsdb):
    assert lsdb.LINE_DTYPE.itemsize == 80      # sizeof(structLinesInfo), LSD/baseFunc.h:33-44 (9 doubles + int + pad)
    assert lsdb.HYP_DTYPE.itemsize == 48
    assert [lsdb.LINE_DTYPE.fields[f][1] for f in ("k", "b", "dx", "dy", "x1", "y1", "x2", "y2", "len", "orient")] == \
        [0, 8, 16, 24, 32, 40, 48, 56, 64, 72]


def test_no_cpu_fallback(lsdb):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(lsdb.LsdbError):
        lsdb.Context(0)
    h = C.c_void_p()
    assert lsdb.lib().lsdb_create(C.byref(h), 0, None) == 5 and not h     # LSDB_ERR_NO_DEVICE
    assert lsdb.lib().lsdb_batch_run(None) != 0
    # the scan front-end entry points need a context / batch as well
    L = lsdb.lib()
    assert L.lsdb_feature_scan_frames(None, 0.05, 0.0, 0.0, None, 0, None, None, None, None, None, 0, None, None, 0, None, None, 0, None) == 2
    assert L.lsdb_scan_estimate_frames(None, None, 0.05, 0.0, 0.0, None, 0, None, None, None, None, None, None) == 2
    assert L.lsdb_batch_upload_scan_rasters(None, 0.05, 0.0, 0.0, None, 0, None, None, None, None) == 2


def test_product_does_not_touch_the_oracle():
    """nothing under the package or include/ may reference oracle/ (the oracle is test infrastructure)"""
    for base in ("linesegmentdetector-slam_b200", "include"):
        for dp, _, fs in os.walk(os.path.join(ROOT, base)):
            if os.path.basename(dp) == "build":
                continue
            for f in fs:
                if f.endswith((".cu", ".cuh", ".h", ".cpp", ".py", "Makefile")):
                    txt = open(os.path.join(dp, f), errors="ignore").read()
                    assert "lsd_oracle" not in txt and "oraclebind" not in txt and "oracle/" not in txt, os.path.join(dp, f)


def test_dropin_library_keeps_the_reference_entry_points():
    """oracle/_ref/libref_dropin.so = the reference's callers + this repo's C++ bodies for myLSD.h / myFA.h: it must load
    (liblsdb200.so resolves through its rpath) and still define the reference's mangled entry points."""
    import subprocess
    so = os.path.join(ROOT, "oracle", "_ref", "libref_dropin.so")
    if not os.path.exists(so):
        pytest.skip("libref_dropin.so not built (needs LSD_REFERENCE_DIR)")
    L = C.CDLL(so)
    L.ref_variant.restype = C.c_char_p
    assert L.ref_variant() == b"dropin"
    syms = subprocess.run(["nm", "-DC", "--defined-only", so], capture_output=True, text=True).stdout
    assert "mylsd::myLineSegmentDetector(cv::Mat, int, int, double, double, double, double, int)" in syms
    assert "myfa::FeatureAssociation(myfa::_structFAInput*)" in syms
    assert "mylsd::createMapCache(cv::Mat, double)" in syms
    assert "mylsd::myLineSegmentDetector_cpu" in syms and "myfa::FeatureAssociation_cpu" in syms   # the reference bodies, renamed
    assert "mylsd::createMapCache_cpu" in syms
    assert "myrdp::FeatureScan(_structMapParam, myrdp::_structLidarPointPolar*, int, int, double, double)" in syms
    assert "myrdp::FeatureScan_cpu" in syms


def test_header_is_plain_c_and_links(tmp_path):
    """include/lsdb200.h compiles as strict C99 and as C++11, and a C program that calls through it links against
    liblsdb200.so and gets LSDB_ERR_NO_DEVICE / LSDB_ERR_ARG back without a GPU (or a context with one)."""
    import subprocess
    hdr = os.path.join(ROOT, "include", "lsdb200.h")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-fsyntax-only", "-x", "c", hdr])
    subprocess.check_call(["g++", "-std=c++11", "-Wall", "-Werror", "-fsyntax-only", "-x", "c++", hdr])
    src = tmp_path / "abi.c"
    src.write_text('''
#include <stdio.h>
#include "lsdb200.h"
int main(void) {
    lsdb_ctx* ctx = 0;
    int rc = lsdb_create(&ctx, 0, 0);
    lsdb_rdp_params rdp = {3, 0.08, 0.5};
    lsdb_scan_info info;
    int off[2] = {0, 0};
    long long ioff[2];
    int rc2 = lsdb_feature_scan_frames(ctx, 0.05, 0, 0, &rdp, 0, 0, 0, off, &info, 0, 0, off, 0, 0, off, 0, 0, ioff);
    printf("%s %d %d\\n", lsdb_version(), rc, rc2);
    if (ctx) lsdb_destroy(ctx);
    return 0;
}
''')
    exe = tmp_path / "abi"
    pkg = os.path.join(ROOT, "linesegmentdetector-slam_b200")
    subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe), "-L", pkg, "-llsdb200",
                           "-Wl,-rpath," + pkg])
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()
    assert "sm_100a" in " ".join(out[:-2])
    rc, rc2 = int(out[-2]), int(out[-1])
    assert (rc, rc2) in ((5, 2), (0, 0))      # no device: NO_DEVICE then ARG (null context); with a B200: both succeed
