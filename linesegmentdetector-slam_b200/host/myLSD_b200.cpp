// Drop-in bodies for mylsd::myLineSegmentDetector (reference LSD/myLSD.h:132, LSD/myLSD.cpp:129-376) and
// mylsd::createMapCache (LSD/myLSD.h:131, LSD/myLSD.cpp:11-127).
//
// Compiled against the reference's own myLSD.h (so the signatures, structLSD and structLinesInfo are the
// reference's, not copies) and linked with liblsdb200.so.  The reference's two bodies are renamed out of
// the way at compile time (-DmyLineSegmentDetector=myLineSegmentDetector_cpu
// -DcreateMapCache=createMapCache_cpu on the myLSD.cpp TU, see INTEGRATION.md) or simply deleted by the
// maintainer; define LSDB_KEEP_CPU_MAP_CACHE here (and drop the second rename) to keep the reference's
// createMapCache.
//
// Contract kept from the reference:
//   * MapGray is a shallow, ref-counted copy, so the 1->255 / 255->0 remap (rows, cols >= 1 only) is
//     written back into the CALLER's pixels (LSD/myLSD.cpp:135-142); main_on_windows.cpp relies on
//     createMapCache having run first (LSD/main_on_windows.cpp:67-70).
//   * linesInfo is malloc'd here and owned by the caller (never freed by the reference's callers, :281).
//   * lineIm is a fresh CV_8UC1 Mat of oriMapRow x oriMapCol (:215).
//   * no error channel: failures abort with the library's message.
#include <myLSD.h>

#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <vector>

#include "lsdb_host.h"

static_assert(sizeof(structLinesInfo) == sizeof(lsdb_line), "structLinesInfo layout (LSD/baseFunc.h:33-44)");

// The catkin snapshot of the header (ROS/lsd/include/myLSD.h:131-132, used by LSD/main_on_linux.cpp:130,132) declares
//   Mat createMapCache(Mat MapGray, double res, double z_occ_max_dis);
//   structLSD myLineSegmentDetector(..., double pseBin);
// build this file with -DLSDB_ROS_FLAVOUR (implies LSDB_PSEBIN_T=double) against that header for the ROS node.
#ifdef LSDB_ROS_FLAVOUR
#define LSDB_PSEBIN_T double
#endif
#ifndef LSDB_PSEBIN_T
#define LSDB_PSEBIN_T int
#endif

namespace mylsd {

structLSD myLineSegmentDetector(Mat MapGray, int oriMapCol, int oriMapRow, double sca, double sig, double angThre,
                                double denThre, LSDB_PSEBIN_T pseBin) {
#ifdef LSDB_ROS_FLAVOUR
    // The snapshot bins with zoom = 1.0*pseBin/maxGrad on the double (as LSD/myLSD.cpp:179 does on the int): a fractional
    // pseBin gives another seed order than any integer the library takes, so it is refused instead of truncated.
    if (!(pseBin >= 1 && pseBin <= 1024 && pseBin == (double)(int)pseBin)) {
        fprintf(stderr, "lsdb200: myLineSegmentDetector: pseBin %.17g is not an integer in [1,1024]; the library bins with an integer pseBin\n",
                (double)pseBin);
        abort();
    }
#endif
    lsdb_ctx* ctx = lsdb_host::context();
    const size_t npx = (size_t)oriMapCol * oriMapRow;
    std::vector<uint8_t> in(npx), remapped(npx), lineIm(npx);
    for (int y = 0; y < oriMapRow; y++) memcpy(&in[(size_t)y * oriMapCol], MapGray.ptr<uint8_t>(y), (size_t)oriMapCol);

    lsdb_lsd_params prm;
    prm.sca = sca; prm.sig = sig; prm.angThre = angThre; prm.denThre = denThre; prm.pseBin = (int)pseBin; prm._pad = 0;
    // the reference has no limit on the number of segments: when the table is too small, ask again with a bigger one
    int cap = 4096;
    std::vector<lsdb_line> lines(cap);
    int n = 0;
    int rc = lsdb_lsd(ctx, in.data(), oriMapCol, oriMapRow, &prm, lines.data(), cap, &n, lineIm.data(), remapped.data());
    while (rc == LSDB_ERR_CAPACITY && cap < (1 << 20)) {
        cap *= 4;
        lines.resize(cap);
        rc = lsdb_lsd(ctx, in.data(), oriMapCol, oriMapRow, &prm, lines.data(), cap, &n, lineIm.data(), remapped.data());
    }
    if (rc != LSDB_OK) lsdb_host::die("lsdb_lsd", rc);

    for (int y = 0; y < oriMapRow; y++) memcpy(MapGray.ptr<uint8_t>(y), &remapped[(size_t)y * oriMapCol], (size_t)oriMapCol);

    structLSD out;
    out.lineIm = Mat::zeros(oriMapRow, oriMapCol, CV_8UC1);
    for (int y = 0; y < oriMapRow; y++) memcpy(out.lineIm.ptr<uint8_t>(y), &lineIm[(size_t)y * oriMapCol], (size_t)oriMapCol);
    out.len_linesInfo = n;
    out.linesInfo = (structLinesInfo*)malloc(sizeof(structLinesInfo) * (size_t)(n > 0 ? n : 1));
    for (int i = 0; i < n; i++) {
        structLinesInfo& L = out.linesInfo[i];
        const lsdb_line& s = lines[i];
        L.k = s.k; L.b = s.b; L.dx = s.dx; L.dy = s.dy; L.x1 = s.x1; L.y1 = s.y1; L.x2 = s.x2; L.y2 = s.y2;
        L.len = s.len; L.orient = s.orient;
#ifdef LSDB_ROS_FLAVOUR
        // The snapshot's atand is atan(x / 180 * pi) (ROS/lsd/src/baseFunc.cpp:14-16; the current source: atan(x) * 180 / pi),
        // so its direction fields differ (ROS/lsd/src/myLSD.cpp:289-293,357-358): recomputed with the tree's OWN atand / cosd /
        // sind, i.e. whatever the node links, from the same slope.
        double ang = atand(s.k);
        int orient = 1;
        if (ang < 0) { ang += 180; orient = -1; }
        L.dx = cosd(ang); L.dy = sind(ang); L.orient = orient;
#endif
    }
    return out;
}

#if defined(LSDB_ROS_FLAVOUR) && !defined(LSDB_KEEP_CPU_MAP_CACHE)
// ROS/lsd/src/myLSD.cpp:11-127: the same brush fire with the truncation distance as an argument; cells it never reaches hold
// the literal 2 (:37).  The snapshot's down / right neighbour tests read one row / column past the map (:86,:105, undefined
// behaviour); the bounds of the current source (LSD/myLSD.cpp:86,105) are what is computed here.
Mat createMapCache(Mat MapGray, double res, double z_occ_max_dis) {
    lsdb_ctx* ctx = lsdb_host::context();
    const int rows = MapGray.rows, cols = MapGray.cols;
    std::vector<uint8_t> in((size_t)rows * cols);
    for (int y = 0; y < rows; y++) memcpy(&in[(size_t)y * cols], MapGray.ptr<uint8_t>(y), (size_t)cols);
    std::vector<double> out((size_t)rows * cols);
    const int rc = lsdb_map_cache_fill(ctx, in.data(), cols, rows, res, z_occ_max_dis, 2.0, out.data());
    if (rc != LSDB_OK) lsdb_host::die("lsdb_map_cache_fill", rc);
    Mat mapCache = Mat::zeros(rows, cols, CV_64FC1);
    for (int y = 0; y < rows; y++) memcpy(mapCache.ptr<double>(y), &out[(size_t)y * cols], sizeof(double) * (size_t)cols);
    return mapCache;
}
#elif !defined(LSDB_KEEP_CPU_MAP_CACHE)
// The truncated distance map the association scores against; reads MapGray BEFORE the LSD remap (callers run it
// first, LSD/main_on_windows.cpp:67-70).  Fresh CV_64FC1 Mat, rows x cols, metres.
Mat createMapCache(Mat MapGray, double res) {
    lsdb_ctx* ctx = lsdb_host::context();
    const int rows = MapGray.rows, cols = MapGray.cols;
    std::vector<uint8_t> in((size_t)rows * cols);
    for (int y = 0; y < rows; y++) memcpy(&in[(size_t)y * cols], MapGray.ptr<uint8_t>(y), (size_t)cols);
    std::vector<double> out((size_t)rows * cols);
    const int rc = lsdb_map_cache(ctx, in.data(), cols, rows, res, z_occ_max_dis, out.data());
    if (rc != LSDB_OK) lsdb_host::die("lsdb_map_cache", rc);
    Mat mapCache = Mat::zeros(rows, cols, CV_64FC1);
    for (int y = 0; y < rows; y++) memcpy(mapCache.ptr<double>(y), &out[(size_t)y * cols], sizeof(double) * (size_t)cols);
    return mapCache;
}
#endif

}  // namespace mylsd
