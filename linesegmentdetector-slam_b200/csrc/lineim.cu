// The lineIm epilogue of myLineSegmentDetector (LSD/myLSD.cpp:296-355) on the device, for all maps of a batch at once: the
// accepted rectangles (already rescaled by commit) are rasterised into one u8 plane per map (255 on the segment, 0 elsewhere),
// which then goes to the host or stays on the device.  Map i's image is either in the batch's own plane (packOff == NULL: at
// srcOff, rows srcPitch bytes apart, the geometry of the source plane) or in a packed caller buffer (map i at packOff[i] =
// sum of rows*cols of the maps before it, rows cols bytes apart).  One warp per segment; a sample is the same double arithmetic as the reference's loop —
// xx = j + xLow, yy = (int)round((xx - x1) * k + y1) along the major axis, samples with x == 0 or y == 0 dropped (:346,:352),
// the marking loop as long as the longer of the two index ranges (:344) — so the image equals the host epilogue's bit for bit.
#include "lsdb_common.cuh"

__global__ void lsdb_line_image_kernel(int nImgs, const LsdbImg* __restrict__ imgs, const LsdbImgDyn* __restrict__ dyn,
                                       const LsdbRect* __restrict__ rects, int maxSeg, uint8_t* __restrict__ plane,
                                       const unsigned long long* __restrict__ packOff) {
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;   // (map, segment) = (warp / maxSeg, warp % maxSeg)
    const int img = warp / maxSeg, seg = warp - img * maxSeg;
    if (img >= nImgs || seg >= dyn[img].nSeg) return;
    const LsdbImg im = imgs[img];
    const LsdbRect& R = rects[(size_t)img * maxSeg + seg];
    const double x1 = R.v[0], y1 = R.v[1], x2 = R.v[2], y2 = R.v[3];
    const double k = (y2 - y1) / (x2 - x1);
    int xLow, xHigh, yLow, yHigh;
    if (x1 > x2) { xLow = lsdb_x86_d2i(floor(x2)); xHigh = lsdb_x86_d2i(ceil(x1)); } else { xLow = lsdb_x86_d2i(floor(x1)); xHigh = lsdb_x86_d2i(ceil(x2)); }
    if (y1 > y2) { yLow = lsdb_x86_d2i(floor(y2)); yHigh = lsdb_x86_d2i(ceil(y1)); } else { yLow = lsdb_x86_d2i(floor(y1)); yHigh = lsdb_x86_d2i(ceil(y2)); }
    const double xRang = fabs(x2 - x1), yRang = fabs(y2 - y1);
    const int xx_len = xHigh - xLow + 1, yy_len = yHigh - yLow + 1;
    const int n = xx_len > yy_len ? xx_len : yy_len;
    uint8_t* out = plane + (packOff ? packOff[img] : im.srcOff);
    const size_t pitch = packOff ? (size_t)im.cols : (size_t)im.srcPitch;
    for (int j = lane; j < n; j += 32) {
        int xx = 0, yy = 0;
        if (xRang > yRang) {
            if (j < xx_len) { xx = j + xLow; yy = lsdb_x86_d2i(round((xx - x1) * k + y1)); }
        } else {
            if (j < yy_len) { yy = j + yLow; xx = lsdb_x86_d2i(round((yy - y1) / k + x1)); }
        }
        if (xx < 0 || xx >= im.cols || yy < 0 || yy >= im.rows) { xx = 0; yy = 0; }
        if (xx != 0 && yy != 0) out[(size_t)yy * pitch + xx] = 255;
    }
}

void lsdb_launch_line_images(cudaStream_t s, int nImgs, int maxSeg, const LsdbImg* imgs, const LsdbImgDyn* dyn, const LsdbRect* rects,
                             uint8_t* plane, const unsigned long long* packOff) {
    if (nImgs <= 0 || maxSeg <= 0) return;
    const long long warps = (long long)nImgs * maxSeg;
    const int perCta = 8;
    lsdb_line_image_kernel<<<(unsigned)((warps + perCta - 1) / perCta), perCta * 32, 0, s>>>(nImgs, imgs, dyn, rects, maxSeg, plane, packOff);
}
