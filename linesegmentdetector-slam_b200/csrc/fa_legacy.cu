// The catkin snapshot's association on sm_100a (SURVEY.md §8 f4): every (scan line, map line of similar length, end-point
// pairing) hypothesis of any number of lidar frames gets its pose and its ray re-projection score in ONE launch — the replacement
// for the serial loops of /root/reference/ROS/lsd/src/FeatureAssociation.cpp (:36-130 FeatureAssociation, :132-200 ScanToMapMatch,
// :202-252 ScanToMapMatchScore, :254-299 RotateScanIm, :5-34 NormalizedLineDirection).
//
// One WARP per hypothesis.  Lane 0's pose algebra is what every lane computes (same inputs, same FMA-free double code as the
// oracle: lsd_math.h), then the lanes take the frame's rays 32 at a time: each re-projects its ray (correctly rounded cos / sin),
// looks its cell up in mapCache and the warp adds the distances IN RAY ORDER — a serial shuffle chain over the in-range rays —
// so the score has the bits of the reference's sequential sum, not just its value.  Counts are integers and order-free.
// The result record is the column the reference stores in its 15 x T `poseAll` (pose, score, the two end-point quadruples, the
// scan-line / map-line / pairing indices), written at the hypothesis' global column; frames are independent (no pose of one
// frame feeds the next), so a batch of frames gives every frame the bits it gets alone.
// mapCache (8 B per map pixel) stays L2-resident; the stage is FP64-issue-bound.
//
// Then one warp per frame picks the column of :117-119 (`t = 0; if (s[i] < s[t]) t = i`) as a (score, column) arg-min and
// writes the two estimates of :120-127.
#include "lsdb_common.cuh"

#define FAL_THREADS 128
#define FAL_PI 3.14159265358979323846   // M_PI, the snapshot's constant (:2-3)

__device__ double fal_norm_line_dir(double x1, double y1, double x2, double y2) {   // :5-34
    double ang = 0;
    const double dy = y2 - y1, dx = x2 - x1;
    if (dy != 0 && !(dx != 0)) ang = dy > 0 ? 90 : -90;
    else if (!(dy != 0) && dx != 0) ang = dx > 0 ? 0 : 180;
    else ang = lsdm_atan(dy / dx) * 180 / FAL_PI;
    if (dx < 0) {
        if (ang < 0) ang += 180;
        else if (ang > 0) ang -= 180;
    }
    return ang;
}

__global__ void __launch_bounds__(FAL_THREADS) lsdb_fa_legacy_kernel(int nHyp, const LsdbFaTask* __restrict__ tasks,
                                                                     const LsdbFaLine* __restrict__ scanLines, const int* __restrict__ scanLineOff,
                                                                     const LsdbFaLine* __restrict__ mapLines, const int* __restrict__ lidarPos,
                                                                     const double* __restrict__ mapCache, int cols, int rows, double resol,
                                                                     const double* __restrict__ ranges, const double* __restrict__ angles,
                                                                     const int* __restrict__ rayOff, double* __restrict__ out) {
    const unsigned int w = blockIdx.x * (FAL_THREADS / 32) + (threadIdx.x >> 5);
    if (w >= (unsigned int)nHyp) return;
    const int hyp = (int)w, lane = threadIdx.x & 31;   // hyp = the global column
    const LsdbFaTask task = tasks[hyp >> 2];
    const int k = hyp & 3;
    const LsdbFaLine S = scanLines[scanLineOff[task.frame] + task.iScan], M = mapLines[task.iMap];
    const int lidarX = lidarPos[2 * task.frame], lidarY = lidarPos[2 * task.frame + 1];
    const int rayBeg = rayOff[task.frame], nRays = rayOff[task.frame + 1] - rayBeg;
    ranges += rayBeg; angles += rayBeg;
    double mp[4], sp[4];   // the four pairings, :157-182
    if (k < 2) { mp[0] = M.x1; mp[1] = M.y1; mp[2] = M.x2; mp[3] = M.y2; } else { mp[0] = M.x2; mp[1] = M.y2; mp[2] = M.x1; mp[3] = M.y1; }
    if ((k & 1) == 0) { sp[0] = S.x1; sp[1] = S.y1; sp[2] = S.x2; sp[3] = S.y2; } else { sp[0] = S.x2; sp[1] = S.y2; sp[2] = S.x1; sp[3] = S.y1; }
    const double mdir = fal_norm_line_dir(mp[0], mp[1], mp[2], mp[3]);
    const double sdir = fal_norm_line_dir(sp[0], sp[1], sp[2], sp[3]);
    const double angDiff = mdir - sdir;                                                  // RotateScanIm :264
    const double cs = lsdm_cos(angDiff / 180 * FAL_PI), sn = lsdm_sin(angDiff / 180 * FAL_PI);   // :282-283
    const double px = floor((lidarX - sp[0]) * cs - (lidarY - sp[1]) * sn + mp[0]);      // :295-297
    const double py = floor((lidarX - sp[0]) * sn + (lidarY - sp[1]) * cs + mp[1]);
    const double pang = sdir + angDiff;

    double score;
    if (px > cols || px < 1 || py > rows || py < 1) score = INFINITY;                    // :211-212
    else {
        const double th = pang * FAL_PI / 180;
        const double sizeX = (double)(unsigned)cols, sizeY = (double)(unsigned)rows;
        double dist = 0.0;
        int distCount = 0, maxCount = 0, scanLen = 0;
        for (int base = 0; base < nRays; base += 32) {
            const int i = base + lane;
            bool in = false, isMax = false;
            double v = 0.0;
            if (i < nRays) {
                const double r = ranges[i], a = angles[i] + th;
                const double gx = floor(r * lsdm_cos(a) / resol) + px - 1;               // :226-227
                const double gy = floor(r * lsdm_sin(a) / resol) + py - 1;
                if (gx > 1 && gx < sizeX && gy > 1 && gy < sizeY) {                      // :233-234
                    in = true;
                    v = mapCache[(size_t)(int)gy * cols + (int)gx];
                    isMax = v == 2;                                                      // :239
                }
            }
            const unsigned int inM = __ballot_sync(0xffffffffu, in), maxM = __ballot_sync(0xffffffffu, isMax);
            scanLen += __popc(inM); maxCount += __popc(maxM);
            unsigned int dm = inM & ~maxM;
            distCount += __popc(dm);
            while (dm) {                                                                 // :243, in ray order
                const int f = __ffs(dm) - 1;
                dm &= dm - 1;
                dist += __shfl_sync(0xffffffffu, v, f);
            }
        }
        if ((double)scanLen < (double)(size_t)nRays * 0.75) score = INFINITY;            // :248-249
        else score = (dist + 7 * (double)maxCount) / ((double)distCount + (double)maxCount) + 10 * ((double)nRays - (double)scanLen) / (double)nRays;
    }
    if (lane == 0) {
        double* o = out + (size_t)hyp * 15;
        o[0] = px; o[1] = py; o[2] = pang; o[3] = score;
        for (int q = 0; q < 4; q++) { o[4 + q] = mp[q]; o[8 + q] = sp[q]; }
        o[12] = (double)(unsigned)task.iScan; o[13] = (double)(unsigned)task.iMap; o[14] = (double)k;
    }
}

// :117-127 for one frame per warp.  The reference's scan `t = 0; for i: if (s[i] < s[t]) t = i` ends at column 0 when s[0] is NaN
// (every comparison with it is false) and otherwise at the FIRST column whose score == the minimum of the non-NaN scores (-0
// ties +0; a frame of +inf scores keeps 0).  Each lane keeps the best (score, column) of its stride — NaN after every number,
// equal scores to the lower column — and the warp merges them with the same order, so the result does not depend on how the
// columns are spread over lanes.  A selection, no arithmetic: the estimates below are the host's expressions on the chosen
// record (-fmad=false keeps `e * resol + ori` uncontracted).
__device__ __forceinline__ bool fal_before(double a, int ca, double b, int cb) {
    if (a != a) return b != b && ca < cb;
    return b != b || a < b || (a == b && ca < cb);
}

__global__ void __launch_bounds__(FAL_THREADS) lsdb_fa_legacy_reduce_kernel(int nFrames, const int* __restrict__ colOff,
                                                                            const double* __restrict__ rec, double resol, double oriX,
                                                                            double oriY, LsdbFaLegacyEst* __restrict__ est) {
    const unsigned int w = blockIdx.x * (FAL_THREADS / 32) + (threadIdx.x >> 5);
    if (w >= (unsigned int)nFrames) return;
    const int f = (int)w, lane = threadIdx.x & 31;
    const int c0 = colOff[f], c1 = colOff[f + 1];
    double best = NAN;
    int bc = INT_MAX;
    for (int c = c0 + lane; c < c1; c += 32) {
        const double v = rec[(size_t)c * 15 + 3];
        if (fal_before(v, c, best, bc)) { best = v; bc = c; }
    }
    for (int d = 16; d > 0; d >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, best, d);
        const int oc = __shfl_xor_sync(0xffffffffu, bc, d);
        if (fal_before(ov, oc, best, bc)) { best = ov; bc = oc; }
    }
    if (lane != 0) return;
    LsdbFaLegacyEst e;
    e.nCols = c1 - c0;
    if (c1 == c0) {
        e.bestCol = -1; e.bestScore = NAN;
        for (int q = 0; q < 3; q++) { e.pose[q] = NAN; e.real[q] = NAN; }
    } else {
        const int t = rec[(size_t)c0 * 15 + 3] != rec[(size_t)c0 * 15 + 3] ? c0 : bc;
        const double* o = rec + (size_t)t * 15;
        e.bestCol = t - c0; e.bestScore = o[3];
        e.pose[0] = o[0]; e.pose[1] = o[1]; e.pose[2] = o[2] / 180 * FAL_PI;
        e.real[0] = e.pose[0] * resol + oriX; e.real[1] = e.pose[1] * resol + oriY; e.real[2] = e.pose[2];
    }
    est[f] = e;
}

void lsdb_launch_fa_legacy(cudaStream_t s, int nHyp, const LsdbFaTask* tasks, const LsdbFaLine* scanLines, const int* scanLineOff,
                           const LsdbFaLine* mapLines, const int* lidarPos, const double* mapCache, int cols, int rows, double resol,
                           const double* ranges, const double* angles, const int* rayOff, double* out) {
    const int warpsPerCta = FAL_THREADS / 32;
    if (nHyp > 0)
        lsdb_fa_legacy_kernel<<<(unsigned)((nHyp + (long long)warpsPerCta - 1) / warpsPerCta), FAL_THREADS, 0, s>>>(
            nHyp, tasks, scanLines, scanLineOff, mapLines, lidarPos, mapCache, cols, rows, resol, ranges, angles, rayOff, out);
}

void lsdb_launch_fa_legacy_reduce(cudaStream_t s, int nFrames, const int* colOff, const double* rec, double resol, double oriX, double oriY,
                                  LsdbFaLegacyEst* est) {
    const int warpsPerCta = FAL_THREADS / 32;
    if (nFrames > 0)
        lsdb_fa_legacy_reduce_kernel<<<(nFrames + warpsPerCta - 1) / warpsPerCta, FAL_THREADS, 0, s>>>(nFrames, colOff, rec, resol, oriX, oriY, est);
}
