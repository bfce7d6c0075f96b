// Shared declarations of the sm_100a LSD pipeline (host + device).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "lsd_math.h"

// Per-map geometry, built once on the host (lsdb_batch_create) and read by every kernel.
struct LsdbImg {
    int cols, rows;       // source occupancy grid
    int W, H;             // scaled image: floor(cols*sca), floor(rows*sca)  (LSD/myLSD.cpp:132-133)
    int n;                // W*H
    int srcPitch;         // bytes per source row in the device copy
    int tile0;            // first stencil tile of this map
    int tilesX, tilesY;
    int pw;               // words per row of the ban bitmap: ceil(W/32)
    unsigned long long banOff;   // word offset of the map's ban bitmap (H*pw words)
    unsigned long long srcOff;   // byte offset of the map in the source buffer
    unsigned long long nOff;     // element offset of the map in every per-pixel plane
    unsigned long long segOff;   // element offset into the rect output
    double logNT;                // 5*(log10(H)+log10(W))/2          (LSD/myLSD.cpp:207)
    double regThre;              // -logNT/log10(angThre/180)        (:208)
};

// Per-map results produced on the device.
struct LsdbImgDyn {
    unsigned long long maxGradBits;  // bits of maxGrad (non-negative doubles order like integers)
    int nCells;                      // length of the sorted seed list
    int nSeg;                        // accepted segments
    int err;                         // LSDB_ERR_* raised by a kernel for this map
    int pad_;
    long long stat[32];              // lsdb_stats fields
};

struct LsdbRect { double v[13]; };   // x1 y1 x2 y2 wid cX cY deg dx dy p prec logNFA

// state word per scaled pixel (u32):
//   bit 0      : usedMap == 1 (below gradient threshold, or member of an accepted region)
//   bit 1      : usedMap == 2 (member of an NFA-rejected region)  [bit 0 wins]
//   bit 2 / 3  : pixel belongs to a PARKED (evaluated, not yet retired) accept / reject candidate.  Speculation by
//                later seeds treats a parked accept as already banned and skips seeds inside either kind; whether
//                that guess was right is re-checked pixel by pixel when the dependent evaluation retires.
//   bits 4-19  : pixel is in the region warp w of the owning CTA is currently growing (curMap)
//   bits 20-31 : seed-list chunk (mod 4096) of the seed whose parked region set bit 2/3 (the earliest one)
#define LSDB_ST_BAN 1u
#define LSDB_ST_REJ 2u
#define LSDB_ST_PACC 4u
#define LSDB_ST_PREJ 8u
#define LSDB_ST_WARP_SHIFT 4
#define LSDB_ST_TAG_SHIFT 20

#define LSDB_TILE 32            // stencil output tile (scaled pixels)
#define LSDB_SRC_MAX 136        // max source-window edge of one tile
#define LSDB_SRC_PITCH 160      // bytes per staged source row of a tile (window + 16-byte alignment slack)
#define LSDB_GROW_WARPS 16
#define LSDB_CHUNK 32           // seed-list cells per ordered-commit chunk
#define LSDB_SUPER 8            // chunks a warp claims and speculates on at once (256 cells)

#define LSDB_NP 12
struct LsdbLsdConst {
    double sca, degThre, gradThre, pi, aliPro, denThre;
    double cosDegThre;           // lsdm_cos(degThre)
    double pTab[LSDB_NP], logP[LSDB_NP], log1mP[LSDB_NP], log10P[LSDB_NP];  // p = aliPro/2^k and its logs
    int pseBin, h;
    double taps[3 * 17];
    double axisDeg[3];           // lsdm_atan2 of axis-aligned gradients: 0, +pi/2, -pi/2
    double axisCS[6];            // lsdm_cos, lsdm_sin of those
};

#ifdef __CUDACC__
__device__ __forceinline__ unsigned int lsdb_ld_state(const unsigned int* p) {
    unsigned int v;
    asm volatile("ld.global.cg.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// x86-64 cvttsd2si semantics for (int)double: NaN / out of range -> INT_MIN (SURVEY.md A.9)
__device__ __forceinline__ int lsdb_x86_d2i(double v) {
    if (!(v > -2147483649.0 && v < 2147483648.0)) return (int)0x80000000;
    return __double2int_rz(v);
}
#endif

// launchers (defined in the .cu files, called from api.cu); the stencil launchers return the number of kernels they launched.
// mode (lsdb_stencil_mode(): LSDB_STENCIL / LSDB_STENCIL_G / LSDB_STENCIL_DEFER read when the batch is created): bits 0-1 the cut
// (1: stencil.cu, 2: stencil2.cu), bits 2-4 tiles per CTA of stencil2.cu (1, 2, 4), bit 5 deferred pixels into a second kernel, bits 8.. a cap
// on the records of the deferred list (0: what the scratch plane holds).
int lsdb_stencil_mode(void);
int lsdb_launch_stencil(cudaStream_t s, int nTiles, const LsdbImg* imgs, const int* tileImg, LsdbImgDyn* dyn,
                         const LsdbLsdConst* kc, const uint8_t* src, double* mag, double* deg, double* cosm, double* sinm,
                         unsigned int* state, unsigned int* banBits, unsigned int* nzBits, double* gaussOut, int tileBase,
                         void* deferBuf, size_t deferBytes, int* deferCount, int mode);
// the second cut of the stage (stencil2.cu): what lsdb_launch_stencil runs unless the mode asks for the first.  deferBuf is
// scratch for the launch (pixels whose angle needs the double-double phase), deferCount a zeroed counter in device memory.
int lsdb_launch_stencil_v2(cudaStream_t s, int nTiles, const LsdbImg* imgs, const int* tileImg, LsdbImgDyn* dyn,
                            const LsdbLsdConst* kc, const uint8_t* src, double* mag, double* deg, double* cosm, double* sinm,
                            unsigned int* state, unsigned int* banBits, unsigned int* nzBits, double* gaussOut, int tileBase,
                            void* deferBuf, size_t deferBytes, int* deferCount, int groups);
void lsdb_launch_order(cudaStream_t s, int nImgs, int nBands, const LsdbImg* imgs, LsdbImgDyn* dyn, const LsdbLsdConst* kc,
                       const double* mag, const unsigned int* nzBits, const int2* bandOf, const int2* bandsOfImg, unsigned int* tabs,
                       unsigned short* bins, unsigned int* cells);
size_t lsdb_order_tab_words_per_band(void);
void lsdb_launch_line_images(cudaStream_t s, int nImgs, int maxSeg, const LsdbImg* imgs, const LsdbImgDyn* dyn, const LsdbRect* rects,
                             uint8_t* plane);
void lsdb_launch_grow(cudaStream_t s, int nImgs, int nCtas, int warpsPerCta, const LsdbImg* imgs, LsdbImgDyn* dyn,
                      const LsdbLsdConst* kc, const double* mag, const double* deg, const double* cosm, const double* sinm,
                      unsigned int* state, const unsigned int* cells, int* labels, LsdbRect* rects, int maxSeg,
                      unsigned int* lists, int listCap, int arenaCap, int runAhead, unsigned char* recBuf, const double* lgammaTab, int lgammaN,
                      int* imgCounter, unsigned int* banBits, int bmCapWords, int steal);
size_t lsdb_grow_rec_bytes_per_cta(void);
size_t lsdb_grow_words_per_cta(int listCap, int arenaCap, int warpsPerCta);
void lsdb_launch_lgamma_table(cudaStream_t s, double* tab, int n);
void lsdb_launch_used_plane(cudaStream_t s, const unsigned int* state, uint8_t* used, int n);
int lsdb_grow_max_ctas(int device, int warpsPerCta, int bmCapWords);
int lsdb_grow_max_bitmap_words(int device);

struct LsdbFaTask { int frame, iScan, iMap, pad; };
struct LsdbFaHyp { int frame, iScan, iMap, iPair; double x, y, ang, score; };  // == lsdb_hypothesis
struct LsdbFaLine { double k, b, dx, dy, x1, y1, x2, y2, len; int orient, pad; };  // == lsdb_line
void lsdb_launch_fa(cudaStream_t s, int nTasks, const LsdbFaTask* tasks, const LsdbFaLine* scanLines, const int* scanLineOff,
                    const double* pts, const int* ptOff, const double* lidarPose, const double* lastPose,
                    const LsdbFaLine* mapLines, const double* mapCache, int cols, int rows, double pi, LsdbFaHyp* out, void* poseBuf);
size_t lsdb_fa_pose_bytes(int nTasks);
struct LsdbFaEst { int nHyp, nKept; double bx, by, bang, bscore, mx, my, mang, mscore; };  // == lsdb_fa_estimate
void lsdb_launch_fa_reduce(cudaStream_t s, int nFrames, const LsdbFaHyp* hyp, const int* hypOff, LsdbFaEst* est);
struct LsdbFaLegacyEst { int nCols, bestCol; double bestScore, pose[3], real[3]; };  // == lsdb_fa_legacy_estimate
void lsdb_launch_fa_legacy(cudaStream_t s, int nHyp, const LsdbFaTask* tasks, const LsdbFaLine* scanLines, const int* scanLineOff,
                           const LsdbFaLine* mapLines, const int* lidarPos, const double* mapCache, int cols, int rows, double resol,
                           const double* ranges, const double* angles, const int* rayOff, double* out);
void lsdb_launch_fa_legacy_reduce(cudaStream_t s, int nFrames, const int* colOff, const double* rec, double resol, double oriX, double oriY,
                                  LsdbFaLegacyEst* est);
size_t lsdb_fa_pairs_scratch_ints(int nL);
size_t lsdb_fa_keep_scratch_ints(int nHyp);
void lsdb_launch_fa_keep(cudaStream_t s, int nHyp, const LsdbFaHyp* hyp, double below, int* scratch, LsdbFaHyp* out, int cap);
void lsdb_launch_fa_pairs_count(cudaStream_t s, int nL, const LsdbFaLine* scanLines, const LsdbFaLine* mapLines, int nMap, int* scratch);
void lsdb_launch_fa_pairs_write(cudaStream_t s, int nL, int nFrames, const LsdbFaLine* scanLines, const int* lineOff, const LsdbFaLine* mapLines,
                                int nMap, const int* scratch, LsdbFaTask* tasks, int* hypOff);

// createMapCache of several maps (mapcache.cu).  Map i: cols x rows cells (<= 65535 each) at src + srcOff, srcPitch bytes per
// row; its rows*cols f64 result at cache + cacheOff.  loc is set by lsdb_map_caches_run (the map's first cell in its group).
struct LsdbMcMap { unsigned long long srcOff, cacheOff, loc; int cols, rows, srcPitch, cellRadius; double res; };
int lsdb_mc_cell_radius(double maxDist, double res);
// every map's cache, cell for cell what the map alone gives; synchronises the stream (it reads one count per BFS level)
cudaError_t lsdb_map_caches_run(cudaStream_t s, int nMaps, const LsdbMcMap* maps, const uint8_t* src, double unreached, double* cache);

// scan front-end (fscan.cu)
struct LsdbFsInfo { int nLines, nPts, W, H; double lidarX, lidarY; };  // == lsdb_scan_info; nLines < 0: internal list overflow
struct LsdbFsPiece { double x1, y1, x2, y2; int off, pad; };            // a kept line piece: end points, offset of its samples in the frame
size_t lsdb_fscan_smem(int maxBeams);
int lsdb_launch_fscan_frames(cudaStream_t s, int nFrames, int maxBeams, const double* ranges, const double* angles, const int* beamOff,
                             double resol, double oriX, double oriY, int leastPoint, double threLine, double leastDistM,
                             LsdbFsInfo* info, LsdbFsPiece* pieces);
int lsdb_launch_fscan_lines(cudaStream_t s, int nFrames, int nLinesTotal, const int* beamOff, const LsdbFsInfo* info,
                            const LsdbFsPiece* pieces, const int* lineOff, const int* ptOff, const long long* imOff, const int* imPitch,
                            int imVal, double pi, LsdbFaLine* lines, double* pts, uint8_t* lineIm);
