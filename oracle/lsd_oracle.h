/* TEST INFRASTRUCTURE — CPU restatement of the reference LSD / association hot path.
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
 * use anything under oracle/.  The product (liblsdb200.so) never links or calls this.
 * Parity status: PINNED — checked bit-for-bit against the unmodified reference compiled into
 * oracle/_ref (tests/test_oracle.py) and against tests/golden fixtures generated from it. */
#ifndef LSD_ORACLE_H
#define LSD_ORACLE_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct {
    long long cells;       /* sorted seed-list length (non-zero bins) */
    long long live_seeds;  /* cells whose usedMap was 0 at their turn */
    long long grows;       /* RegionGrower calls */
    long long grown_px;    /* pixels accepted by all grows */
    long long small;       /* regions below regThre */
    long long regrows;     /* Refiner re-grows */
    long long rrr_passes;  /* RegionRadiusReducer shrink passes */
    long long nfa_calls;   /* RectangleNFACalculator calls */
    long long nfa_px;      /* rectangle pixels visited */
    long long rejects;     /* logNFA <= 0 */
    long long accepts;
} lsdo_stats;

/* mylsd::myLineSegmentDetector restated (LSD/myLSD.cpp:129-376).  All output pointers may be NULL.
 *   map      : rows*cols u8, NOT modified;  map_out : the in-place remap the reference applies
 *   gauss/mag/deg : H'*W' f64;  used : H'*W' u8 (0/1/2);  labels : H'*W' int32 (accept index+1,
 *                   un-wrapped; the reference's u8 regIdx equals labels & 0xFF)
 *   seeds    : [n_seeds][3] = bin,x,y in seed order
 *   rects    : [n][13] = x1 y1 x2 y2 wid cX cY deg dx dy p prec logNFA (after the 1/sca rescale)
 *   lines    : [n][10] = k b dx dy x1 y1 x2 y2 len orient;  line_im : rows*cols u8
 * Returns the segment count n (outputs are truncated to max_lines). */
int lsdo_lsd(const uint8_t* map, int cols, int rows, double sca, double sig, double angThre,
             double denThre, int pseBin, uint8_t* map_out, double* gauss, double* mag, double* deg,
             uint8_t* used, int32_t* labels, int32_t* seeds, int max_seeds, int* n_seeds,
             double* rects, double* lines, int max_lines, uint8_t* line_im, lsdo_stats* stats);

/* the three 17-tap phase kernels of GaussianSampler (LSD/myLSD.cpp:398-417); out = [3][2h+1];
 * returns h */
int lsdo_gauss_taps(double sca, double sig, double* out, int cap);

/* debug taps of the next lsdo_lsd calls: the size of every region grown, and the tolerance of every Refiner
 * re-grow (LSD/myLSD.cpp:857), up to cap entries; a NULL buffer turns the tap off */
void lsdo_set_grow_size_log(int* buf, int cap);
int lsdo_grow_size_count(void);
void lsdo_set_regrow_tol_log(double* buf, int cap);
int lsdo_regrow_tol_count(void);
/* debug tap of the next lsdo_lsd calls: every RectangleNFACalculator call as 5 doubles (allPix, aliPix, p, logNT, result),
 * up to cap records; a NULL buffer turns the tap off */
void lsdo_set_nfa_log(double* buf, int cap);
int lsdo_nfa_log_count(void);

/* RectangleNFACalculator after the pixel count (LSD/myLSD.cpp:1006-1059): -log10 NFA of allPix pixels, aliPix of them
 * aligned at precision p.  *exit_idx (may be NULL) = the index i of the binomial-tail loop it broke at, allPix + 1 when
 * the loop ran to the end, or one of the early returns below (csrc/nfa.cuh reports the same codes). */
enum { LSDO_NFA_EXIT_EMPTY = -1,           /* allPix == 0 or aliPix == 0 */
       LSDO_NFA_EXIT_ALL_ALIGNED = -2,     /* allPix == aliPix */
       LSDO_NFA_EXIT_TINY_TERM_HIGH = -3,  /* first term below 100 eps, aliPix > allPix * p */
       LSDO_NFA_EXIT_TINY_TERM_LOW = -4 }; /* first term below 100 eps, otherwise */
double lsdo_nfa_tail(int allPix, int aliPix, double p, double logNT, int* exit_idx);
/* n tails at once; probe (may be NULL) = [n][5] counts of the break tests each tail ran: all of them, m == 1,
 * 0 < |1 - m| <= few, those the device leaves to its correctly rounded pow / log10 when its hardware ones round
 * correctly (|1 - m| < near, or |err - rhs| <= margin * scale, csrc/nfa.cuh), and those a margin without scale's
 * |m^n| / |1 - m| term would leave there */
void lsdo_nfa_tail_many(int n, const int* allPix, const int* aliPix, const double* p, const double* logNT, double few, double near,
                        double margin, double* out, int* exit_idx, int* probe);
/* LogGammaCalculator (LSD/myLSD.cpp:882-924) */
double lsdo_log_gamma(int x);

/* mylsd::createMapCache restated (LSD/myLSD.cpp:11-127) */
void lsdo_map_cache(const uint8_t* map, int cols, int rows, double res, double* out);

/* scoring part of myfa::FeatureAssociation (LSD/myFA.cpp:27-59,186-396), serial.
 * Same record layout as oracle/ref_harness.cpp:ref_fa_scores. */
int lsdo_fa_scores(const double* scan_lines, int n_scan, const double* map_lines, int n_map,
                   const double* pts, int n_pts, const double* map_cache, int cols, int rows,
                   const double* lidar_pose, const double* last_pose, int32_t* out_idx,
                   double* out_val, int max_rec);

/* the catkin snapshot's association (ROS/lsd/src/FeatureAssociation.cpp:36-299), serial: every (scan line, map line of similar
 * length, pairing) hypothesis with its ray re-projection score.  pose_all: T records of 15 doubles = the columns of the reference's
 * 15 x T poseAll; est / est_real = estimatePose / estimatePose_realworld (set when T > 0).  Returns T. */
int lsdo_fa_legacy(const double* scan_lines, int n_scan, const double* map_lines, int n_map, double resol, double ori_x, double ori_y,
                   const int* lidar_pos, int cols, int rows, const double* map_cache, const double* ranges, const double* angles,
                   int n_rays, double* pose_all, int max_cols, double* est, double* est_real);

/* myrdp::FeatureScan restated (LSD/myRDP.cpp:9-375), one frame of finite beams.  map_param = cols rows resol oriX oriY.
 * Same outputs as oracle/ref_harness.cpp:ref_feature_scan: lines [max_lines][10] (k b dx dy x1 y1 x2 y2 len orient),
 * pts [max_pts][2], lidar_pos[2], im_size = cols, rows of the raster, line_im (0/255) when it fits line_im_cap.
 * Returns the number of lines; *n_pts = number of raster samples. */
int lsdo_feature_scan(const double* map_param, const double* range, const double* angle, int n,
                      int leastPoint, double threLine, double leastDistM, double* lines, int max_lines,
                      double* pts, int max_pts, int* n_pts, double* lidar_pos, int* im_size,
                      uint8_t* line_im, int line_im_cap);

long long lsdo_feature_scan_many(const double* map_param, const double* range, const double* angle, const int* beam_off,
                                 int n_frames, long long* n_pts_total);

#ifdef __cplusplus
}
#endif
#endif
