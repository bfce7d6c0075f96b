/* lsdb200.h — C ABI of the B200-native LSD / association hot path (liblsdb200.so).
 *
 * This is the drop-in boundary: plain pointers and sizes, no C++/torch types.  Each entry point
 * names the reference interface it replaces (paths relative to the reference repo):
 *
 *   lsdb_lsd / lsdb_batch_*   <- mylsd::myLineSegmentDetector          LSD/myLSD.h:132, LSD/myLSD.cpp:129-376
 *                                 (stage functions LSD/myLSD.h:133-141 have no external callers)
 *   lsdb_line                 <- structLinesInfo                        LSD/baseFunc.h:33-44
 *   lsdb_lsd_params           <- lsd_sca/lsd_sig/lsd_angThre/lsd_denThre/pseBin   LSD/baseFunc.h:64-68
 *   lsdb_fa_map_* / lsdb_fa_score <- the scoring half of myfa::FeatureAssociation
 *                                 LSD/myFA.h:83-87, LSD/myFA.cpp:27-63 (dispatch), :186-272
 *                                 (thread_ScanToMapMatch), :274-305, :307-355, :357-396
 *   lsdb_hypothesis           <- structScore                            LSD/myFA.h:49-54
 *   lsdb_map_cache            <- mylsd::createMapCache                  LSD/myLSD.h:131, LSD/myLSD.cpp:11-127
 *   lsdb_batch_map_caches     <- the same for every map of a batch, on the device
 *
 * There is no CPU fallback: every compute entry point fails with LSDB_ERR_NO_DEVICE / LSDB_ERR_CUDA
 * when no sm_100 device is usable.  All functions return LSDB_OK (0) or an error code; the text of
 * the last error is available from lsdb_last_error().  A context is not thread-safe; use one per
 * host thread / GPU.
 */
#ifndef LSDB200_H
#define LSDB200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LSDB_OK 0
#define LSDB_ERR_CUDA 1       /* a CUDA call or kernel failed */
#define LSDB_ERR_ARG 2        /* invalid argument */
#define LSDB_ERR_CAPACITY 3   /* an output/region capacity was exceeded (see message) */
#define LSDB_ERR_TIMEOUT 4    /* device-side watchdog fired (ordered-commit pipeline stalled) */
#define LSDB_ERR_NO_DEVICE 5  /* no usable CUDA device */

/* Largest |angle| (radians) a caller may pass as a beam / ray angle (lsdb_feature_scan_frames, lsdb_fa_legacy,
 * lsdb_fa_legacy_frames): 2^19.  The device's sin / cos are exact-reduction, correctly rounded functions up to 2^20 and NaN
 * beyond; the association adds up to 3 pi to a ray's angle, so 2^19 leaves headroom.  Larger angles are LSDB_ERR_ARG. */
#define LSDB_MAX_ANGLE 524288.0

typedef struct lsdb_ctx lsdb_ctx;
typedef struct lsdb_batch lsdb_batch;
typedef struct lsdb_fa_map lsdb_fa_map;

/* arguments 4-8 of myLineSegmentDetector (LSD/myLSD.h:132); defaults LSD/baseFunc.h:64-68.
 * Domain (lsdb_batch_create and lsdb_lsd return LSDB_ERR_ARG outside it, before anything is allocated):
 * sca in (0,1], angThre in the open interval (0,180) degrees, denThre finite, pseBin in [1,1024].  Inside it the result is
 * the reference's for any value (tests/test_gpu_lsd_params.py sweeps angThre from 1 to 179, denThre from 0 to 1.5, pseBin
 * from 1 to 1023). */
typedef struct {
    double sca;      /* 0.3  (the 3-phase Gaussian is only defined for 0.3, LSD/baseFunc.h:64) */
    double sig;      /* 0.6  */
    double angThre;  /* 22.5 */
    double denThre;  /* 0.7  */
    int pseBin;      /* 1024 */
    int _pad;
} lsdb_lsd_params;

/* structLinesInfo, field for field (LSD/baseFunc.h:33-44); sizeof == 80 like the reference's */
typedef struct {
    double k, b, dx, dy, x1, y1, x2, y2, len;
    int orient;
    int _pad;
} lsdb_line;

/* the fitted rectangle of an accepted region, after the 1/sca rescale (structRec, LSD/myLSD.h:78-92) */
typedef struct {
    double x1, y1, x2, y2, wid, cX, cY, deg, dx, dy, p, prec, logNFA;
} lsdb_rect;

enum { LSDB_STAGE_STENCIL = 0, LSDB_STAGE_ORDER = 1, LSDB_STAGE_GROW = 2, LSDB_NSTAGES = 3 };

typedef struct {
    long long cells, live_seeds, grows, grown_px, small, regrows, rrr_passes, nfa_calls, nfa_px,
        rejects, accepts, spec_evals, respec_evals, chunks;
    /* SM cycles summed over the warps of the region pipeline (lane-0 clock64 deltas): time inside
     * RegionGrower / RectangleConverter / RectangleNFACalculator, waiting for the commit frontier,
     * in the retire phase, in the speculative phase, and in frontier re-evaluations */
    long long cyc_grow, cyc_rect, cyc_nfa, cyc_wait, cyc_retire, cyc_spec, cyc_respec;
    /* per map, summed: SM cycles and wall nanoseconds (globaltimer) a CTA spent on the map; and one spare */
    long long cyc_map, ns_map, spare_;
    /* frontier re-evaluations by cause: never evaluated / parked result invalidated; how many of them committed a region;
     * parked accept/reject results that were invalidated */
    long long rs_none, rs_conflict, rs_commit, rs_lost_commit, rs_pad[4];
} lsdb_stats;

/* ---- context ---- */
/* `stream` is a cudaStream_t (e.g. torch.cuda.current_stream().cuda_stream) or NULL for a private stream. */
int lsdb_create(lsdb_ctx** out, int device, void* stream);
/* Warps per map of the region stage (the seed loop, LSD/myLSD.cpp:218-272) for batches created from now on; 0 = chosen from the batch
 * size as if the batch were alone on the device (16 warps for a lone map ... 4 for 256 maps ... 1 for thousands of rasters).  A caller
 * that keeps SEVERAL small batches in flight on one device (contexts on different streams) fills it better with 4.  Results do not
 * depend on it.  Has no counterpart in the reference (its seed loop is one thread). */
int lsdb_set_team_warps(lsdb_ctx* ctx, int warps);
void lsdb_destroy(lsdb_ctx* ctx);
const char* lsdb_last_error(const lsdb_ctx* ctx);
const char* lsdb_version(void);

/* ---- LSD: batched, device-resident (the path bench.py times) ---- */
/* Allocates every device buffer for n_maps maps of the given sizes once; reusable across runs. */
int lsdb_batch_create(lsdb_ctx* ctx, int n_maps, const int* cols, const int* rows,
                      const lsdb_lsd_params* params, int max_lines_per_map, lsdb_batch** out);
void lsdb_batch_destroy(lsdb_batch* b);
/* host -> device copy of the occupancy grids (maps[i] = rows[i]*cols[i] u8, row-major), async */
int lsdb_batch_upload(lsdb_batch* b, const uint8_t* const* maps);
/* enqueue remap+Gaussian+gradient, pseudo-ordering and the region/rectangle/NFA pipeline */
int lsdb_batch_run(lsdb_batch* b);
/* wait for the stream and check device-side error flags */
int lsdb_batch_sync(lsdb_batch* b);
/* device -> host: counts[n_maps]; lines[n_maps][max_lines_per_map] and rects (same shape) may be NULL.
 * Implies lsdb_batch_sync.  Lines are produced by the epilogue of LSD/myLSD.cpp:282-368. */
int lsdb_batch_download(lsdb_batch* b, int* counts, lsdb_line* lines, lsdb_rect* rects);
/* rasterise map i's segments the way LSD/myLSD.cpp:296-355 fills lineIm (rows*cols u8, 0/255) */
int lsdb_batch_line_image(lsdb_batch* b, int i, uint8_t* line_im);
/* the same for every map of the batch at once, rasterised on the device: line_ims[i] = rows[i]*cols[i] u8 or NULL to skip map i */
int lsdb_batch_line_images(lsdb_batch* b, uint8_t* const* line_ims);
/* intermediate planes of map i for parity tests; every pointer may be NULL.
 *   mag/deg : H'*W' f64 (magMap/degMap, LSD/myLSD.cpp:146-147); used : H'*W' u8 (usedMap, :145);
 *   labels : H'*W' int32 (accept index + 1; reference regIdx == labels & 0xFF, :214,261);
 *   seeds : sorted seed list as linear pixel indices y*W'+x (binCell after qsort, :204) */
int lsdb_batch_planes(lsdb_batch* b, int i, double* mag, double* deg, uint8_t* used, int32_t* labels,
                      int32_t* seeds, int max_seeds, int* n_seeds, double* max_grad);
/* per-stage device time of the last lsdb_batch_run, CUDA events on the context stream */
int lsdb_batch_stage_ms(lsdb_batch* b, float* ms /* [LSDB_NSTAGES] */);
int lsdb_batch_stats(lsdb_batch* b, lsdb_stats* total);
/* the same counters for map i alone */
int lsdb_batch_map_stats(lsdb_batch* b, int i, lsdb_stats* out);
/* number of kernel launches issued by the last lsdb_batch_run */
int lsdb_batch_launches(const lsdb_batch* b);

/* ---- LSD: one map tiled over several GPUs (the stages apart) ---- */
/* For a single-map batch.  Every GPU uploads the whole source map and runs the stencil stage (LSD/myLSD.cpp:135-174,378-484) on
 * the tile rows [tile_row0, tile_row1) only (a tile row = 32 scaled rows); the Gaussian's halo rows (floor(y/0.3+0.5) +- 8,
 * :460,469) are read from the GPU's own copy of the source.  The caller then exchanges the row bands of the planes listed by
 * lsdb_batch_band_planes (NCCL over NVLink: linesegmentdetector-slam_b200/giant.py), takes the max of lsdb_batch_max_grad over
 * the GPUs — the bins need the GLOBAL maxGrad (:179) — and runs lsdb_batch_run_regions (pseudo-ordering + the sequential seed
 * loop, :176-272) on the assembled planes; lsdb_batch_download as usual. */
int lsdb_batch_run_stencil_rows(lsdb_batch* b, int tile_row0, int tile_row1);
int lsdb_batch_max_grad(lsdb_batch* b, int set, double* value);   /* set = 0: read, 1: write */
int lsdb_batch_band_planes(lsdb_batch* b, int max_planes, void** dev_ptrs, long long* row_bytes, int* n_planes, int* tile_rows,
                           int* rows_per_tile);
int lsdb_batch_run_regions(lsdb_batch* b);

/* ---- LSD: one map, host buffers in / host buffers out (what the myLSD.h wrapper calls) ---- */
/* map is NOT modified; map_remapped (nullable) receives the in-place remap the reference applies to
 * its caller's Mat (LSD/myLSD.cpp:135-142); line_im (nullable) = rows*cols u8. */
int lsdb_lsd(lsdb_ctx* ctx, const uint8_t* map, int cols, int rows, const lsdb_lsd_params* params,
             lsdb_line* lines, int max_lines, int* n_lines, uint8_t* line_im, uint8_t* map_remapped);

/* ---- mapCache (the lookup table of the association scoring) ---- */
/* createMapCache (LSD/myLSD.cpp:11-127): truncated brush-fire distance map of the occupied cells (value 1) of `map`
 * (rows*cols u8, BEFORE the LSD remap), in metres, f64, rows*cols.  max_dist = z_occ_max_dis (LSD/baseFunc.h:60, 1 m).
 * Identical to the reference cell for cell, including its FIFO tie-breaking between sources. */
int lsdb_map_cache(lsdb_ctx* ctx, const uint8_t* map, int cols, int rows, double res, double max_dist, double* out);
/* The same with the value of the cells the brush fire never reaches given apart.  The catkin snapshot's three-argument
 * createMapCache (ROS/lsd/include/myLSD.h:131, ROS/lsd/src/myLSD.cpp:11-127) stores the literal 2 there (:37) where the current
 * source stores z_occ_max_dis (LSD/myLSD.cpp:37).  Its down / right neighbour tests (`cur_i >= 1`, ROS/lsd/src/myLSD.cpp:86,105)
 * read one row / column past the map — undefined behaviour; the bounds of the current source (LSD/myLSD.cpp:86,105) are the
 * defined behaviour and the one implemented. */
int lsdb_map_cache_fill(lsdb_ctx* ctx, const uint8_t* map, int cols, int rows, double res, double max_dist, double unreached,
                        double* out);
/* createMapCache (LSD/myLSD.cpp:11-127; the snapshot's 3-argument flavour via `unreached`) for every map of the batch, on the device,
 * from the source planes lsdb_batch_upload / lsdb_batch_upload_scan_rasters left (value 1 = occupied).  res[n_maps] (> 0, finite);
 * max_dist >= 0; unreached = value of cells the fire never reaches (max_dist for the current source, 2 for the snapshot).
 * out: NULL (keep on the device only) or n_maps host pointers (rows*cols f64 each; NULL entries skipped).  Independent of
 * lsdb_batch_run: before or after it, the result is the same.  Cell for cell what lsdb_map_cache_fill returns for each map alone.
 * The caches stay in a plane the batch owns (8 bytes per source pixel, allocated on the first call, overwritten by the next).
 * LSDB_ERR_ARG: res NULL, a res not finite and > 0, max_dist < 0 or NaN, a map with more than 65535 columns or rows. */
int lsdb_batch_map_caches(lsdb_batch* b, const double* res, double max_dist, double unreached, double* const* out);
/* An association map from map i of the batch: its cache (lsdb_batch_map_caches must have run) copied device to device, and its
 * segment table exactly as lsdb_batch_download returns it (the batch must have run).  The lsdb_fa_map owns its copies.
 * LSDB_ERR_ARG: out NULL, i out of range, before lsdb_batch_run or before lsdb_batch_map_caches. */
int lsdb_fa_map_create_from_batch(lsdb_batch* b, int i, lsdb_fa_map** out);

/* ---- one process, several GPUs ---- */
/* A batch of independent maps split contiguously over the listed devices (the first n % k devices get one map more), one host
 * thread and one private stream per device, no collective; tables come back in batch order exactly as from one device
 * (SURVEY.md 8b `lsdb_create(ctx, device_ids[])`, 8e).  The same device may be listed more than once. */
typedef struct lsdb_multi lsdb_multi;
int lsdb_multi_create(lsdb_multi** out, const int* device_ids, int n_devices);
void lsdb_multi_destroy(lsdb_multi* m);
int lsdb_multi_devices(const lsdb_multi* m);
const char* lsdb_multi_last_error(const lsdb_multi* m);
void lsdb_multi_shard(int n_items, int d, int n_devices, int* first, int* count);
/* counts[n_maps]; lines / rects: [n_maps][max_lines] (nullable) */
int lsdb_multi_lsd(lsdb_multi* m, int n_maps, const uint8_t* const* maps, const int* cols, const int* rows,
                   const lsdb_lsd_params* params, int max_lines, int* counts, lsdb_line* lines, lsdb_rect* rects);

/* ---- the reference's text files (host only, no device) ---- */
/* mapParam.txt: `cols rows resol oriX oriY` (LSD/main_on_windows.cpp:28-34) */
int lsdb_read_map_param(const char* path, int* cols, int* rows, double* resol, double* ori_x, double* ori_y);
/* mapValue*.txt: rows*cols integers; a pixel = value & 0xFF, as the reference's `%d` into a uint8 slot leaves it (:38-46) */
int lsdb_read_map_value(const char* path, int cols, int rows, uint8_t* out);
/* mapCache.txt: rows*cols doubles, whitespace separated, row-major (LSD/test.cpp:11-17); the writer prints %.17g, which the
 * reference's `%lf` reader turns back into the same doubles */
int lsdb_read_map_cache(const char* path, int cols, int rows, double* out);
int lsdb_write_map_cache(const char* path, int cols, int rows, const double* in);

/* ---- association scoring ---- */
/* structScore (LSD/myFA.h:49-54) plus the indices that identify the hypothesis */
typedef struct {
    int frame, i_scan, i_map, i_pair; /* i_pair = 1..4, the endpoint pairing of LSD/myFA.cpp:194-235 */
    double x, y, ang, score;          /* score = +inf when gated out / < 70 % of points in the map */
} lsdb_hypothesis;

/* uploads mapCache (rows*cols f64 metres, output of createMapCache) and the map's LSD lines once */
int lsdb_fa_map_create(lsdb_ctx* ctx, const double* map_cache, int cols, int rows,
                       const lsdb_line* map_lines, int n_map_lines, lsdb_fa_map** out);
void lsdb_fa_map_destroy(lsdb_fa_map* m);
/* Scores every (scan line, map line, pairing) triple that passes the reference's length filter
 * (LSD/myFA.cpp:29-41) for n_frames scan frames in one launch.
 *   scan_lines : concatenated per frame, scan_line_off[n_frames+1] offsets
 *   scan_pts   : concatenated (x,y) pairs (FS.scanImPoint), scan_pt_off[n_frames+1] offsets (in points)
 *   lidar_pose : [n_frames][2]   (already rounded as LSD/main_on_windows.cpp:229-230 does)
 *   last_pose  : [n_frames][3]   (x == -1 disables the 60 px gate, LSD/myFA.cpp:330)
 * Output: up to max_hyp records in (frame, i_scan, i_map, i_pair) order; *n_hyp = number produced. */
int lsdb_fa_score(lsdb_ctx* ctx, const lsdb_fa_map* m, int n_frames, const lsdb_line* scan_lines,
                  const int* scan_line_off, const double* scan_pts, const int* scan_pt_off,
                  const double* lidar_pose, const double* last_pose, lsdb_hypothesis* out, int max_hyp,
                  int* n_hyp);
/* The hypotheses the reference keeps (score < keep_below; LSD/myFA.cpp:261-265 keeps < 3), in (frame, scan line, map line,
 * pairing) order, for any number of frames.  Lines and raster samples go from the caller's buffers straight to the device,
 * the pair filter runs there, only the kept hypotheses come back.  *n_kept = how many there are (LSDB_ERR_CAPACITY if more
 * than max_kept), *n_hyp (nullable) = how many were scored. */
int lsdb_fa_score_kept(lsdb_ctx* ctx, const lsdb_fa_map* m, int n_frames, const lsdb_line* scan_lines, const int* scan_line_off,
                       const double* scan_pts, const int* scan_pt_off, const double* lidar_pose, const double* last_pose,
                       double keep_below, lsdb_hypothesis* out, int max_kept, int* n_kept, int* n_hyp);
/* The catkin snapshot's association, SURVEY.md §8 f4 — replaces myfa::FeatureAssociation of ROS/lsd/include/FeatureAssociation.h:46-60
 * (ROS/lsd/src/FeatureAssociation.cpp:36-130; ScanToMapMatch :132-200, ScanToMapMatchScore :202-252, RotateScanIm :254-299), the
 * 13-argument call of LSD/main_on_linux.cpp:132.  `m` holds MapCache (the three-argument createMapCache: cells beyond z_occ_max_dis
 * read exactly 2.0, which the score counts apart, :239) and MaplinesInfo; its size is the size of MaplineIm.
 *   scan_lines : ScanlinesInfo (x1 y1 x2 y2 len are used)      lidar_pos : LidarPos[2], scan-image pixels
 *   ranges/angles : ScanRanges / ScanAngles, n_rays of each (Inf / NaN ranges fall outside the map, as in the reference);
 *                   an angle with |angle| > LSDB_MAX_ANGLE (2^19, Inf included) is LSDB_ERR_ARG, found before anything launches
 * Output: pose_all = up to max_cols records of 15 doubles, the COLUMNS of the reference's 15 x T poseAll in its order (pose x y
 * angle[deg], score, map end points, scan end points, scan-line index, map-line index, pairing 0..3); *n_cols = T;
 * estimate_pose[3] (pixels, radians) / estimate_pose_realworld[3] (metres) = the first strict minimum of the score row (:117-127),
 * both nullable.  Scores carry the bits of the reference's sequential sum.  T == 0 (the reference then reads an empty matrix):
 * LSDB_OK, nothing estimated.  T > max_cols > 0: the first max_cols records, the estimates, and LSDB_ERR_CAPACITY. */
int lsdb_fa_legacy(lsdb_ctx* ctx, const lsdb_fa_map* m, const lsdb_line* scan_lines, int n_scan, double map_resol, double map_ori_x,
                   double map_ori_y, const int* lidar_pos, const double* ranges, const double* angles, int n_rays, double* pose_all,
                   int max_cols, int* n_cols, double* estimate_pose, double* estimate_pose_realworld);
/* one record per frame of lsdb_fa_legacy_frames */
typedef struct {
    int n_cols;                        /* T of the frame = 4 x candidate pairs */
    int best_col;                      /* t of :117-119, frame-local column; -1 when T == 0 */
    double best_score;                 /* poseAll(3, t); NaN when T == 0 */
    double estimate_pose[3];           /* pixels, radians (:120-123); NaN when T == 0 */
    double estimate_pose_realworld[3]; /* metres (:124-127); NaN when T == 0 */
} lsdb_fa_legacy_estimate;             /* 64 bytes */
/* lsdb_fa_legacy for n_frames sweeps against one map in one call (a log replayed, a parameter sweep).  Frames are independent in
 * the snapshot (no pose of one frame gates the next), so every frame gets exactly what lsdb_fa_legacy returns for it alone, however
 * the frames are grouped into calls:
 *   scan_lines : ScanlinesInfo of every frame concatenated, scan_line_off[n_frames+1]; lidar_pos : [n_frames][2]
 *   ranges / angles : concatenated, ray_off[n_frames+1] (Inf / NaN ranges fall outside the map; |angle| <= LSDB_MAX_ANGLE)
 * Per frame: the length filter of :61-70 with 0.3 / map_resol in the reference's (scan line, map line) order, the four pairings,
 * RotateScanIm and the ray re-projection score.  Frame f's records are the columns [col_off[f], col_off[f+1]) of pose_all (15
 * doubles each, as lsdb_fa_legacy); column 12 is the frame-local scan-line index, so a frame's slice equals its lsdb_fa_legacy output.
 * est[f].best_col is the column the reference's `t = 0; for i: if (s[i] < s[t]) t = i` ends at, i.e.: 0 if s[0] is NaN, otherwise
 * the FIRST column whose score == the minimum of the non-NaN scores (-0 ties +0; a frame of +inf scores gives 0).  A frame without
 * rays scores NaN (0/0) everywhere and gets best_col = 0; a frame without a candidate pair gets best_col = -1 and NaNs.
 * Sizes: est and col_off (nullable) are always filled first.  pose_all == NULL asks for the estimates only.  pose_all != NULL and a
 * total T > max_cols: LSDB_ERR_CAPACITY with est and col_off filled and pose_all untouched (the sizing query).  A total T above
 * 2^31-1 is LSDB_ERR_CAPACITY.  n_frames == 0 is LSDB_OK.  LSDB_ERR_ARG: offsets that do not start at 0 or decrease, null arrays
 * with non-zero counts, est or lidar_pos NULL (n_frames > 0), max_cols < 0, map_resol <= 0, an angle beyond LSDB_MAX_ANGLE.
 * One host-to-device copy, two launches (scores, per-frame selection), one synchronise. */
int lsdb_fa_legacy_frames(lsdb_ctx* ctx, const lsdb_fa_map* m, int n_frames,
                          const lsdb_line* scan_lines, const int* scan_line_off,
                          double map_resol, double map_ori_x, double map_ori_y,
                          const int* lidar_pos,
                          const double* ranges, const double* angles, const int* ray_off,
                          lsdb_fa_legacy_estimate* est,
                          double* pose_all, int max_cols, int* col_off);
/* The per-frame reduction that follows the scoring in FeatureAssociation (LSD/myFA.cpp:65-171, everything before ukf),
 * done on the device so that only one record per frame comes back instead of every hypothesis:
 *   n_kept  : hypotheses with score < 3 (:261); 0 = "no match, start a new chain" (:70-90)
 *   best_*  : the lowest-score hypothesis — the pose of the first frame of a chain (:100-110)
 *   mean_*  : the 1/score^2 weighted mean over the kept hypotheses in ascending score order (:160-171) and
 *             mean_score = 1/sqrt(sum(w)/n_kept): the poseEstimate handed to ukf */
typedef struct {
    int n_hyp, n_kept;
    double best_x, best_y, best_ang, best_score;
    double mean_x, mean_y, mean_ang, mean_score;
} lsdb_fa_estimate;
/* same inputs as lsdb_fa_score; out[n_frames] */
int lsdb_fa_estimate_frames(lsdb_ctx* ctx, const lsdb_fa_map* m, int n_frames, const lsdb_line* scan_lines,
                            const int* scan_line_off, const double* scan_pts, const int* scan_pt_off,
                            const double* lidar_pose, const double* last_pose, lsdb_fa_estimate* out);
/* device time of the kernels of the last association call on this context (ms): lsdb_fa_score, lsdb_fa_score_kept,
 * lsdb_fa_estimate_frames, lsdb_scan_estimate_frames (its association part), lsdb_fa_legacy, lsdb_fa_legacy_frames */
float lsdb_fa_last_ms(const lsdb_ctx* ctx);

/* ---- scan front-end: lidar frames -> scan lines + raster samples (the inputs of the association) ---- */
/* myrdp::FeatureScan (LSD/myRDP.h:63, LSD/myRDP.cpp:9-185: RegionSegmentation, Ramer-Douglas-Peucker split, line records,
 * rasterisation) for n_frames frames in one call; scanPose = (0,0,0) as in the reference.  Defaults of the three
 * parameters: rdp_leastPoint = 3, rdp_threLine = 0.08, rdp_leastDist = 0.5 (LSD/baseFunc.h:70-72). */
typedef struct {
    int least_point;      /* RegionPointLimitNumber: minimum index span of a cluster */
    double thre_line;     /* split threshold (m; scaled by the range beyond 9 m); must be > 0 */
    double least_dist_m;  /* shortest line piece kept (m) */
} lsdb_rdp_params;
typedef struct {
    int n_lines, n_pts;        /* FS.len_linesInfo, FS.scanImPoint.size() */
    int im_cols, im_rows;      /* size of FS.lineIm */
    double lidar_x, lidar_y;   /* FS.lidarPos */
} lsdb_scan_info;
/* Inputs: ranges / angles concatenated per frame (finite values only — the callers drop Inf beams,
 * LSD/main_on_windows.cpp:110-123 — and |angle| <= LSDB_MAX_ANGLE, 2^19; anything else is LSDB_ERR_ARG before any launch),
 * beam_off[n_frames+1]; every frame needs at least one beam.
 * Outputs (host buffers):
 *   info[n_frames]; line_off / pt_off [n_frames+1] (prefix sums of n_lines / n_pts); im_off[n_frames+1] (bytes)
 *   lines  : records in the reference's order, frame f at lines[line_off[f]]  (lsdb_line; `orient` as FeatureScan sets it)
 *   pts    : (x,y) pairs = FS.scanImPoint, frame f at pts[2*pt_off[f]] — exactly what lsdb_fa_score takes
 *   line_im: optional (NULL = skip): the 0/255 rasters FS.lineIm, frame f = im_rows*im_cols bytes at line_im[im_off[f]]
 * lines == NULL and pts == NULL is a sizing query: only info and the three offset arrays are produced.
 * LSDB_ERR_CAPACITY (max_lines, max_pts or line_im_cap too small) still leaves info and the offsets filled. */
int lsdb_feature_scan_frames(lsdb_ctx* ctx, double map_resol, double map_ori_x, double map_ori_y,
                             const lsdb_rdp_params* prm, int n_frames, const double* ranges, const double* angles,
                             const int* beam_off, lsdb_scan_info* info, lsdb_line* lines, int max_lines, int* line_off,
                             double* pts, int max_pts, int* pt_off, uint8_t* line_im, long long line_im_cap,
                             long long* im_off);
/* LSD on rasterised scans (the reference rasterises a sweep into FS.lineIm and can run myLineSegmentDetector on it): writes
 * the FeatureScan rasters of n_frames sweeps straight into the source planes of `batch` as occupancy grids (occupied = 1, the
 * mapValue convention) — frame f becomes map f; the rasters never exist on the host.  `batch` must have been created with
 * n_frames maps of the sizes (im_cols, im_rows) a sizing query of lsdb_feature_scan_frames reports for the same sweeps;
 * LSDB_ERR_ARG otherwise.  Replaces lsdb_batch_upload for that batch; lsdb_batch_run follows. */
int lsdb_batch_upload_scan_rasters(lsdb_batch* batch, double map_resol, double map_ori_x, double map_ori_y,
                                   const lsdb_rdp_params* prm, int n_frames, const double* ranges, const double* angles,
                                   const int* beam_off, lsdb_scan_info* info);
/* The whole scan side of one localisation step for n_frames sweeps: FeatureScan, then the scoring and reduction of
 * lsdb_fa_estimate_frames against map `m`, with lidar_pose = (int)round(FS.lidarPos) as LSD/main_on_windows.cpp:229-230
 * builds it.  Same results as lsdb_feature_scan_frames followed by lsdb_fa_estimate_frames, but scan lines and raster samples
 * never leave the device (the length filter of LSD/myFA.cpp:29-41 runs there as well).
 *   last_pose [n_frames][3], info [n_frames] out, est [n_frames] out. */
int lsdb_scan_estimate_frames(lsdb_ctx* ctx, const lsdb_fa_map* m, double map_resol, double map_ori_x, double map_ori_y,
                              const lsdb_rdp_params* prm, int n_frames, const double* ranges, const double* angles,
                              const int* beam_off, const double* last_pose, lsdb_scan_info* info, lsdb_fa_estimate* est);
/* device time of the two kernels of the last lsdb_feature_scan_frames call (ms) */
float lsdb_feature_scan_last_ms(const lsdb_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif
