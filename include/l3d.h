/*
 * l3d.h -- C ABI of libl3d.so, the B200 (sm_100a) implementation of the per-frame dense vision
 * hot path of alo-i-sia/laser_3d_reconstruction.
 *
 * The reference has no FFI seam of its own: its hot path is Python calling cv2 / numpy.  Each
 * entry point below replaces one of those call sites (cited as reference file:line); the Python
 * classes in laser_3d_reconstruction_b200/ bind them with ctypes (see INTEGRATION.md).
 *
 * Conventions: plain C, `int` status (0 = OK, <0 = error, text via l3d_last_error); one context
 * per (thread, GPU); a context owns one CUDA stream and grow-only device scratch; all pointers
 * are HOST pointers unless the name says `_dev`; host buffers are only touched during the call;
 * images are row-major, tightly packed unless a stride is given.  No CPU fallback exists.
 */
#ifndef L3D_H
#define L3D_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct l3d_ctx l3d_ctx;

enum { L3D_OK = 0, L3D_ERR_ARG = -1, L3D_ERR_CUDA = -2, L3D_ERR_UNSUPPORTED = -3, L3D_ERR_STATE = -4 };
enum { L3D_MODE_SGBM = 0, L3D_MODE_HH = 1, L3D_MODE_SGBM_3WAY = 2, L3D_MODE_HH4 = 3 }; /* cv2.STEREO_SGBM_MODE_* */

/* -------- context (plumbing: the reference has no counterpart; it is what `import cv2` gives the Python process) -------- */
int l3d_ctx_create(int device, l3d_ctx** out);
void l3d_ctx_destroy(l3d_ctx* ctx);
const char* l3d_last_error(l3d_ctx* ctx); /* ctx may be NULL: last create error */
int l3d_sync(l3d_ctx* ctx);
int l3d_device_count(void);
const char* l3d_version(void);
/* number of kernels this context has launched since creation (bench.py "gpu_launches") */
long long l3d_launch_count(l3d_ctx* ctx);

/* -------- K1: rectification remap + gray -------------------------------------------------- */
/* Replaces cv2.initUndistortRectifyMap's CV_32FC1 maps as consumed by cv2.remap
 * (camera/single_usb_stereo_camera.py:190-206,313-314): converts to the 5-bit fixed-point form once. */
int l3d_set_rectify_maps(l3d_ctx* ctx, int eye, const float* mapx, const float* mapy, int W, int H);
/* cv2.remap(img, mapx, mapy, INTER_LINEAR) + cv2.cvtColor(BGR2GRAY)
 * (camera/single_usb_stereo_camera.py:313-314,320-321).  src is sw x sh BGR with row stride
 * src_stride bytes; rect_bgr (W*H*3) and gray (W*H) may each be NULL. */
int l3d_remap_gray(l3d_ctx* ctx, int eye, const uint8_t* src_bgr, int sw, int sh, long src_stride,
                   uint8_t* rect_bgr, uint8_t* gray);
/* cv2.cvtColor(BGR2GRAY) alone (core/laser_extractor.py:60,174) */
int l3d_bgr2gray(l3d_ctx* ctx, const uint8_t* bgr, int W, int H, uint8_t* gray);

/* -------- point-cloud sink (SURVEY 8f N2) ------------------------------------------------------
 * PointCloudProcessor.voxel_downsample / .statistical_outlier_removal of utils/point_cloud.py in the form that file
 * runs without Open3D (:54-78, :108-131).  points = n x 3 f64 (host); out has room for n x 3; *n_out = rows written.
 * voxel_downsample: one point per occupied voxel (floor(p / voxel_size)), the f64 mean of its points, voxels in order
 * of first appearance; voxel indices must lie inside +-2^20.  f32_arithmetic != 0: the points are float32 values (passed
 * as doubles) and division, floor, running sum and mean are float32 operations, as numpy does for the float32 cloud
 * main.py:208 builds.  statistical_outlier_removal: the reference's predicate
 * as written (mean of the nb_neighbors nearest distances < mean + std_ratio * std), exact brute-force neighbours
 * (O(n^2): meant for down-sampled clouds); nb_neighbors <= 63. */
int l3d_voxel_downsample(l3d_ctx* ctx, const double* points, int n, double voxel_size, int f32_arithmetic, double* out,
                         int* n_out);
int l3d_statistical_outlier_removal(l3d_ctx* ctx, const double* points, int n, int nb_neighbors, double std_ratio,
                                    double* out, int* n_out);

/* -------- laser-plane fit (no reference counterpart: the reference takes the plane as a constant, config.py) --------
 * RANSAC + least-squares refinement of a plane a x + b y + c z + d = 0 through n points (xyz: n x 3 f64, host).
 * Hypothesis h in [0, hypotheses) takes the points i_k = splitmix64(seed + (3h + k + 1) * 0x9E3779B97F4A7C15) mod n,
 * k = 0..2; its plane is n = (p1 - p0) x (p2 - p0), n / |n|, d = -n.p0, and a point is its inlier iff
 * |((n.x p.x + n.y p.y) + n.z p.z) + d| <= threshold, every operation f64 round-to-nearest without FMA contraction
 * (DESIGN.md section 4f has the exact contract).  A hypothesis with a non-finite point or |n| not in (0, inf) is
 * invalid.  The winner has the most inliers (ties: lowest h).  Refinement, at most 10 times: centroid and covariance
 * (divided by the count) of the inlier set S, normal = eigenvector of the smallest eigenvalue, d = -n.c, reselect S';
 * stop when S' == S.  Output: the last fit with d >= 0, its S' (inliers, inlier_mask: n bytes 0/1, may be NULL), the
 * rms residual over S'.  L3D_ERR_ARG: n < 3, threshold not finite or <= 0, hypotheses outside [1, 2^20], no valid
 * hypothesis, a fit left with fewer than 3 inliers.  Deterministic: the same input gives the same bits. */
typedef struct { double threshold; int hypotheses; unsigned long long seed; } l3d_plane_fit_params;
typedef struct {
    double plane[4];        /* unit normal, d >= 0 */
    int inliers;            /* points within threshold of `plane` */
    double rms;             /* sqrt(mean residual^2) over those inliers */
    double eig[3];          /* ascending eigenvalues of the last least-squares fit's inlier covariance */
    int hypothesis;         /* index of the winning RANSAC hypothesis */
    int hypothesis_inliers; /* its inlier count */
    int refits;             /* least-squares fits done */
} l3d_plane_fit_result;
int l3d_fit_plane(l3d_ctx* ctx, const double* xyz, int n, const l3d_plane_fit_params* p, l3d_plane_fit_result* out,
                  uint8_t* inlier_mask);

/* -------- init-time rectification maps (SURVEY 8f N3) ------------------------------------------
 * cv2.initUndistortRectifyMap(K, dist, R, P, (W, H), CV_32FC1) -> mapx, mapy (f32 HxW), as called once per eye in
 * camera/single_usb_stereo_camera.py:190-206.  K = 3x3 row-major; dist = ndist <= 14 coefficients
 * (k1 k2 p1 p2 k3 k4 k5 k6 s1 s2 s3 s4 [tau_x tau_y = 0]); iR = inverse of P[:3,:3] * R (3x3 row-major, computed by the
 * caller in f64).  Bit-exact against cv2 4.13. */
int l3d_init_undistort_rectify_map(l3d_ctx* ctx, const double* K, const double* dist, int ndist, const double* iR,
                                   int W, int H, float* mapx, float* mapy);

/* -------- StereoBM (SURVEY 8f N4) ------------------------------------------------------------
 * cv2.StereoBM_create(numDisparities, blockSize).compute(left, right) -> int16 disparity x16, the matcher
 * readme.md:392-397 offers as a drop-in for StereoSGBM.  PREFILTER_XSOBEL; minDisparity <= 0 only
 * (L3D_ERR_UNSUPPORTED otherwise: OpenCV itself writes past the row end for positive values); disp12MaxDiff >= 0 with
 * preFilterCap <= 31 and blockSize <= 21 only; bit-exact against cv2 4.13. */
typedef struct {
    int minDisparity, numDisparities, blockSize, preFilterCap, textureThreshold, uniquenessRatio,
        speckleWindowSize, speckleRange, disp12MaxDiff;
} l3d_bm_params;
int l3d_bm_compute(l3d_ctx* ctx, const l3d_bm_params* p, const uint8_t* left, const uint8_t* right,
                   int W, int H, int16_t* disp);

/* -------- K2: StereoSGBM ------------------------------------------------------------------ */
typedef struct {
    int minDisparity, numDisparities, blockSize, P1, P2, disp12MaxDiff, preFilterCap,
        uniquenessRatio, speckleWindowSize, speckleRange, mode;
} l3d_sgbm_params; /* cv2.StereoSGBM_create arguments, camera/single_usb_stereo_camera.py:252-274;
                    * numDisparities: a multiple of 16 in [16, 512] in every mode; blockSize: odd in [1, 21], and at most 15
                    * when numDisparities > 272 (L3D_ERR_UNSUPPORTED otherwise) */

/* cv2.StereoSGBM.compute(left, right) -> int16 disparity x16
 * (camera/single_usb_stereo_camera.py:324-325, test_improved_laser.py:151, test_depth.py:68) */
int l3d_sgbm_compute(l3d_ctx* ctx, const l3d_sgbm_params* p, const uint8_t* left,
                     const uint8_t* right, int W, int H, int16_t* disp);
/* Same, plus intermediates for parity tests (each may be NULL): raw = before median/speckle,
 * C/S = HV*width1*D int16 volumes (HV = H for modes 0/1). */
int l3d_sgbm_debug(l3d_ctx* ctx, const l3d_sgbm_params* p, const uint8_t* left,
                   const uint8_t* right, int W, int H, int16_t* disp, int16_t* raw,
                   int16_t* C_out, int16_t* S_out);
/* The matcher pair of the reference's get_frames(): stereo_matcher.compute(left, right) and
 * right_matcher.compute(right, left) (camera/single_usb_stereo_camera.py:324-325) in one call.  BT operands are
 * built once per view and -- for the geometries the shared pass covers (right->minDisparity = -(D-1), equal
 * blockSize / P2, D 64 with block 5 or D 128 with block 9) -- both cost volumes come from ONE pixel-cost pass.
 * Cl_out / Cr_out (may be NULL): the two HV*width1*D int16 cost volumes, for parity tests. */
int l3d_sgbm_compute_pair(l3d_ctx* ctx, const l3d_sgbm_params* left_params, const l3d_sgbm_params* right_params,
                          const uint8_t* left, const uint8_t* right, int W, int H, int16_t* disp_left,
                          int16_t* disp_right, int16_t* Cl_out, int16_t* Cr_out);
/* rows of the C/S volumes l3d_sgbm_debug writes (H, or the sum of 3WAY stripe heights) */
int l3d_sgbm_volume_rows(const l3d_sgbm_params* p, int W, int H);
/* cv2.medianBlur(disp, 3) and cv2.filterSpeckles as applied inside StereoSGBM.compute
 * (camera/single_usb_stereo_camera.py:324-325 with speckleWindowSize / speckleRange of :266-267) */
int l3d_median3_s16(l3d_ctx* ctx, const int16_t* src, int W, int H, int16_t* dst);
int l3d_filter_speckles(l3d_ctx* ctx, int16_t* img, int W, int H, int newVal, int maxSize, int maxDiff);

/* -------- K3: WLS disparity filter -------------------------------------------------------- */
typedef struct {
    double lambda, sigma_color; /* wls_filter.setLambda / setSigmaColor, camera/...:281-282 */
    int min_disp, num_disp;     /* of the left matcher */
    int dd_radius;              /* depth-discontinuity radius = ceil(0.5*blockSize) for SGBM */
    int lrc_thresh;             /* 24 */
    int solver;                 /* 0: partitioned parallel tridiagonal solves (default); 1: serial Thomas solves in the
                                 * oracle's f32 operation order (bit-identical to oracle/csrc/orc_wls.c) */
    int variant;                /* L3D_WLS_* bits: readings of opencv_contrib the oracle cannot pin (cv2.ximgproc is not
                                 * installed anywhere this was built); 0 = the documented defaults, see DESIGN.md */
} l3d_wls_params;
enum {
    L3D_WLS_LAMBDA_PER_PASS = 1,   /* lambda is attenuated after every pass (x, y) instead of after each iteration */
    L3D_WLS_LRC_OUTSIDE_ZERO = 2,  /* a pixel whose matching column falls outside the right ROI gets confidence 0
                                    * (default: it keeps its own depth-discontinuity confidence) */
    L3D_WLS_BOX_FULL_IMAGE = 4,    /* the variance box filters read across the ROI edge into the full disparity image
                                    * (default: they run on a copy of the ROI, REFLECT_101 at the ROI edge) */
    L3D_WLS_CONF_CLAMP_1 = 8       /* 1 - 0.001 var is clamped to [0, 1] (default: only below at 0) */
};
/* wls_filter.filter(dl, guide, disparity_map_right=dr) (camera/single_usb_stereo_camera.py:328-332) */
int l3d_wls_filter(l3d_ctx* ctx, const l3d_wls_params* p, const int16_t* dl, const int16_t* dr,
                   const uint8_t* guide, int W, int H, int16_t* out, float* conf_out);
/* Test seam: the FGS passes of l3d_wls_filter alone. num/den (w x h f32) are solved in place with
 * row weights ch and column weights cv (<= 0, as the LUT makes them). Runs `iters` (1..3)
 * iterations of (row pass, column pass) with the lambda schedule of `variant`. solver: as in
 * l3d_wls_params. *parallel_used = 1 when the partitioned kernels ran, 0 for the serial
 * fallback (gate: solver, shared-memory size, w >= 2 && h >= 2). */
int l3d_fgs_solve(l3d_ctx* ctx, int solver, int variant, double lambda, int iters,
                  const float* ch, const float* cv, int w, int h, float* num, float* den, int* parallel_used);

/* -------- K5a: disparity -> depth --------------------------------------------------------- */
/* camera/single_usb_stereo_camera.py:335-346 (Q != NULL) or :347-357 (Q == NULL) */
int l3d_disp_to_depth(l3d_ctx* ctx, const int16_t* disp16, int W, int H, const double* Q, float* depth);

/* -------- get_frames() depth path, fused --------------------------------------------------- */
typedef struct {
    l3d_sgbm_params left;  /* as (possibly) mutated by createDisparityWLSFilter */
    l3d_sgbm_params right; /* createRightMatcher(left) */
    l3d_wls_params wls;
    int use_wls;           /* 0: depth from the left matcher alone */
    int use_maps;          /* 0: no rectification (map_left_x is None branch, camera/...:315-317) */
    int use_Q;             /* 0: no-calibration depth branch */
    double Q[16];
} l3d_depth_config;
/* camera/single_usb_stereo_camera.py:311-359 without the capture: left/right BGR (W x H, stride
 * bytes) -> rectified left BGR + depth (metres, f32).  disp_out (int16, optional) = filtered disparity. */
int l3d_compute_depth(l3d_ctx* ctx, const l3d_depth_config* cfg, const uint8_t* left_bgr,
                      const uint8_t* right_bgr, int W, int H, long stride, uint8_t* left_rect,
                      float* depth, int16_t* disp_out);

/* -------- K4a: Simple laser extractor ------------------------------------------------------ */
/* SimpleLaserExtractor.extract_centerline (core/laser_extractor.py:45-100).  xy receives n (x,y)
 * pairs (capacity H), rows ascending.  mask_morph (:69) and mask_final (:81-82) may be NULL. */
int l3d_simple_extract(l3d_ctx* ctx, const uint8_t* bgr, int W, int H, const int* hsv_lo,
                       const int* hsv_hi, int bright_thr, double min_area, uint8_t* mask_morph,
                       uint8_t* mask_final, double* xy, int* n);

/* Steps (1)-(3) of the same function alone (core/laser_extractor.py:56-64): mask = inRange(cvtColor(bgr, HSV), lo, hi) &
 * (cvtColor(bgr, GRAY) > bright_thr), 0 / 255 per pixel (bright_thr < 0: the HSV range test alone). */
int l3d_colour_mask(l3d_ctx* ctx, const uint8_t* bgr, int W, int H, const int* hsv_lo, const int* hsv_hi,
                    int bright_thr, uint8_t* mask);

/* -------- K4b: Steger extractors ----------------------------------------------------------- */
enum {
    L3D_STEGER_FAST = 0,      /* FastStegerExtractor.extract_centerline   core/laser_extractor.py:160-261 */
    L3D_STEGER_IMPROVED = 1,  /* ImprovedStegerExtractor.extract_centerline improved_steger.py:39-126    */
    L3D_STEGER_OPTIMIZED = 2, /* .extract_centerline_optimized             improved_steger.py:128-223   */
    L3D_STEGER_HYBRID = 3     /* HybridLaserExtractor.extract_centerline   improved_steger.py:250-344   */
};
typedef struct {
    int variant;
    double sigma;
    int bright_thr;
    double resp_thr;      /* response_threshold (IMPROVED/OPTIMIZED) */
    int roi[4];           /* x,y,w,h for FAST; w<=0: none */
    int hsv_lo[3], hsv_hi[3]; /* HYBRID */
} l3d_steger_params;
/* img: channels = 3 (BGR) or 1 (gray).  xy: capacity cap points (x,y as f32 pairs), raster order.
 * *n = number of points found (may exceed cap: then only cap were written, status L3D_OK). */
int l3d_steger_extract(l3d_ctx* ctx, const l3d_steger_params* p, const uint8_t* img, int channels,
                       int W, int H, float* xy, int cap, int* n);

/* -------- K5b: 2D -> 3D -------------------------------------------------------------------- */
enum {
    L3D_RECON_PLANE = 0,        /* Reconstructor.reconstruct_laser_line  core/reconstruction.py:30-143 */
    L3D_RECON_DEPTH = 1,        /* Reconstructor.reconstruct_from_depth  core/reconstruction.py:145-182 */
    L3D_RECON_DISPARITY = 2,    /* ImprovedLaserReconstructor.reconstruct_from_disparity  improved_reconstruction.py:37-86 */
    L3D_RECON_DISPARITY_MEDIAN = 3 /* .reconstruct_with_interpolation (window odd, <= 9)  improved_reconstruction.py:88-152 */
};
typedef struct {
    int kind;
    double K[9];        /* camera intrinsic (PLANE, DEPTH) */
    double plane[4];    /* laser plane a,b,c,d (PLANE) */
    int use_refraction; /* PLANE */
    double n_water;     /* 1.33 */
    double fx, baseline, cx, cy; /* DISPARITY kinds (from Q) */
    double min_disparity;
    int window;         /* DISPARITY_MEDIAN: odd, 1..9 (the reference defaults to 3) */
} l3d_recon_params;
/* xy: n points (f64 pairs).  img: depth or disparity map (f32, W x H) for the kinds that need it.
 * xyz: up to n rows of 3 f64; *n_out rows written (invalid points dropped, order kept). */
int l3d_reconstruct(l3d_ctx* ctx, const l3d_recon_params* p, const double* xy, int n,
                    const float* img, int W, int H, double* xyz, int* n_out);
/* ImprovedLaserReconstructor.create_laser_depth_map (improved_reconstruction.py:154-186): out (f32, W x H) is zero except at
 * the rounded laser pixels with disparity > 1, where it holds fx * baseline / disparity if that lies in (0, 10) m. */
int l3d_laser_depth_map(l3d_ctx* ctx, const double* xy, int n, const float* disp, int W, int H, double fx,
                        double baseline, float* out);

/* -------- batched, device-resident frame pipeline: LaserReconstructionSystem.process_frame (main.py:164-189 = get_frames,
 * camera/single_usb_stereo_camera.py:294-359, + extract_centerline + reconstruct_from_depth) for many frames per call;
 * what bench.py times.  The launch-count / timing / packing calls below are measurement and sharding plumbing. */
typedef struct l3d_pipeline l3d_pipeline;
typedef struct {
    int W, H;                 /* per-eye size */
    l3d_depth_config depth;
    int extractor;            /* -1 none, 0..3 = L3D_STEGER_*, 4 = Simple */
    l3d_steger_params steger;
    int simple_hsv_lo[3], simple_hsv_hi[3], simple_bright_thr; double simple_min_area;
    l3d_recon_params recon;   /* per-frame 3D: PLANE reads no image, DEPTH the frame's depth plane (main.py:176),
                               * DISPARITY / DISPARITY_MEDIAN its int16 x16 disparity (the disp16 of l3d_pipeline_fetch:
                               * WLS output with depth.use_wls, else the left matcher's) as disp16 / 16.0.  Create fails
                               * with L3D_ERR_ARG for a DISPARITY_MEDIAN window that is not odd in [1, 9]. */
    int max_points;           /* per-frame point capacity */
    int lanes;                /* frames in flight (streams), >= 1 */
} l3d_pipeline_config;
int l3d_pipeline_create(l3d_ctx* ctx, const l3d_pipeline_config* cfg, l3d_pipeline** out);
void l3d_pipeline_destroy(l3d_pipeline* p);
int l3d_pipeline_set_maps(l3d_pipeline* p, int eye, const float* mapx, const float* mapy);
/* nframes frames, inputs already in HBM: left/right_dev = nframes*H*W*3 bytes (device pointers).
 * Results stay on the device; counts (host int[nframes]) receives points per frame. */
int l3d_pipeline_run_dev(l3d_pipeline* p, const uint8_t* left_dev, const uint8_t* right_dev,
                         int nframes, int* counts);
/* End to end with HOST buffers (pinned or pageable): copies inputs up, runs, copies back depth
 * (nframes*H*W f32, optional), xyz (nframes*max_points*3 f64) and counts. */
int l3d_pipeline_run_host(l3d_pipeline* p, const uint8_t* left, const uint8_t* right, int nframes,
                          float* depth, double* xyz, int* counts);
/* The same two steps on nframes stereo captures as cap.read() delivers them, split as _split_frame does
 * (camera/single_usb_stereo_camera.py:143-150):
 *   split = 0: each capture is H x 2W x 3 (left = columns [0, W), right = columns [W, 2W));
 *   split = 1: each capture is 2H x W x 3 (left = rows [0, H), right = rows [H, 2H)).
 * The views are read in place as strided rows: the host form uploads each capture with one copy, the device form reads
 * the caller's buffer (nframes * 6*W*H bytes).  Results, counts and the optional depth / xyz outputs exactly as
 * l3d_pipeline_run_host / _run_dev; L3D_ERR_ARG for a split other than 0 / 1, a null buffer or nframes <= 0. */
int l3d_pipeline_run_captures_host(l3d_pipeline* p, const uint8_t* frames, int nframes, int split,
                                   float* depth, double* xyz, int* counts);
int l3d_pipeline_run_captures_dev(l3d_pipeline* p, const uint8_t* frames_dev, int nframes, int split, int* counts);
/* fetch results of the last run for frame slot i (device -> host); any pointer may be NULL.  xy (f32 pairs) and xyz
 * (f64 triples) must hold max_points entries; l3d_pipeline_fetch_points is the form with explicit capacities. */
int l3d_pipeline_fetch(l3d_pipeline* p, int frame, uint8_t* left_rect, float* depth, int16_t* disp,
                       float* xy, double* xyz, int* n_xy, int* n_xyz);
/* Laser points of frame slot i of the last run, with explicit capacities: up to xy_cap 2D centres (f64; the Simple
 * extractor's exact f64 centroids, the Steger variants' f32 centres widened) and up to xyz_cap 3D points.
 * *n_xy / *n_xyz are the counts the frame produced -- n_xy may exceed the pipeline's max_points, in which case the
 * frame's lists were truncated and the caller should re-create the pipeline with max_points >= n_xy. */
int l3d_pipeline_fetch_points(l3d_pipeline* p, int frame, double* xy, int xy_cap, double* xyz, int xyz_cap,
                              int* n_xy, int* n_xyz);
/* largest 2D point count any frame of the last run produced (compare with max_points); -1 on a null handle */
int l3d_pipeline_points_needed(l3d_pipeline* p);
/* Pack the 3D points of the first nframes frame slots of the last run into ONE device table of rows
 * (frame_id, x, y, z) (f64), frames in slot order: the payload of the NCCL gather to rank 0.
 * frame_ids[nframes] = global frame numbers; table_dev holds >= sum(counts) * 4 doubles (device
 * pointer owned by the caller, e.g. a torch tensor); *total_rows = rows written.  Synchronises. */
int l3d_pipeline_pack_points_dev(l3d_pipeline* p, int nframes, const int* frame_ids, double* table_dev,
                                 long long* total_rows);
long long l3d_pipeline_launch_count(l3d_pipeline* p);
/* Number of steps the pipeline replayed as a captured CUDA graph so far.  A step (run_dev / run_host /
 * run_captures_*) that is repeated with the same buffers, input form and frame count and whose direct enqueue is launch-bound (host enqueue time
 * > 40 % of its GPU time, e.g. 320x360 frames) is captured on its third occurrence and replayed afterwards;
 * L3D_GRAPH=1 forces, L3D_NO_GRAPH=1 disables the replay. */
long long l3d_pipeline_graph_replays(l3d_pipeline* p);
/* CUDA-event time (ms) of the whole last run (first enqueue -> last lane done) */
float l3d_pipeline_last_ms(l3d_pipeline* p);
/* Per-kernel CUDA-event timing (bench.py's roofline leg).  set_timing(1) brackets every launch of
 * the named kernel groups ("sgbm_cost", "sgbm_scan", "sgbm_wta", "wls") with events on the
 * launching stream; kernel_time returns their summed duration and count for the last run. */
int l3d_pipeline_set_timing(l3d_pipeline* p, int on);
int l3d_pipeline_kernel_time(l3d_pipeline* p, const char* which, float* ms, int* launches);
/* pinned host allocation helpers (for the e2e path; plumbing, no reference counterpart) */
void* l3d_host_alloc(long bytes);
void l3d_host_free(void* p);
/* raw device helpers for bench.py/tests (so they need no torch to stage data) */
void* l3d_dev_alloc(l3d_ctx* ctx, long bytes);
void l3d_dev_free(l3d_ctx* ctx, void* p);
int l3d_memcpy_h2d(l3d_ctx* ctx, void* dst_dev, const void* src, long bytes);
int l3d_memcpy_d2h(l3d_ctx* ctx, void* dst, const void* src_dev, long bytes);

#ifdef __cplusplus
}
#endif
#endif
