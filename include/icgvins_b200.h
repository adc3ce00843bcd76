/*
 * icgvins_b200.h -- C ABI of libicgvins_b200.so: B200-native (sm_100a) replacements for the two compute hot paths
 * of i2Nav-WHU/IC-GVINS.  Plain pointers and sizes only; no C++ / torch / OpenCV / Ceres types cross this boundary.
 *
 * Every entry point names the reference interface it replaces (paths relative to the reference checkout,
 * IG/ = ic_gvins/ic_gvins/).  The reference has no FFI of its own: the seams are direct library calls into
 * OpenCV (front end) and Ceres (window solve); INTEGRATION.md shows the shim a maintainer adds at each call site.
 *
 * Conventions
 *   - All functions return 0 on success, a negative ICG_E* code on failure (no exceptions, no aborts).
 *   - "host" pointers are ordinary process memory; "dev" pointers are CUDA device memory of the handle's device.
 *   - A handle is bound to one CUDA device and one stream and is NOT re-entrant (the reference calls each seam
 *     from a single thread: tracking thread IG/ic_gvins.cc:535, optimization thread IG/ic_gvins.cc:434-448).
 *   - Points are interleaved float (x, y) pairs == std::vector<cv::Point2f>::data().
 *   - There is NO CPU fallback: without a CUDA device every create() fails with ICG_ENODEVICE.
 */
#ifndef ICGVINS_B200_H
#define ICGVINS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ICG_OK 0
#define ICG_EINVAL (-1)     /* bad argument */
#define ICG_ENODEVICE (-2)  /* no usable CUDA device / driver */
#define ICG_ECUDA (-3)      /* CUDA runtime error (see icg_last_error) */
#define ICG_EUNSUPPORTED (-4) /* parameter combination the sm_100a kernels are not built for */
#define ICG_ENOMEM (-5)
/* (-6) is retired: do not reuse it */

#define ICG_OPTFLOW_USE_INITIAL_FLOW 4 /* == cv::OPTFLOW_USE_INITIAL_FLOW */

const char *icg_last_error(void);
int icg_version(void);
/* number of kernels launched by this library in this process since load / last reset (bench "gpu_launches") */
uint64_t icg_launch_count(void);
void icg_launch_count_reset(void);

/* ===================================================================================================== *
 *  Path A: pyramidal KLT front end
 * ===================================================================================================== */
typedef struct icg_klt icg_klt;

/*
 * Create a tracker for width x height u8 images.  n_slots device-resident image slots (each holds a 4-level
 * pyramid, levels 0..3 as cv::buildOpticalFlowPyramid(img, winSize 21, maxLevel 3) produces them);
 * max_points = largest n of one call.  stream may be NULL (handle creates its own) or a cudaStream_t.
 */
int icg_klt_create(icg_klt **h, int width, int height, int n_slots, int max_points, int device, void *stream);
void icg_klt_destroy(icg_klt *h);

/*
 * Drop-in for cv::calcOpticalFlowPyrLK as the reference calls it (IG/tracking/tracking.cc:385,390,487,493):
 *   cv::calcOpticalFlowPyrLK(prev, next, prevPts, nextPts, status, err, Size(win,win), max_level,
 *                            TermCriteria(COUNT+EPS, max_iter, eps), flags)
 * Host buffers, synchronous.  next_xy is in/out (initial flow when flags has ICG_OPTFLOW_USE_INITIAL_FLOW).
 * err may be NULL (the reference never reads it).  Only win == 21 and max_level <= 3 are built
 * (the values at all four call sites); anything else returns ICG_EUNSUPPORTED.
 * Pyramids are cached per image content (the reference passes the same two images to 4 calls per frame).
 */
int icg_klt_calc_optical_flow_pyr_lk(icg_klt *h, const uint8_t *prev, const uint8_t *next, int stride,
                                     const float *prev_xy, float *next_xy, uint8_t *status, float *err, int n,
                                     int win, int max_level, int max_iter, double eps, int flags);

/*
 * Fused replacement for the forward LK + backward LK + gate block (IG/tracking/tracking.cc:385-403 and :487-506):
 *   status[k] = st_fwd && st_bwd && !isOnBorder(fwd) && ptsDistance(bwd, prev) < 0.5
 * next_xy in: predicted positions, out: forward result.  back_xy (may be NULL) receives the backward result.
 */
int icg_klt_track_fb(icg_klt *h, const uint8_t *prev, const uint8_t *next, int stride, const float *prev_xy,
                     float *next_xy, float *back_xy, uint8_t *status, int n);

/* ---- device-resident / batched API (throughput mode: many independent streams per GPU) ---- */

/* async H2D of one frame into slot's level 0 (host memory should be pinned for overlap) + pyramid build */
int icg_klt_upload(icg_klt *h, int slot, const uint8_t *host_img, int stride);
/* async H2D of one frame into slot's level 0 only (no pyramid build; pair with icg_klt_build_pyramids) */
int icg_klt_upload_level0(icg_klt *h, int slot, const uint8_t *host_img, int stride);
/* async H2D of `count` frames into the level-0 planes of slots [first_slot, first_slot + count) in one call (throughput mode: one new frame
 * of every stream per step): linear DMA copies into a device staging buffer + one scatter kernel; no pyramid build
 * (pair with icg_klt_build_pyramids).  host_imgs[k] should be pinned. */
int icg_klt_upload_batch(icg_klt *h, int first_slot, int count, const uint8_t *const *host_imgs, int stride);
/* synchronous D2H of one pyramid level of a slot into a host buffer of row stride `stride` (parity tests) */
int icg_klt_download_level(icg_klt *h, int slot, int level, uint8_t *host_img, int stride);
/* device pointer + pitch of a slot's level-0 plane, so a producer on the same device can write frames in place */
int icg_klt_slot_level0(icg_klt *h, int slot, void **dev_ptr, int *pitch);
/* device pointer + pitch + size of level `level` (read-back for parity tests) */
int icg_klt_slot_level(icg_klt *h, int slot, int level, void **dev_ptr, int *pitch, int *w, int *hgt);
/* build levels 1..3 for slots [first, first+count) from their level-0 planes (one launch) */
int icg_klt_build_pyramids(icg_klt *h, int first_slot, int count);
/*
 * Batched forward+backward tracking of n_total points, all arrays in DEVICE memory:
 *   slots[2k], slots[2k+1] = (prev slot, next slot) of point k;  prev_xy/init_xy/fwd_xy/bwd_xy: float2 per point.
 * Asynchronous on the handle's stream.  mode 0: forward only (status = raw LK status);
 * mode 1: fused forward+backward+gates (as icg_klt_track_fb).
 */
int icg_klt_track_batch_dev(icg_klt *h, int n_total, const int32_t *dev_slots, const float *dev_prev_xy,
                            const float *dev_init_xy, float *dev_fwd_xy, float *dev_bwd_xy, uint8_t *dev_status,
                            int mode);
int icg_klt_sync(icg_klt *h);

/* ----- camera model of path A (SURVEY 8a row A6): HOST functions by design (<= 300 points per frame, FP64) ----- */
typedef struct icg_camera {
    double fx, fy, cx, cy, skew; /* intrinsic_(0,0), (1,1), (0,2), (1,2), (0,1)   (IG/tracking/camera.cc:29-33) */
    double k1, k2, p1, p2, k3;   /* distortion_ in OpenCV order                    (:35-39) */
} icg_camera;
/* Camera::undistortPoints (IG/tracking/camera.cc:72-74) == cv::undistortPoints(pts, pts, K, D, Mat(), K); in place on n (x, y) floats */
int icg_camera_undistort_points(const icg_camera *c, float *pts_xy, int n);
/* Camera::distortPoints / distortPoint (:76-104): pixel2cam -> radtan -> cam2pixel, in place */
int icg_camera_distort_points(const icg_camera *c, float *pts_xy, int n);
/* Camera::distortCameraPoint (:106-120) for n camera-frame points (x, y, z) -> distorted pixels */
int icg_camera_distort_camera_points(const icg_camera *c, const double *pc_xyz, float *px_xy, int n);
/* Camera::pixel2cam (:126-130): pixels -> normalised camera points (x, y, 1) */
int icg_camera_pixel2cam(const icg_camera *c, const float *px_xy, double *cam_xyz, int n);
/* Camera::world2pixel (:144-146) = cam2pixel(R^T (pw - t)); R9 row-major body/camera attitude, t3 its position */
int icg_camera_world2pixel(const icg_camera *c, const double *R9, const double *t3, const double *pw_xyz, float *px_xy, int n);

/* Drop-in for cv::findFundamentalMat(pts1, pts2, cv::FM_RANSAC, threshold, confidence, status) as Tracking::trackReferenceFrame calls it
 * (IG/tracking/tracking.cc:547, maxIters = 1000): status[i] = 1 for the inliers of the best 7-point model; F9 (row-major, may be NULL)
 * receives that model.  HOST function in this round (<= 300 pairs, serially adaptive loop); the inlier mask is identical to OpenCV's
 * (tests/golden/fundamental_golden.npz).  n >= 15 as at the call site. */
int icg_find_fundamental_mat_ransac(const float *pts1_xy, const float *pts2_xy, int n, double threshold, double confidence, int max_iters,
                                    uint8_t *status, double *F9);

/* Tracking::triangulatePoint (IG/tracking/tracking.cc:796-808) for n point pairs: Tcw0 = n x (3 x 4 row-major T_c_w of the reference frames),
 * Tcw1 = the current frame's, pc0 / pc1 = normalised camera coordinates (x, y); pw = dehomogenised null vector of the 4 x 4 design matrix.
 * Host function. */
int icg_triangulate_points(const double *Tcw0, const double *Tcw1, const double *pc0_xy, const double *pc1_xy, int n, double *pw_xyz);

/* Tracking::calculateHistigram (IG/tracking/tracking.cc:88-104): the brightness statistic of the histogram gate in
 * Tracking::preprocessing (:115-133).  Host function (one pass over the frame). */
int icg_tracking_histogram(const uint8_t *img, int width, int height, int stride, double *out);

/* ----- SURVEY 8f ranks 2-4 on the DEVICE (csrc/geom.cu): the same functions as the host entry points above / icg_imu_preintegrate below, batched as
 * CUDA kernels (one __host__ __device__ definition of the arithmetic, csrc/geom_core.cuh).  Host buffers in / out, synchronous. ----- */
typedef struct icg_geom icg_geom;
int icg_geom_create(icg_geom **h, int device, void *stream);
void icg_geom_destroy(icg_geom *h);
/* Camera::undistortPoints / distortPoints (IG/tracking/camera.cc:72-104), thread per point, any n */
int icg_geom_undistort_points(icg_geom *h, const icg_camera *c, float *pts_xy, int n);
int icg_geom_distort_points(icg_geom *h, const icg_camera *c, float *pts_xy, int n);
/* cv::findFundamentalMat(FM_RANSAC) (IG/tracking/tracking.cc:547): all max_iters subsets of the cv::RNG stream are drawn up front (they do not depend on
 * which model wins), every hypothesis is solved (7-point) and scored against the n pairs on the device, the host replays OpenCV's serial acceptance
 * rule and adaptive iteration bound on the inlier counts.  Same inlier mask as icg_find_fundamental_mat_ransac / OpenCV. */
int icg_geom_find_fundamental_mat_ransac(icg_geom *h, const float *pts1_xy, const float *pts2_xy, int n, double threshold, double confidence, int max_iters,
                                         uint8_t *status, double *F9);
/* Tracking::triangulatePoint (IG/tracking/tracking.cc:796-808), thread per pair */
int icg_geom_triangulate_points(icg_geom *h, const double *Tcw0, const double *Tcw1, const double *pc0_xy, const double *pc1_xy, int n, double *pw_xyz);
/* icg_imu_preintegrate for n_intervals intervals at once (doReintegration over a window, IG/ic_gvins.cc:1680-1695; throughput mode): state16 is
 * n_intervals x 16, imu the concatenated sample rows, imu_off[k] .. imu_off[k+1] the rows of interval k (row imu_off[k] = the sample at its start);
 * iewn3 / gravity3 / noise5 shared; iewn3 == NULL: PreintegrationNormal.  blobs_out n_intervals x ICG_IMU_BLOB_DOUBLES, end_states10 may be NULL. */
int icg_geom_imu_preintegrate_batch(icg_geom *h, int n_intervals, const double *state16, const double *iewn3, const double *gravity3, const double *noise5,
                                    const double *imu, const int32_t *imu_off, double *blobs_out, double *end_states10);

/* ----- pre-pass of path A: cv::CLAHE (IG/tracking/tracking.cc:62 createCLAHE(3.0, Size(21, 21)); :141 clahe_->apply(img, img)) ----- */
typedef struct icg_clahe icg_clahe;
int icg_clahe_create(icg_clahe **h, int width, int height, int tiles_x, int tiles_y, double clip_limit, int device, void *stream);
void icg_clahe_destroy(icg_clahe *h);
/* Drop-in for cv::CLAHE::apply(src, dst) on 8-bit single-channel host buffers (dst may alias src): H2D, per-tile LUTs, bilinear LUT
 * interpolation, D2H; synchronous.  Bit-exact with OpenCV (tests/golden/clahe_golden.npz). */
int icg_clahe_apply(icg_clahe *h, const uint8_t *src, int src_stride, uint8_t *dst, int dst_stride);
/* Device-resident variant (asynchronous on the handle's stream): src / dst are device pointers, e.g. the level-0 plane of a KLT slot
 * (icg_klt_slot_level0) so that upload -> CLAHE -> pyramid -> track never leaves HBM; dst may alias src. */
int icg_clahe_apply_dev(icg_clahe *h, const uint8_t *dev_src, int src_pitch, uint8_t *dev_dst, int dst_pitch);
/* Frame-batched device-resident variant: n_frames frames (frame f at dev_src + f * src_frame_stride, written to dev_dst + f * dst_frame_stride;
 * in place allowed) in one launch pair.  hist_out (host, n_frames doubles, may be NULL): Tracking::calculateHistigram of every RAW frame
 * (IG/tracking/tracking.cc:88-104), accumulated by the LUT pass at no extra read of the frame -- the statistic of the histogram gate in
 * Tracking::preprocessing (:115-133).  With hist_out the call synchronises (the host decides whether to skip the frame); without, it is asynchronous. */
int icg_clahe_apply_batch_dev(icg_clahe *h, int n_frames, const uint8_t *dev_src, int src_pitch, size_t src_frame_stride, uint8_t *dev_dst, int dst_pitch,
                              size_t dst_frame_stride, double *hist_out);
int icg_clahe_sync(icg_clahe *h);

/* ----- detection leg of path A: Tracking::featuresDetection (IG/tracking/tracking.cc:576-688) ----- */
typedef struct icg_rect {
    int32_t x, y, w, h;
} icg_rect;
typedef struct icg_detect icg_detect;
/* width x height frames; up to max_blocks ROIs per call, each at most max_roi_pixels pixels, at most
 * max_corners_per_block corners returned per block. */
int icg_detect_create(icg_detect **h, int width, int height, int max_blocks, int max_corners_per_block, int max_roi_pixels, int device, void *stream);
void icg_detect_destroy(icg_detect *h);
/*
 * The body of the tbb::parallel_for over blocks (IG/tracking/tracking.cc:627-656) for all blocks in one call:
 *   cv::goodFeaturesToTrack(frame(roi), out, max_corners[b], quality, min_distance, mask(roi))          (:647)
 *   cv::cornerSubPix(frame(roi), out, Size(5,5), Size(-1,-1), TermCriteria(COUNT+EPS, 20, 0.01))        (:651, when do_subpix)
 * with C++ ROI semantics (the derivative of a block reads the frame beyond the block edge).  img / mask are full frames
 * (mask may be NULL == all 255).  out_xy: n_blocks x max_corners_per_block x 2 floats, block-LOCAL coordinates in
 * OpenCV's order (strength descending, ties by address descending); out_n: corners per block.  Host buffers, synchronous.
 * A single ROI covering the frame reproduces the stand-alone cv::goodFeaturesToTrack / cv::cornerSubPix calls.
 */
int icg_detect_blocks(icg_detect *h, const uint8_t *img, const uint8_t *mask, int stride, int n_blocks, const icg_rect *rois,
                      const int32_t *max_corners, double quality, double min_distance, int do_subpix, float *out_xy, int32_t *out_n);
/* The same for n_frames DEVICE-resident frames in one call (throughput mode / the keyframe path of many streams): frame f starts at
 * dev_img + f * frame_stride (row pitch `pitch` bytes; e.g. the level-0 planes of consecutive KLT slots, icg_klt_slot_level0), dev_mask (NULL or the
 * same geometry) likewise; the n_blocks ROIs apply to every frame; max_corners is n_frames x n_blocks (or NULL); outputs are host arrays of
 * n_frames x n_blocks (x cap x 2).  The handle's max_blocks must cover n_frames * n_blocks. */
int icg_detect_blocks_dev(icg_detect *h, int n_frames, const uint8_t *dev_img, int pitch, size_t frame_stride, const uint8_t *dev_mask, int n_blocks,
                          const icg_rect *rois, const int32_t *max_corners, double quality, double min_distance, int do_subpix, float *out_xy,
                          int32_t *out_n);
/* Drop-in for cv::cornerSubPix(img, corners, Size(5,5), Size(-1,-1), (COUNT+EPS, 20, 0.01)) on the whole frame; corners in/out */
int icg_corner_subpix(icg_detect *h, const uint8_t *img, int stride, float *corners_xy, int n);

/* ===================================================================================================== *
 *  Path B: sliding-window factor-graph solve
 * ===================================================================================================== */
/*
 * One window problem == what GVINS::gvinsOptimization hands to Ceres (IG/ic_gvins.cc:1130-1239, 1697-1909):
 *   parameter blocks  statedatalist_[k].pose[7] = (p, q_xyzw), .mix[9] = (v, bg, ba)      (IG/preintegration/integration_state.h:53-66)
 *                     extrinsic_[8] = (t_bc, q_bc xyzw, td)                                 (IG/ic_gvins.cc:1736-1756)
 *                     invdepthlist_ values, one per landmark                                (IG/ic_gvins.cc:1727)
 *   residual blocks   ReprojectionFactor(pose_ref, pose_obs, extrinsic, invdepth, td) + HuberLoss(1.0)   (:1826-1831)
 *                     PreintegrationFactor(pose_k, mix_k, pose_k+1, mix_k+1)                              (:1870-1872)
 *                     ImuErrorFactor(mix_last), ImuPosePriorFactor(pose_0), ImuMixPriorFactor(mix_0)       (:1877-1887)
 *                     GnssFactor(pose_node) + HuberLoss(1.0) in the first pass                             (:1896-1903)
 *                     MarginalizationFactor(remained blocks)                                               (:1158-1161)
 * All arrays are caller-owned host memory; pose/mix/ext/invdepth are updated in place by the solve
 * (as Ceres mutates the reference's parameter arrays in place).
 */
#define ICG_IMU_BLOB_DOUBLES 480
/* IMU preintegration blob (doubles): [0] delta_time, [1..3] delta p, [4..6] delta v, [7..10] delta q (x,y,z,w),
 * [11..13] bg, [14..16] ba (linearisation biases), [17..19] gravity, [20..22] iewn,
 * [23] S0 = sum_i dt_i, [24..26] S1 = sum_i dt_i * pn_i   (the two moments of pn_ that
 *      PreintegrationEarth::evaluate's position-compensation loop needs, IG/preintegration/preintegration_earth.cc:55-59),
 * [27..251] jacobian_ 15x15 row-major, [252..476] covariance_ 15x15 row-major,
 * [477] factor form: 0 = PreintegrationEarth (IG/preintegration/preintegration_earth.cc), 1 = PreintegrationNormal
 *       (preintegration_normal.cc, `iswithearth: false`: iewn = 0, S0 = S1 = 0), [478..479] reserved. */
typedef struct icg_ba_problem {
    int32_t K, L, F;
    double *pose;     /* K*7 in/out */
    double *mix;      /* K*9 in/out */
    double *ext;      /* 8   in/out */
    double *invdepth; /* L   in/out */
    int32_t ext_const, td_const; /* SetParameterBlockConstant (IG/ic_gvins.cc:1750,1758) */
    const int32_t *f_lm, *f_ref, *f_obs; /* F each: landmark, reference node, observing node */
    const double *f_const;               /* F*14: pts0[3] pts1[3] vel0[3] vel1[3] td0 td1 */
    const uint8_t *f_active;             /* F, or NULL == all active (RemoveResidualBlock, IG/ic_gvins.cc:1291) */
    double reproj_std;
    int32_t reproj_huber;
    int32_t n_imu;
    const double *imu_blob; /* n_imu * ICG_IMU_BLOB_DOUBLES; factor k joins node k and k+1 */
    int32_t has_imu_error;
    int32_t has_pose_prior;
    const double *pose_prior, *pose_prior_std; /* 7, 6 */
    int32_t has_mix_prior;
    const double *mix_prior, *mix_prior_std; /* 9, 9 */
    int32_t n_gnss;
    const int32_t *gnss_node;
    const double *gnss_blh, *gnss_std; /* n_gnss*3 each */
    double lever[3];
    int32_t gnss_huber;
    int32_t marg_r, marg_nblocks;                    /* 0 == no prior */
    const int32_t *marg_block_type, *marg_block_node; /* type 0 pose(node) 1 mix(node) 2 extrinsic 3 td */
    const double *marg_x0, *marg_J0, *marg_e0;        /* concatenated x0 (global sizes), J0 row-major r x r, e0 */
} icg_ba_problem;

typedef struct icg_ba_summary {
    int32_t iterations;           /* LM iterations executed */
    int32_t num_successful_steps; /* ceres::Solver::Summary::num_successful_steps (IG/ic_gvins.cc:1186) */
    int32_t termination;          /* 0 NO_CONVERGENCE (max iterations), 1 CONVERGENCE, 2 FAILURE */
    int32_t reserved;
    double initial_cost, final_cost, final_radius;
} icg_ba_summary;

/* B3 (host side, as in the reference: fusion thread, IG/ic_gvins.cc:917-919): IMU preintegration propagation
 * PreintegrationEarth::resetState/integrationProcess/updateJacobianAndCovariance (IG/preintegration/preintegration_earth.cc:205-338).
 * state16 = p[3] q_xyzw[4] v[3] bg[3] ba[3] at the interval start; noise5 = gyr_arw, acc_vrw, gyr_bias_std, acc_bias_std, corr_time;
 * imu = n rows of (dt, dtheta[3], dvel[3]), row 0 being the sample at the interval start.  Writes the factor blob and the
 * mechanised end state (p, q_xyzw, v).  Sequential recurrence; runs on the calling host thread.
 * iewn3 == NULL selects PreintegrationNormal (PreintegrationBase::integration + PreintegrationNormal::updateJacobianAndCovariance,
 * IG/preintegration/preintegration_base.cc:39-70, preintegration_normal.cc:195-232). */
int icg_imu_preintegrate(const double *state16, const double *iewn3, const double *gravity3, const double *noise5, const double *imu,
                         int n, double *blob_out, double *end_state10);

typedef struct icg_ba icg_ba;
/*
 * Solver for batches of up to max_windows windows of at most max_K nodes / max_L landmarks / max_F reprojection
 * factors each (throughput mode: one window per independent stream).  stream may be NULL.
 */
int icg_ba_create(icg_ba **h, int max_windows, int max_K, int max_L, int max_F, int max_gnss, int max_marg_r, int device,
                  void *stream);
void icg_ba_destroy(icg_ba *h);
/*
 * Drop-in for `ceres::Solver::Solve(options, &problem, &summary)` with LEVENBERG_MARQUARDT + DENSE_SCHUR
 * (IG/ic_gvins.cc:1143-1146, 1183, 1217) on n_windows independent problems at once.  Parameters are updated in place.
 */
int icg_ba_solve(icg_ba *h, int n_windows, const icg_ba_problem *problems, int max_num_iterations, icg_ba_summary *summaries);
/* The three stages of icg_ba_solve, exposed for device-resident operation (throughput mode / benchmarking):
 *   upload   : pack + H2D of n problems (what AddParameterBlock / AddResidualBlock build, IG/ic_gvins.cc:1697-1909)
 *   run      : enqueue max_num_iterations LM iterations, asynchronously on the handle's stream; restart != 0 first restores
 *              the parameters that were uploaded (re-solve the same problems)
 *   download : D2H of the parameters into the problems' arrays (problems may be NULL) + summaries; synchronises. */
int icg_ba_upload(icg_ba *h, int n_windows, const icg_ba_problem *problems);
int icg_ba_run(icg_ba *h, int max_num_iterations, int restart);
int icg_ba_download(icg_ba *h, int n_windows, const icg_ba_problem *problems, icg_ba_summary *summaries);
/*
 * Drop-in for the body of GVINS::gvinsOptimization (IG/ic_gvins.cc:1130-1239) on n_windows problems:
 *   Solve(max_num_iterations = N/4) with HuberLoss on GNSS + reprojection         (:1183)
 *   gnssOutlierCullingByChi2 (chi2 > 7.815 -> std *= sqrt(chi2/7.815))            (:1241-1267)
 *   removeReprojectionFactorsByChi2(5.991)                                        (:1269-1297)
 *   GNSS factors re-added without loss, Solve(max_num_iterations = N - N/4)       (:1202-1217)
 * entirely on the device (no host round trip between the passes).  Parameters are updated in place; the problems'
 * f_active (must be non-NULL to receive the removals) and gnss_std arrays are updated in place too, as the reference mutates
 * `gnss->std` and removes residual blocks.  summaries: 2 per window (pass 1, pass 2), may be NULL.
 * culled: 2 ints per window (reprojection factors removed, GNSS fixes re-weighted), may be NULL.
 * icg_ba_run_gvins is the asynchronous device-only stage for problems already uploaded.
 */
int icg_ba_gvins_optimization(icg_ba *h, int n_windows, const icg_ba_problem *problems, int num_iterations, icg_ba_summary *summaries,
                              int32_t *culled);
int icg_ba_run_gvins(icg_ba *h, int num_iterations, int restart);
/* The same call split in two so that a caller driving several handles (streams) can overlap them: _begin packs, uploads and
 * enqueues (asynchronous on the handle's stream), _end synchronises and writes the results back. */
int icg_ba_gvins_optimization_begin(icg_ba *h, int n_windows, const icg_ba_problem *problems, int num_iterations);
int icg_ba_gvins_optimization_end(icg_ba *h, int n_windows, const icg_ba_problem *problems, icg_ba_summary *summaries, int32_t *culled);
int icg_ba_sync(icg_ba *h);
/*
 * Drop-in for `MarginalizationInfo::marginalization()` as GVINS::gvinsMarginalization drives it (IG/ic_gvins.cc:1412-1640,
 * IG/factors/marginalization_info.h:73-253): for each window, the num_marg oldest nodes (pose + mix) and the inverse depths of the
 * landmarks anchored in them are marginalized out of [previous prior, GNSS at those nodes, preintegration factors 0..num_marg-1,
 * first-window pose / mix priors, reprojection factors of those landmarks] (no loss functions, every Jacobian, as
 * ResidualBlockInfo::Evaluate does), linearised at the parameter values in `problems`.  Output: the new prior in the layout
 * icg_ba_problem.marg_* consumes -- remained blocks (node indices already shifted by num_marg), x0 = remainedBlockData(),
 * J0 = linearizedJacobians() (r x r row-major, rows in ascending eigenvalue order), e0 = linearizedResiduals() -- plus, optionally,
 * the Schur complement itself (Hp, bp).  Arrays are caller-allocated: block_type/block_node 2K+2 ints, x0 16K+8, J0/Hp rcap*rcap,
 * e0/bp rcap doubles with rcap >= 15*(K - num_marg) + 7.  Column order inside the marginalized / remained groups is
 * [pose_k, mix_k ascending k | landmarks ascending] / [pose_k, mix_k (touched blocks only) | ext | td]; the reference's order is that of
 * an unordered_map (implementation-defined) and only permutes rows / columns.
 */
typedef struct icg_ba_prior {
    int32_t m, r, nblocks;            /* out: marginalizedSize(), remainedSize(), number of remained blocks */
    int32_t rcap;                     /* in: capacity of J0 / e0 / Hp / bp */
    int32_t *block_type, *block_node; /* out */
    double *x0, *J0, *e0;             /* out */
    double *Hp, *bp;                  /* out, may be NULL */
} icg_ba_prior;
int icg_ba_marginalize(icg_ba *h, int n_windows, const icg_ba_problem *problems, const int32_t *num_marg, icg_ba_prior *out);
/* The same on the windows the handle already holds: gvinsMarginalization runs right after gvinsOptimization on the same window
 * (IG/ic_gvins.cc:560-567 -> 1412), so after icg_ba_gvins_optimization[_end] / icg_ba_solve the device copy already has the optimised
 * parameters, the culled factor set and the re-weighted GNSS sigmas; nothing is packed or uploaded again.  `problems` must be the array
 * of that solve (n_windows equal to the uploaded count; read for the factor structure and x0 only). */
int icg_ba_marginalize_resident(icg_ba *h, int n_windows, const icg_ba_problem *problems, const int32_t *num_marg, icg_ba_prior *out);
/*
 * The end of GVINS::gvinsOptimization on the windows the handle holds: updateParametersFromOptimizer (IG/ic_gvins.cc:1299-1389) and
 * gvinsOutlierCulling (:1035-1128), in one launch over the batch.  Per window:
 *   1. extrinsic gate (only with estimate_extrinsic): the solved extrinsic replaces (R_bc, t_bc) unless |dt| > 1 m or
 *      |vec(quaternion(R R_bc^T))| * 180 / pi > 5 (sin(theta / 2) in "degrees", as the reference writes it);
 *   2. camera pose of every node, MISC::stateToCameraPose (IG/misc.cc:102-108), with the gated extrinsic;
 *   3. map point of every landmark: R_ref (pixel2cam(lm_ref_kp) / invdepth) + t_ref;
 *   4. every observation in mappoint->observations() order -- the reference observation at position lm_ref_pos, the landmark's factors in
 *      ascending factor index around it (the order addReprojectionFactors creates them in, :1777-1834) -- through
 *      Tracking::isGoodToTrack(kp, pose, pos, 3.0) (1 < z_c < 200, |world2pixel - kp| <= 3 std): a bad one is a feature outlier; a bad
 *      reference observation makes the landmark an outlier (num1) and ends its loop; then fewer than 2 good errors (num2) or a mean error
 *      above std (num3) makes it an outlier.  f_active is ignored: every factor of the window is evaluated.
 * Afterwards f_active[f] = !f_outlier[f] && !lm_outlier[f_lm[f]] on the device and in problems[w].f_active (updated in place, as
 * icg_ba_gvins_optimization does), so icg_ba_marginalize_resident builds the prior from the factors gvinsMarginalization finds in the map
 * (:1559-1590).  Removing the map points (Map::removeMappoint) stays with the caller.  `problems` must be the array of the last upload
 * (n_windows equal to the uploaded count); it is read for f_lm / f_ref and written through f_active only.
 * Errors: ICG_EINVAL when a required array is NULL, f_ref[f] != lm_ref_node[f_lm[f]], lm_ref_pos is outside [0, factors of the landmark]
 * or n_windows differs from the uploaded count (nothing is launched); ICG_EUNSUPPORTED on a landmark-sharded handle.
 */
typedef struct icg_ba_cull_input {
    icg_camera cam;                /* pinhole part only: fx, fy, cx, cy, skew (Camera::world2pixel, IG/tracking/camera.cc:129-146) */
    double reprojection_error_std; /* pixels (IG/ic_gvins.cc:133) */
    int32_t estimate_extrinsic;    /* optimize_estimate_extrinsic_ */
    int32_t reserved;
    double R_bc[9], t_bc[3];       /* pose_b_c_ before the call (R row-major): the gate's baseline */
    const float *f_kp;             /* F x 2: keyPoint() of each factor's observing feature */
    const float *lm_ref_kp;        /* L x 2: referenceKeypoint() */
    const int32_t *lm_ref_node;    /* L: reference node (a landmark may have no factor) */
    const int32_t *lm_ref_pos;     /* L: position of the reference observation in observations(), 0 .. factors of the landmark */
} icg_ba_cull_input;
typedef struct icg_ba_cull_output {
    int32_t ext_updated;           /* 1: pose_b_c_ took the solved extrinsic */
    int32_t counts[5];             /* outliers_[0] (map-point outliers, num1 + (num2 or num3)), outliers_[1] (feature outliers), num1, num2, num3 */
    double R_bc[9], t_bc[3];       /* pose_b_c_ after the gate */
    double *cam_pose;              /* K x 12 (R_wc row-major, t_wc), may be NULL */
    double *lm_pos, *lm_depth;     /* L x 3 and L, may be NULL */
    uint8_t *f_outlier;            /* F: feature outlier (setOutlier on the observing feature) */
    uint8_t *lm_ref_outlier;       /* L: the reference observation was flagged */
    uint8_t *lm_outlier;           /* L: bit 0 num1, bit 1 num2, bit 2 num3 */
} icg_ba_cull_output;
int icg_ba_outlier_culling_resident(icg_ba *h, int n_windows, const icg_ba_problem *problems, const icg_ba_cull_input *in, icg_ba_cull_output *out);
/*
 * Landmark sharding of the window solve across the GPUs of one box (SURVEY.md 8e), over PEER MEMORY: every process (one per GPU) uploads
 * the same camera-side problem but only ITS landmarks and their reprojection factors; window w of the batch is owned by rank w mod world.
 * Every rank STORES its packed reduction operand straight into the owner's inbox over NVLink; the owner sums the `world` slots in rank
 * order while assembling the reduced camera system (the reduction is fused into the consumer, no collective kernel), evaluates the
 * camera-only factors, solves the system on a thread-block cluster and stores the camera step into every rank's step buffer; a 5-scalar
 * all-to-all closes the attempt.  Three release/acquire flag synchronisations per LM attempt, no host round trip, deterministic (fixed
 * summation order, independent of arrival order).
 *   icg_ba_shard_export : allocates this rank's exchange buffer for a group of `world` ranks (<= 8, one box) and writes the
 *                         ICG_SHARD_BLOB_BYTES blob the other ranks need (CUDA IPC handle + process-local pointer);
 *   icg_ba_shard_connect: blobs = world x ICG_SHARD_BLOB_BYTES in rank order (the caller gathers them, e.g. torch.distributed
 *                         all_gather_object); handles living in the same process are connected by pointer (peer access enabled);
 *   icg_ba_shard_error  : non-zero if a flag wait timed out (a rank did not enqueue the same sequence).
 * All ranks must create their handles with the same max_windows and max_K and call the solve entry points with the same arguments.
 * Once a handle has called icg_ba_shard_export it stays on this pipeline until it is destroyed.
 */
#define ICG_SHARD_BLOB_BYTES 128
int icg_ba_shard_export(icg_ba *h, int rank, int world, uint8_t *blob);
int icg_ba_shard_connect(icg_ba *h, const uint8_t *blobs);
int icg_ba_shard_error(icg_ba *h);
/* Problem::EvaluateResidualBlock(id, false, &cost, NULL, NULL) for every reprojection / GNSS block
 * (the two chi-square passes, IG/ic_gvins.cc:1251,1278): cost = 0.5 |r|^2 without the loss function. */
int icg_ba_residual_costs(icg_ba *h, const icg_ba_problem *problem, double *reproj_cost /* F */, double *gnss_cost /* n_gnss */);
/* Single-factor evaluation with the Ceres CostFunction::Evaluate contract (IG/factors/reprojection_factor.h:55):
 * residuals[2]; jacobians row-major 2x7, 2x7, 2x7, 2x1, 2x1 (any may be NULL).  Computed on the device. */
int icg_ba_reproj_evaluate(icg_ba *h, const double *pose0, const double *pose1, const double *ext, const double *invdepth,
                           const double *td, const double *f_const14, double std, double *residuals, double **jacobians);
/* PreintegrationFactor::Evaluate (IG/preintegration/preintegration_factor.h:45): residuals[15], jacobians 15x7,15x9,15x7,15x9 */
int icg_ba_imu_evaluate(icg_ba *h, const double *imu_blob, const double *pose0, const double *mix0, const double *pose1,
                        const double *mix1, double *residuals, double **jacobians);

/* The remaining CostFunction::Evaluate seams of the window graph (same contract: residuals, then one row-major Jacobian per parameter
 * block with its GLOBAL size, any may be NULL; computed on the device):
 *   GnssFactor::Evaluate            (IG/factors/gnss_factor.h:43-71)                 residuals[3], jacobians[0] 3x7
 *   ImuPosePriorFactor::Evaluate    (IG/preintegration/imu_pose_prior_factor.h:42-68) residuals[6], jacobians[0] 6x7
 *   ImuMixPriorFactor::Evaluate     (IG/preintegration/imu_mix_prior_factor.h:40-75)  residuals[9], jacobians[0] 9x9
 *   ImuErrorFactor::Evaluate        (IG/preintegration/imu_error_factor.h:45-91)      residuals[6], jacobians[0] 6x9
 *   MarginalizationFactor::Evaluate (IG/factors/marginalization_factor.h:47-101)      residuals[r], jacobians[b] r x (7 | 9 | 7 | 1);
 *       parameters[b] = the current value of remained block b (block_type as in icg_ba_problem.marg_block_type), x0 / J0 / e0 the prior. */
int icg_ba_gnss_evaluate(icg_ba *h, const double *pose, const double *blh, const double *std3, const double *lever, double *residuals,
                         double **jacobians);
int icg_ba_pose_prior_evaluate(icg_ba *h, const double *pose, const double *prior7, const double *std6, double *residuals, double **jacobians);
int icg_ba_mix_prior_evaluate(icg_ba *h, const double *mix, const double *prior9, const double *std9, double *residuals, double **jacobians);
int icg_ba_imu_error_evaluate(icg_ba *h, const double *mix, double *residuals, double **jacobians);
int icg_ba_marg_factor_evaluate(icg_ba *h, int r, int nblocks, const int32_t *block_type, const double *const *parameters, const double *x0,
                                const double *J0, const double *e0, double *residuals, double **jacobians);

#ifdef __cplusplus
}
#endif
#endif /* ICGVINS_B200_H */
