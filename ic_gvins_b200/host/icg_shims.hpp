// icg_shims.hpp -- header-only C++ shims that keep the reference's call signatures and forward to the C ABI
// (include/icgvins_b200.h).  A maintainer includes this in IG/tracking/tracking.cc and IG/ic_gvins.cc; see INTEGRATION.md.
//
// When OpenCV headers are present the shims take cv:: types; otherwise (this image has no OpenCV C++ headers) minimal
// stand-ins with the same data layout are used so that the header still compiles and can be unit-tested.
#pragma once
#include <cstdint>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/icgvins_b200.h"

#if __has_include(<opencv2/core.hpp>)
#include <opencv2/core.hpp>
namespace icg_b200 {
using Point2f = cv::Point2f;
using Mat = cv::Mat;
using Size = cv::Size;
using TermCriteria = cv::TermCriteria;
inline const uint8_t *mat_data(const Mat &m) { return m.data; }
inline int mat_stride(const Mat &m) { return (int) m.step; }
inline int mat_cols(const Mat &m) { return m.cols; }
inline int mat_rows(const Mat &m) { return m.rows; }
}  // namespace icg_b200
#else
namespace icg_b200 {
struct Point2f {
    float x, y;
};
struct Size {
    int width, height;
    Size(int w = 0, int h = 0) : width(w), height(h) {}
};
struct TermCriteria {
    enum { COUNT = 1, EPS = 2 };
    int type, maxCount;
    double epsilon;
    TermCriteria(int t = 3, int c = 30, double e = 0.01) : type(t), maxCount(c), epsilon(e) {}
};
struct Mat {  // 8-bit single channel view
    const uint8_t *data;
    int rows, cols, step;
};
inline const uint8_t *mat_data(const Mat &m) { return m.data; }
inline int mat_stride(const Mat &m) { return m.step; }
inline int mat_cols(const Mat &m) { return m.cols; }
inline int mat_rows(const Mat &m) { return m.rows; }
}  // namespace icg_b200
#endif

namespace icg_b200 {

inline void check(int rc, const char *what) {
    if (rc != ICG_OK) throw std::runtime_error(std::string(what) + ": " + icg_last_error());
}

// One tracker per Tracking object (single tracking thread, IG/ic_gvins.cc:535).
class KltContext {
public:
    KltContext(int width, int height, int max_points = 4096, int device = 0) { check(icg_klt_create(&h_, width, height, 4, max_points, device, nullptr), "icg_klt_create"); }
    ~KltContext() { icg_klt_destroy(h_); }
    KltContext(const KltContext &) = delete;
    KltContext &operator=(const KltContext &) = delete;

    // cv::calcOpticalFlowPyrLK(prev, next, prevPts, nextPts, status, err, winSize, maxLevel, criteria, flags)
    // exactly as called at IG/tracking/tracking.cc:385,390,487,493.
    void calcOpticalFlowPyrLK(const Mat &prev, const Mat &next, const std::vector<Point2f> &prevPts, std::vector<Point2f> &nextPts,
                              std::vector<uint8_t> &status, std::vector<float> &err, Size winSize, int maxLevel, TermCriteria criteria, int flags) {
        const int n = (int) prevPts.size();
        if (!(flags & ICG_OPTFLOW_USE_INITIAL_FLOW)) nextPts = prevPts;
        nextPts.resize(n);
        status.resize(n);
        err.resize(n);
        const int max_iter = (criteria.type & 1) ? criteria.maxCount : 30;
        const double eps = (criteria.type & 2) ? criteria.epsilon : 0.0;
        check(icg_klt_calc_optical_flow_pyr_lk(h_, mat_data(prev), mat_data(next), mat_stride(prev), reinterpret_cast<const float *>(prevPts.data()),
                                               reinterpret_cast<float *>(nextPts.data()), status.data(), err.data(), n, winSize.width, maxLevel, max_iter, eps,
                                               flags),
              "icg_klt_calc_optical_flow_pyr_lk");
    }

    // The whole forward + backward + gate block of Tracking::trackMappoint (IG/tracking/tracking.cc:385-403):
    // status[k] = st_fwd && st_bwd && !isOnBorder(fwd) && ptsDistance(bwd, prev) < 0.5
    void trackForwardBackward(const Mat &prev, const Mat &next, const std::vector<Point2f> &prevPts, std::vector<Point2f> &nextPts, std::vector<uint8_t> &status) {
        const int n = (int) prevPts.size();
        nextPts.resize(n);
        status.resize(n);
        check(icg_klt_track_fb(h_, mat_data(prev), mat_data(next), mat_stride(prev), reinterpret_cast<const float *>(prevPts.data()),
                               reinterpret_cast<float *>(nextPts.data()), nullptr, status.data(), n),
              "icg_klt_track_fb");
    }

private:
    icg_klt *h_ = nullptr;
};

// The window solve seam: what GVINS::gvinsOptimization hands to ceres::Solver::Solve (IG/ic_gvins.cc:1130-1239).
class WindowSolver {
public:
    WindowSolver(int max_K, int max_L, int max_F, int max_gnss = 16, int max_marg_r = 160, int device = 0) {
        check(icg_ba_create(&h_, 1, max_K, max_L, max_F, max_gnss, max_marg_r, device, nullptr), "icg_ba_create");
    }
    ~WindowSolver() { icg_ba_destroy(h_); }
    WindowSolver(const WindowSolver &) = delete;
    WindowSolver &operator=(const WindowSolver &) = delete;

    // solver.Solve(options, &problem, &summary) with options.max_num_iterations = max_iter
    icg_ba_summary Solve(const icg_ba_problem &problem, int max_iter) {
        icg_ba_summary s{};
        check(icg_ba_solve(h_, 1, &problem, max_iter, &s), "icg_ba_solve");
        return s;
    }
    // the two-pass body of gvinsOptimization (first N/4, chi2 culling, then N - N/4 iterations); out[0], out[1] = pass summaries
    void gvinsOptimization(const icg_ba_problem &problem, int num_iterations, icg_ba_summary out[2], int32_t culled[2]) {
        check(icg_ba_gvins_optimization(h_, 1, &problem, num_iterations, out, culled), "icg_ba_gvins_optimization");
    }

    // marginalization_info->marginalization() as GVINS::gvinsMarginalization drives it (IG/ic_gvins.cc:1412-1640): the prior that
    // replaces last_marginalization_info_ / last_marginalization_parameter_blocks_.  Vectors are sized here.
    struct Prior {
        int m = 0, r = 0;
        std::vector<int32_t> block_type, block_node;  // remainedBlock*: type 0 pose 1 mix 2 extrinsic 3 td; node index after the removal
        std::vector<double> x0, J0, e0;               // remainedBlockData(), linearizedJacobians() (r x r row-major), linearizedResiduals()
    };
    Prior marginalization(const icg_ba_problem &problem, int num_marg, bool after_solve = false) {  // after_solve: the window this solver just optimised (no re-upload)
        Prior P;
        const int rcap = 15 * problem.K + 7;
        P.block_type.resize(2 * problem.K + 2), P.block_node.resize(2 * problem.K + 2);
        P.x0.resize(16 * problem.K + 8), P.J0.resize((size_t) rcap * rcap), P.e0.resize(rcap);
        icg_ba_prior o{};
        o.rcap = rcap, o.block_type = P.block_type.data(), o.block_node = P.block_node.data(), o.x0 = P.x0.data(), o.J0 = P.J0.data(), o.e0 = P.e0.data();
        const int32_t nm = num_marg;
        check(after_solve ? icg_ba_marginalize_resident(h_, 1, &problem, &nm, &o) : icg_ba_marginalize(h_, 1, &problem, &nm, &o), "icg_ba_marginalize");
        P.m = o.m, P.r = o.r;
        P.block_type.resize(o.nblocks), P.block_node.resize(o.nblocks);
        P.J0.resize((size_t) o.r * o.r), P.e0.resize(o.r);
        return P;
    }

    // updateParametersFromOptimizer() + gvinsOutlierCulling() (IG/ic_gvins.cc:1232-1236): the culling verdicts of the window this solver has
    // just optimised (after_solve; otherwise the problem is uploaded first and culled at its own parameters).  problem.f_active becomes the mask
    // gvinsMarginalization finds in the map; the caller removes the flagged map points (Map::removeMappoint) and sets pose_b_c_ = R_bc, t_bc.
    struct Culling {
        icg_ba_cull_output out{};                           // ext_updated, counts, R_bc, t_bc
        std::vector<uint8_t> f_outlier, lm_ref_outlier, lm_outlier;
        std::vector<double> cam_pose, lm_pos, lm_depth;     // K x 12, L x 3, L
    };
    Culling outlierCulling(const icg_ba_problem &problem, const icg_ba_cull_input &in, bool after_solve = true) {
        Culling C;
        C.f_outlier.resize(problem.F), C.lm_ref_outlier.resize(problem.L), C.lm_outlier.resize(problem.L);
        C.cam_pose.resize((size_t) problem.K * 12), C.lm_pos.resize((size_t) problem.L * 3), C.lm_depth.resize(problem.L);
        C.out.f_outlier = C.f_outlier.data(), C.out.lm_ref_outlier = C.lm_ref_outlier.data(), C.out.lm_outlier = C.lm_outlier.data();
        C.out.cam_pose = C.cam_pose.data(), C.out.lm_pos = C.lm_pos.data(), C.out.lm_depth = C.lm_depth.data();
        if (!after_solve) check(icg_ba_upload(h_, 1, &problem), "icg_ba_upload");
        check(icg_ba_outlier_culling_resident(h_, 1, &problem, &in, &C.out), "icg_ba_outlier_culling_resident");
        return C;
    }

private:
    icg_ba *h_ = nullptr;
};

// Camera (IG/tracking/camera.cc): the point-wise model functions Tracking calls (host code in the library)
class CameraModel {
public:
    explicit CameraModel(const icg_camera &c) : c_(c) {}
    void undistortPoints(std::vector<Point2f> &pts) const { check(icg_camera_undistort_points(&c_, reinterpret_cast<float *>(pts.data()), (int) pts.size()), "icg_camera_undistort_points"); }
    void distortPoints(std::vector<Point2f> &pts) const { check(icg_camera_distort_points(&c_, reinterpret_cast<float *>(pts.data()), (int) pts.size()), "icg_camera_distort_points"); }
    Point2f distortCameraPoint(const double pc[3]) const {
        Point2f out{};
        check(icg_camera_distort_camera_points(&c_, pc, reinterpret_cast<float *>(&out), 1), "icg_camera_distort_camera_points");
        return out;
    }

private:
    icg_camera c_;
};

// cv::Ptr<cv::CLAHE> clahe_ = cv::createCLAHE(3.0, cv::Size(21, 21)) (IG/tracking/tracking.cc:62); clahe_->apply(img, img) (:141)
class Clahe {
public:
    Clahe(int width, int height, double clipLimit = 3.0, Size tileGridSize = Size(21, 21), int device = 0) {
        check(icg_clahe_create(&h_, width, height, tileGridSize.width, tileGridSize.height, clipLimit, device, nullptr), "icg_clahe_create");
    }
    ~Clahe() { icg_clahe_destroy(h_); }
    Clahe(const Clahe &) = delete;
    Clahe &operator=(const Clahe &) = delete;
    // apply(src, dst) on 8-bit single-channel images; dst may be src
    void apply(const uint8_t *src, int src_step, uint8_t *dst, int dst_step) { check(icg_clahe_apply(h_, src, src_step, dst, dst_step), "icg_clahe_apply"); }

private:
    icg_clahe *h_ = nullptr;
};

// Tracking::featuresDetection's tbb::parallel_for body (IG/tracking/tracking.cc:627-656) for all blocks in one call.
class BlockDetector {
public:
    BlockDetector(int width, int height, int max_blocks, int max_corners_per_block, int max_roi_pixels, int device = 0) : cap_(max_corners_per_block) {
        check(icg_detect_create(&h_, width, height, max_blocks, max_corners_per_block, max_roi_pixels, device, nullptr), "icg_detect_create");
    }
    ~BlockDetector() { icg_detect_destroy(h_); }
    BlockDetector(const BlockDetector &) = delete;
    BlockDetector &operator=(const BlockDetector &) = delete;

    // goodFeaturesToTrack(frame(roi), out, max_corners[b], quality, min_distance, mask(roi)) + cornerSubPix(...) per block;
    // features[b] holds block-local coordinates in OpenCV's order
    void detect(const Mat &frame, const Mat *mask, const std::vector<icg_rect> &rois, const std::vector<int32_t> &max_corners, double quality,
                double min_distance, std::vector<std::vector<Point2f>> &features) {
        const int nb = (int) rois.size();
        std::vector<float> xy((size_t) nb * cap_ * 2);
        std::vector<int32_t> cnt(nb);
        check(icg_detect_blocks(h_, mat_data(frame), mask ? mat_data(*mask) : nullptr, mat_stride(frame), nb, rois.data(), max_corners.data(), quality,
                                min_distance, 1, xy.data(), cnt.data()),
              "icg_detect_blocks");
        features.assign(nb, {});
        for (int b = 0; b < nb; b++)
            for (int k = 0; k < cnt[b]; k++) features[b].push_back(Point2f{xy[((size_t) b * cap_ + k) * 2], xy[((size_t) b * cap_ + k) * 2 + 1]});
    }

private:
    icg_detect *h_ = nullptr;
    int cap_;
};

}  // namespace icg_b200
