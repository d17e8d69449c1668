// img_completion.h -- the header the reference includes but never shipped
// (`#include "img_completion.h"`: src/DC_lidar_only/img_completion.cpp:15, main.cpp:1, utils.cpp:3), implemented
// on top of the C ABI of libdcmt.so (include/dcmt.h).
//
// With OpenCV available (the reference's own build) the reference's signatures are defined on cv::Mat, so that
// main.cpp / main_lc.cpp / main_sl.cpp link against libdcmt.so instead of compiling img_completion.cpp /
// img_completion_lc.cpp and the function bodies of main_sl.cpp:715-885:
//
//     void img_completion(const cv::Mat&, cv::Mat&, const bool& extr, const std::string& blur_type);      img_completion.cpp:17
//     void interpolate_with_superpixels(Slic&, const cv::Mat&, cv::Mat&, const std::string&, int);        img_completion_lc.cpp:34
//     void calculateMeasuementDerivatives(cv::Mat& img);                                                  main_sl.cpp:715
//     bool calculateObservationDerivatives(const cv::Mat&, const Eigen::Vector2f, float&, Eigen::Vector2f&);        :747
//     void optimize_IG(cv::Mat& left, cv::Mat& right, cv::Mat& disparity);                                          :804
//     void get_initial_disparity(cv::Mat& initial_guess, cv::Mat& disparity);                                      :846
//     void retrieve_optimized_depth(cv::Mat& disparity, cv::Mat& depth);                                            :863
//     void evaluate_performance / evaluate_performances                      main.cpp:16, main_lc.cpp:85, main_sl.cpp:1031
//
// and, beyond the reference, dcmt::evaluate_kitti: the KITTI depth-completion benchmark's figures of a result, and
// dcmt::interpolate_with_superpixels_bgr[_to_u16]: main_lc.cpp's cvtColor + generate_superpixels + interpolate_with_superpixels
// in one call from the BGR frame.
//
// The stereo functions take the reference's own containers: EntryType matrices (struct { float value;
// Eigen::Vector2f derivative; }, main_sl.cpp:23-26) stored as cv::Mat(rows, cols, CV_32FC(sizeof(EntryType))) (:1165).
// EntryType itself stays the caller's (main_sl.cpp defines it); this header only relies on its 12-byte layout.
//
// Without OpenCV (this repository's CI) the same functions exist on dcmt::MatView, a plain {rows, cols, step, data}
// view with cv::Mat's memory layout, so the shim can be compiled and tested anywhere.  Errors of the C ABI become
// std::runtime_error (the reference functions return void).
#ifndef DCMT_IMG_COMPLETION_H_
#define DCMT_IMG_COMPLETION_H_

#include <cstdint>
#include <cstring>
#include <stdexcept>
#include <string>
#include <vector>

#include "dcmt.h"

#if !defined(DCMT_NO_OPENCV) && defined(__has_include)
#if __has_include(<opencv2/core.hpp>)
#include <opencv2/core.hpp>
#define DCMT_HAVE_OPENCV 1
#endif
#endif

namespace dcmt {

// cv::Mat-compatible view of an image: element (r, c) lives at data + r * step + c * sizeof(T)
struct MatView {
    int rows = 0, cols = 0;
    size_t step = 0;  // bytes between rows (cv::Mat::step)
    void* data = nullptr;
};

// bytes of one EntryType (main_sl.cpp:23-26): float value + Eigen::Vector2f derivative
constexpr size_t kEntryBytes = 12;

inline void check(int status) {
    if (status != DCMT_OK) throw std::runtime_error(std::string("dcmt: ") + dcmt_status_string(status) + ": " + dcmt_last_error());
}

// blur_type semantics of img_completion.cpp:172-189
inline int blur_code(const std::string& blur_type) {
    return blur_type == "bilateral" ? DCMT_BLUR_BILATERAL : blur_type == "gaussian" ? DCMT_BLUR_GAUSSIAN : DCMT_BLUR_NONE;
}

inline void need_same_layout(const MatView& a, const MatView& b, const char* what) {
    if (a.rows != b.rows || a.cols != b.cols || !a.data || !b.data) throw std::invalid_argument(std::string("dcmt: ") + what + ": views must be allocated with one shape");
    // the completion ABI takes ONE pitch for input and output (dcmt_img_completion_f32): views with different steps would
    // be written with the wrong row pitch.  The cv::Mat overloads below always pass continuous matrices.
    if (a.step != b.step) throw std::invalid_argument(std::string("dcmt: ") + what + ": input and output views must share one step");
}

// img_completion.cpp:17-204.  `dense` must describe a rows x cols float buffer with the step of `sparse` (the cv::Mat
// overload allocates it, like the reference's clone()).  `extr` is ignored, as in the reference (:103).
inline void img_completion(const MatView& sparse, MatView& dense, const bool& /*extr*/, const std::string& blur_type,
                           int path = DCMT_PATH_AUTO) {
    need_same_layout(sparse, dense, "img_completion");
    check(dcmt_img_completion_f32_host(static_cast<const float*>(sparse.data), static_cast<float*>(dense.data), sparse.rows,
                                       sparse.cols, sparse.step, 0, 1, blur_code(blur_type), path, nullptr));
}

// main.cpp:75-93 in one call: the uint16 payload of a KITTI depth PNG (CV_16UC1 view, metres * 256) -> dense float32 metres;
// stands for image_r.convertTo(projected_depths, CV_32F, 1.0 / 256.0) (:79) followed by img_completion (:93).  Input and
// output have their own steps here.
inline void img_completion_u16(const MatView& sparse_u16, MatView& dense, const std::string& blur_type, int path = DCMT_PATH_AUTO) {
    if (dense.rows != sparse_u16.rows || dense.cols != sparse_u16.cols || !dense.data) throw std::invalid_argument("dcmt: dense view not allocated");
    check(dcmt_img_completion_u16_host(static_cast<const uint16_t*>(sparse_u16.data), static_cast<float*>(dense.data), sparse_u16.rows,
                                       sparse_u16.cols, sparse_u16.step, 0, dense.step, 0, 1, blur_code(blur_type), path, nullptr));
}

// main.cpp:75-93 followed by the caller's convertTo(png, CV_16U, 256) in front of cv::imwrite: KITTI uint16 in, KITTI uint16
// out (metres * 256, rounded half to even; dcmt_img_completion_u16_u16).  Input and output have their own steps.
inline void img_completion_u16_u16(const MatView& sparse_u16, MatView& dense_u16, const std::string& blur_type, int path = DCMT_PATH_AUTO) {
    if (dense_u16.rows != sparse_u16.rows || dense_u16.cols != sparse_u16.cols || !dense_u16.data) throw std::invalid_argument("dcmt: dense view not allocated");
    check(dcmt_img_completion_u16_u16_host(static_cast<const uint16_t*>(sparse_u16.data), static_cast<uint16_t*>(dense_u16.data),
                                           sparse_u16.rows, sparse_u16.cols, sparse_u16.step, 0, dense_u16.step, 0, 1, blur_code(blur_type),
                                           path, nullptr));
}

// The evaluation loops of the three programs (SURVEY.md 8f #3); GT and result must share one step.
inline dcmt_eval_result evaluate(const MatView& GT_img, const MatView& r_img, float tolerance, int mode) {
    if (GT_img.rows != r_img.rows || GT_img.cols != r_img.cols || GT_img.step != r_img.step) throw std::invalid_argument("dcmt: evaluate needs same-shaped Mats");
    dcmt_eval_result res;
    check(dcmt_evaluate_f32_host(static_cast<const float*>(GT_img.data), static_cast<const float*>(r_img.data), GT_img.rows, GT_img.cols,
                                 GT_img.step, 0, 1, tolerance, mode, &res));
    return res;
}
// The same on KITTI ground truth as read: the uint16 payload of the depth PNG (CV_16UC1 view, metres * 256), which stands for
// the GT's convertTo(CV_32F, 1.0 / 256.0) of main.cpp:82 / main_lc.cpp:159-224 (dcmt_evaluate_u16), scored against a float32
// result, or against a KITTI uint16 result such as img_completion_u16_u16's (dcmt_evaluate_u16_u16).  GT and result have
// their own steps here.  The records equal evaluate() on the decoded views (u / 256) when those have the same steps in
// elements.
inline dcmt_eval_result evaluate_u16(const MatView& GT_u16, const MatView& r_img, float tolerance, int mode) {
    if (GT_u16.rows != r_img.rows || GT_u16.cols != r_img.cols) throw std::invalid_argument("dcmt: evaluate_u16 needs same-shaped Mats");
    dcmt_eval_result res;
    check(dcmt_evaluate_u16_host(static_cast<const uint16_t*>(GT_u16.data), static_cast<const float*>(r_img.data), GT_u16.rows, GT_u16.cols,
                                 GT_u16.step, 0, r_img.step, 0, 1, tolerance, mode, &res));
    return res;
}
inline dcmt_eval_result evaluate_u16_u16(const MatView& GT_u16, const MatView& r_u16, float tolerance, int mode) {
    if (GT_u16.rows != r_u16.rows || GT_u16.cols != r_u16.cols) throw std::invalid_argument("dcmt: evaluate_u16_u16 needs same-shaped Mats");
    dcmt_eval_result res;
    check(dcmt_evaluate_u16_u16_host(static_cast<const uint16_t*>(GT_u16.data), static_cast<const uint16_t*>(r_u16.data), GT_u16.rows,
                                     GT_u16.cols, GT_u16.step, 0, r_u16.step, 0, 1, tolerance, mode, &res));
    return res;
}
// The KITTI depth-completion benchmark's figures for one frame (dcmt_evaluate_kitti_*; include/dcmt.h states the rule,
// a restatement of the devkit's background interpolation and error loop): MAE / RMSE in mm, iMAE / iRMSE in 1/km and
// density, with the sums behind them.  A float32 pair (evaluate_kitti), or the KITTI GT as read (CV_16UC1 view, metres *
// 256) with a float32 or a KITTI uint16 prediction.  Each view has its own step.
inline dcmt_kitti_metrics evaluate_kitti(const MatView& gt, const MatView& pred) {
    if (gt.rows != pred.rows || gt.cols != pred.cols) throw std::invalid_argument("dcmt: evaluate_kitti needs same-shaped Mats");
    dcmt_kitti_metrics res;
    check(dcmt_evaluate_kitti_f32_host(static_cast<const float*>(gt.data), static_cast<const float*>(pred.data), gt.rows, gt.cols, gt.step, 0,
                                       pred.step, 0, 1, &res));
    return res;
}
inline dcmt_kitti_metrics evaluate_kitti_u16(const MatView& gt_u16, const MatView& pred) {
    if (gt_u16.rows != pred.rows || gt_u16.cols != pred.cols) throw std::invalid_argument("dcmt: evaluate_kitti_u16 needs same-shaped Mats");
    dcmt_kitti_metrics res;
    check(dcmt_evaluate_kitti_u16_host(static_cast<const uint16_t*>(gt_u16.data), static_cast<const float*>(pred.data), gt_u16.rows,
                                       gt_u16.cols, gt_u16.step, 0, pred.step, 0, 1, &res));
    return res;
}
inline dcmt_kitti_metrics evaluate_kitti_u16_u16(const MatView& gt_u16, const MatView& pred_u16) {
    if (gt_u16.rows != pred_u16.rows || gt_u16.cols != pred_u16.cols)
        throw std::invalid_argument("dcmt: evaluate_kitti_u16_u16 needs same-shaped Mats");
    dcmt_kitti_metrics res;
    check(dcmt_evaluate_kitti_u16_u16_host(static_cast<const uint16_t*>(gt_u16.data), static_cast<const uint16_t*>(pred_u16.data),
                                           gt_u16.rows, gt_u16.cols, gt_u16.step, 0, pred_u16.step, 0, 1, &res));
    return res;
}
// src/DC_lidar_only/main.cpp:16-34: "mse" = mean of (gt - r) over gt > 0 (a signed mean, sic)
inline void evaluate_performance(const MatView& GT_img, const MatView& r_img, float& mse) {
    mse = evaluate(GT_img, r_img, 0.0f, DCMT_EVAL_GT_VALID).mean_err;
}
// src/DC_lidar_camera/main_lc.cpp:85-116: `int tolerance = 0.1` is 0; "mse" = sqrt(sum d^2 / count) (sic), mae
inline void evaluate_performance(const MatView& GT_img, const MatView& r_img, float& mse, float& mae) {
    const dcmt_eval_result r = evaluate(GT_img, r_img, 0.0f, DCMT_EVAL_BOTH_VALID);
    mse = r.rmse;
    mae = r.mae;
}
// src/DC_stereo_lidar/main_sl.cpp:1031-1061: tolerance 2
inline void evaluate_performances(const MatView& GT_img, const MatView& r_img, float& mae, float& rmse) {
    const dcmt_eval_result r = evaluate(GT_img, r_img, 2.0f, DCMT_EVAL_BOTH_VALID);
    mae = r.mae;
    rmse = r.rmse;
}

// main_sl.cpp:478-523: the Velodyne .bin payload (n_points x 4 floats) -> projected_depths and its cv::normalize(0, 80).
// T (4x4) and P (3x4) are row-major here; from Eigen pass `Eigen::Matrix<float, 4, 4, Eigen::RowMajor>(T).data()`.
inline int project_lidar(const float* points, int n_points, const float* T_row_major, const float* P_row_major, MatView& projected_depths,
                         MatView& normalized_depths, float norm_a = 0.0f, float norm_b = 80.0f) {
    const int rows = projected_depths.rows, cols = projected_depths.cols;
    if (normalized_depths.rows != rows || normalized_depths.cols != cols || projected_depths.step != (size_t)cols * 4 ||
        normalized_depths.step != (size_t)cols * 4)
        throw std::invalid_argument("dcmt: project_lidar needs continuous same-shaped Mats");
    int32_t n = 0;
    check(dcmt_lidar_project_f32_host(points, n_points, T_row_major, P_row_major, rows, cols, static_cast<float*>(projected_depths.data),
                                      static_cast<float*>(normalized_depths.data), norm_a, norm_b, &n));
    return n;
}

// img_completion_lc.cpp:34-203.  `clusters_col_major` is Slic::clusters, indexed [col][row] (:83); it is transposed
// into the row-major int32 label map of the ABI here.  `n_centers` is slic.centers.size().
inline std::vector<int32_t> row_major_labels(const std::vector<std::vector<int>>& clusters_col_major, int rows, int cols) {
    if (clusters_col_major.size() < (size_t)cols) throw std::invalid_argument("dcmt: Slic::clusters has fewer columns than the image");
    std::vector<int32_t> labels((size_t)rows * cols);
    for (int j = 0; j < cols; ++j) {
        if (clusters_col_major[j].size() < (size_t)rows) throw std::invalid_argument("dcmt: Slic::clusters has fewer rows than the image");
        for (int i = 0; i < rows; ++i) labels[(size_t)i * cols + j] = clusters_col_major[j][i];
    }
    return labels;
}

inline void interpolate_with_superpixels(const std::vector<std::vector<int>>& clusters_col_major, size_t n_centers,
                                         const MatView& sparse, MatView& dense, const std::string& /*blur_type*/,
                                         int use_superpixel) {
    need_same_layout(sparse, dense, "interpolate_with_superpixels");
    std::vector<int32_t> labels;
    if (use_superpixel) labels = row_major_labels(clusters_col_major, sparse.rows, sparse.cols);
    check(dcmt_interpolate_with_superpixels_f32_host(static_cast<const float*>(sparse.data), use_superpixel ? labels.data() : nullptr,
                                                     (int)n_centers, static_cast<float*>(dense.data), sparse.rows, sparse.cols,
                                                     sparse.step, 0, 1, use_superpixel, nullptr));
}

// main_lc.cpp:159-180 + :220 in one call: the uint16 payload of the KITTI depth PNG (CV_16UC1 view, metres * 256) -> dense
// float32 metres (interpolate_with_superpixels_u16) or KITTI uint16 (..._u16_u16, the convertTo(CV_16U, 256) of a caller that
// writes the PNG).  Input and output have their own steps.
inline void interpolate_with_superpixels_u16(const std::vector<std::vector<int>>& clusters_col_major, size_t n_centers,
                                             const MatView& sparse_u16, MatView& dense, int use_superpixel, int path = DCMT_PATH_AUTO) {
    if (dense.rows != sparse_u16.rows || dense.cols != sparse_u16.cols || !dense.data) throw std::invalid_argument("dcmt: dense view not allocated");
    std::vector<int32_t> labels;
    if (use_superpixel) labels = row_major_labels(clusters_col_major, sparse_u16.rows, sparse_u16.cols);
    check(dcmt_interpolate_with_superpixels_u16_host(static_cast<const uint16_t*>(sparse_u16.data), use_superpixel ? labels.data() : nullptr,
                                                     (int)n_centers, static_cast<float*>(dense.data), sparse_u16.rows, sparse_u16.cols,
                                                     sparse_u16.step, 0, dense.step, 0, 1, use_superpixel, path, nullptr));
}

inline void interpolate_with_superpixels_u16_u16(const std::vector<std::vector<int>>& clusters_col_major, size_t n_centers,
                                                 const MatView& sparse_u16, MatView& dense_u16, int use_superpixel,
                                                 int path = DCMT_PATH_AUTO) {
    if (dense_u16.rows != sparse_u16.rows || dense_u16.cols != sparse_u16.cols || !dense_u16.data) throw std::invalid_argument("dcmt: dense view not allocated");
    std::vector<int32_t> labels;
    if (use_superpixel) labels = row_major_labels(clusters_col_major, sparse_u16.rows, sparse_u16.cols);
    check(dcmt_interpolate_with_superpixels_u16_u16_host(static_cast<const uint16_t*>(sparse_u16.data),
                                                         use_superpixel ? labels.data() : nullptr, (int)n_centers,
                                                         static_cast<uint16_t*>(dense_u16.data), sparse_u16.rows, sparse_u16.cols,
                                                         sparse_u16.step, 0, dense_u16.step, 0, 1, use_superpixel, path, nullptr));
}

// main_lc.cpp:182-220 in one call: the BGR frame as read (CV_8UC3 view) and the uint16 payload of the KITTI depth PNG
// (CV_16UC1 view) -> dense float32 metres (interpolate_with_superpixels_bgr) or KITTI uint16 (..._bgr_to_u16): the
// cvtColor(COLOR_BGR2Lab), Slic::generate_superpixels(lab, step, nc) and interpolate_with_superpixels of the reference
// with the Lab image and the labels kept on the device (dcmt_interpolate_with_superpixels_bgr_u16[_u16]_host).  `step` is
// the reference's int parameter (main_lc.cpp:197-201 passes a double, truncated).  Every view has its own step.
inline void interpolate_with_superpixels_bgr(const MatView& bgr, const MatView& sparse_u16, MatView& dense, int step, int nc,
                                             int use_superpixel = 1, int path = DCMT_PATH_AUTO) {
    if (bgr.rows != sparse_u16.rows || bgr.cols != sparse_u16.cols || dense.rows != sparse_u16.rows || dense.cols != sparse_u16.cols || !dense.data)
        throw std::invalid_argument("dcmt: interpolate_with_superpixels_bgr needs same-shaped, allocated views");
    check(dcmt_interpolate_with_superpixels_bgr_u16_host(static_cast<const uint8_t*>(bgr.data), bgr.step, 0,
                                                         static_cast<const uint16_t*>(sparse_u16.data), static_cast<float*>(dense.data),
                                                         sparse_u16.rows, sparse_u16.cols, sparse_u16.step, 0, dense.step, 0, 1, step, nc,
                                                         10, use_superpixel, path, nullptr));
}

inline void interpolate_with_superpixels_bgr_to_u16(const MatView& bgr, const MatView& sparse_u16, MatView& dense_u16, int step, int nc,
                                                    int use_superpixel = 1, int path = DCMT_PATH_AUTO) {
    if (bgr.rows != sparse_u16.rows || bgr.cols != sparse_u16.cols || dense_u16.rows != sparse_u16.rows || dense_u16.cols != sparse_u16.cols ||
        !dense_u16.data)
        throw std::invalid_argument("dcmt: interpolate_with_superpixels_bgr_to_u16 needs same-shaped, allocated views");
    check(dcmt_interpolate_with_superpixels_bgr_u16_u16_host(static_cast<const uint8_t*>(bgr.data), bgr.step, 0,
                                                             static_cast<const uint16_t*>(sparse_u16.data),
                                                             static_cast<uint16_t*>(dense_u16.data), sparse_u16.rows, sparse_u16.cols,
                                                             sparse_u16.step, 0, dense_u16.step, 0, 1, step, nc, 10, use_superpixel, path,
                                                             nullptr));
}

// ---- the stereo functions on EntryType matrices (views whose rows hold `cols` entries of kEntryBytes at the start) ----
// main_sl.cpp:715-745
inline void calculateMeasuementDerivatives(MatView& entries) {
    check(dcmt_entries_measurement_derivatives_host(entries.data, entries.rows, entries.cols, entries.step, kEntryBytes));
}
// main_sl.cpp:846-861 (in place: pixels with depth <= 0 keep what `disparity_IG` held)
inline void get_initial_disparity(const MatView& initial_guess, MatView& disparity_IG, float baseline = 0.54f, float focal = 9.597910e+02f) {
    if (initial_guess.rows != disparity_IG.rows || initial_guess.cols != disparity_IG.cols) throw std::invalid_argument("dcmt: get_initial_disparity needs same-shaped Mats");
    check(dcmt_get_initial_disparity_mat_f32_host(static_cast<const float*>(initial_guess.data), initial_guess.step,
                                                  static_cast<float*>(disparity_IG.data), disparity_IG.step, disparity_IG.rows,
                                                  disparity_IG.cols, baseline, focal));
}
// main_sl.cpp:804-843 (main_sl_OFFICIAL.cpp:832-876: num_iterations from the caller, damp 1370, clip 221)
inline void optimize_IG(const MatView& entries_left, const MatView& entries_right, MatView& disparity_map_IG, int num_iterations = 4,
                        float damp_factor = 500.0f, float err_clip = 255.0f) {
    if (entries_left.rows != entries_right.rows || entries_left.cols != entries_right.cols || entries_left.rows != disparity_map_IG.rows ||
        entries_left.cols != disparity_map_IG.cols)
        throw std::invalid_argument("dcmt: optimize_IG needs same-shaped Mats");
    check(dcmt_entries_optimize_ig_host(entries_left.data, entries_left.step, entries_right.data, entries_right.step, kEntryBytes,
                                        static_cast<float*>(disparity_map_IG.data), disparity_map_IG.step, disparity_map_IG.rows,
                                        disparity_map_IG.cols, num_iterations, damp_factor, err_clip));
}
// main_sl.cpp:863-885 (in place: pixels with disparity <= 0 keep what `optimized_depth` held; OFFICIAL clips at 80)
inline void retrieve_optimized_depth(const MatView& disparity_refined, MatView& optimized_depth, float depth_clip = 100.0f,
                                     float baseline = 0.54f, float focal = 9.597910e+02f) {
    if (disparity_refined.rows != optimized_depth.rows || disparity_refined.cols != optimized_depth.cols) throw std::invalid_argument("dcmt: retrieve_optimized_depth needs same-shaped Mats");
    check(dcmt_retrieve_optimized_depth_mat_f32_host(static_cast<const float*>(disparity_refined.data), disparity_refined.step,
                                                     static_cast<float*>(optimized_depth.data), optimized_depth.step, optimized_depth.rows,
                                                     optimized_depth.cols, baseline, focal, depth_clip));
}
// main_sl.cpp:747-801: one bilinear sample of an EntryType matrix at (row r, column c) = (img_point[0], img_point[1]).
// This is the per-sample accessor optimize_IG calls once per pixel and iteration in the reference; the library runs it
// inside its optimize_IG kernel, and callers that probe single points get this host-side sampler of their own (host)
// matrix.  Same arithmetic in the same order; entries the reference reads at index == rows / == cols (undefined
// behaviour there: its bounds tests use `>`) read as 0 here, like in the kernels.
inline bool sample_entries(const MatView& target, float r, float c, float& value, float& dx, float& dy) {
    const int rows = target.rows, cols = target.cols;
    const int r0 = (int)(r + 0.5), c0 = (int)(c + 0.5);
    if (r0 < 0 || r0 > rows || c0 < 0 || c0 > cols) return false;
    const int r1 = r0 + 1, c1 = c0 + 1;
    if (r1 < 0 || r1 > rows || c1 < 0 || c1 > cols) return false;
    auto entry = [&](int rr, int cc, int k) -> float {
        if (rr >= rows || cc >= cols) return 0.0f;
        float v;
        std::memcpy(&v, static_cast<const char*>(target.data) + (size_t)rr * target.step + (size_t)cc * kEntryBytes + 4 * (size_t)k, 4);
        return v;
    };
    const float dr = r - (float)r0, dc = c - (float)c0;
    const float dr1 = (float)(1. - dr), dc1 = (float)(1. - dc);
    float out[3];
    for (int k = 0; k < 3; ++k)
        out[k] = (entry(r0, c0, k) * dc1 + entry(r0, c1, k) * dc) * dr1 + (entry(r1, c0, k) * dc1 + entry(r1, c1, k) * dc) * dr;
    value = out[0];
    dx = out[1];
    dy = out[2];
    return true;
}

// cv::cvtColor(img, gray, cv::COLOR_BGR2GRAY) (main_sl.cpp:1167,1171) on CV_8UC3 / CV_8UC1 views
inline void bgr2gray(const MatView& bgr, MatView& gray) {
    if (bgr.rows != gray.rows || bgr.cols != gray.cols || !bgr.data || !gray.data) throw std::invalid_argument("dcmt: bgr2gray needs same-shaped Mats");
    check(dcmt_bgr2gray_u8_host(static_cast<const uint8_t*>(bgr.data), static_cast<uint8_t*>(gray.data), bgr.rows, bgr.cols, bgr.step, gray.step, 1));
}

// cv::cvtColor(img, lab, cv::COLOR_BGR2Lab) (main_lc.cpp:182-183, main_sl.cpp:438) on CV_8UC3 views: OpenCV's 8-bit
// conversion, the input of Slic::generate_superpixels (dcmt_slic_bgr_u8c3_host does both in one call)
inline void bgr2lab(const MatView& bgr, MatView& lab) {
    if (bgr.rows != lab.rows || bgr.cols != lab.cols || !bgr.data || !lab.data) throw std::invalid_argument("dcmt: bgr2lab needs same-shaped Mats");
    check(dcmt_bgr2lab_u8_host(static_cast<const uint8_t*>(bgr.data), static_cast<uint8_t*>(lab.data), bgr.rows, bgr.cols, bgr.step, lab.step, 1));
}

// main_sl.cpp:1165-1253 in one call: gray images (CV_8UC1 views) + initial dense depth -> refined depth
inline void stereo_refine(const MatView& depth_ig, const MatView& left_gray, const MatView& right_gray, MatView& depth_out,
                          const dcmt_stereo_params* params = nullptr) {
    dcmt_stereo_params p;
    if (params) p = *params;
    else dcmt_stereo_params_default(&p);
    const int rows = depth_ig.rows, cols = depth_ig.cols;
    if (depth_ig.step != (size_t)cols * 4 || depth_out.step != (size_t)cols * 4 || left_gray.step != (size_t)cols ||
        right_gray.step != (size_t)cols)
        throw std::invalid_argument("dcmt: stereo_refine needs continuous Mats");
    check(dcmt_stereo_refine_f32_host(static_cast<const float*>(depth_ig.data), static_cast<const uint8_t*>(left_gray.data),
                                      static_cast<const uint8_t*>(right_gray.data), static_cast<float*>(depth_out.data), nullptr, rows,
                                      cols, 1, &p));
}

// withSuperPixels (main_sl.cpp:435-563) and :1162-1253 in one call (dcmt_stereo_chain_f32_host): one Velodyne cloud (the .bin
// payload, n_points x 4 floats) and the BGR stereo pair as read (CV_8UC3 views with one step) -> the refined depth and,
// optionally, the disparity (continuous CV_32FC1 views).  cv::normalize(0, 80), SLIC with `step` (the reference's int) and
// `nc`, interpolate_with_superpixels, cvtColor(BGR2GRAY) of both images and the refinement run on the device.  T (4x4) and
// P (3x4) are row-major, as for project_lidar: from Eigen pass `Eigen::Matrix<float, 4, 4, Eigen::RowMajor>(T).data()`.
// `params` defaults to the main_sl.cpp literals (dcmt_stereo_params_default).
inline void stereo_chain(const float* points, int n_points, const float* T_row_major, const float* P_row_major, const MatView& left_bgr,
                         const MatView& right_bgr, MatView& depth, int step, int nc = 40, MatView* disparity = nullptr,
                         const dcmt_stereo_params* params = nullptr, int use_superpixel = 1, int path = DCMT_PATH_AUTO) {
    const int rows = left_bgr.rows, cols = left_bgr.cols;
    if (right_bgr.rows != rows || right_bgr.cols != cols || depth.rows != rows || depth.cols != cols || !depth.data ||
        (disparity && (disparity->rows != rows || disparity->cols != cols || !disparity->data)))
        throw std::invalid_argument("dcmt: stereo_chain needs same-shaped, allocated views");
    if (left_bgr.step != right_bgr.step) throw std::invalid_argument("dcmt: stereo_chain needs left and right images with one step");
    if (depth.step != (size_t)cols * 4 || (disparity && disparity->step != (size_t)cols * 4))
        throw std::invalid_argument("dcmt: stereo_chain needs continuous depth and disparity views");
    dcmt_stereo_params p;
    if (params) p = *params;
    else dcmt_stereo_params_default(&p);
    check(dcmt_stereo_chain_f32_host(points, nullptr, n_points, (size_t)n_points, T_row_major, P_row_major, 0.0f, 80.0f,
                                     static_cast<const uint8_t*>(left_bgr.data), static_cast<const uint8_t*>(right_bgr.data), left_bgr.step, 0,
                                     static_cast<float*>(depth.data), disparity ? static_cast<float*>(disparity->data) : nullptr, rows, cols, 1,
                                     step, nc, 10, use_superpixel, path, &p, nullptr));
}

}  // namespace dcmt

#ifdef DCMT_HAVE_OPENCV
// ---- the reference's own signatures -------------------------------------------------------------------------

namespace dcmt {
inline MatView view_of(const cv::Mat& m) { return MatView{m.rows, m.cols, (size_t)m.step, m.data}; }
inline cv::Mat continuous(const cv::Mat& m) { return m.isContinuous() ? m : m.clone(); }
}  // namespace dcmt

// img_completion.cpp:17-20.  The reference replaces the header of `dense_r_img` by a fresh matrix (`= sparse.clone()`,
// :27); so does this: the result is computed into a new continuous Mat and assigned, whatever `dense_r_img` was (an
// ROI, a non-continuous or differently typed matrix).  A CV_16UC1 input (the KITTI PNG as read by
// cv::imread(..., IMREAD_ANYDEPTH), main.cpp:75) is accepted as well and stands for convertTo(CV_32F, 1.0 / 256.0) +
// img_completion.
inline void img_completion(const cv::Mat& sparse_r_img, cv::Mat& dense_r_img, const bool& extr, const std::string& blur_type) {
    cv::Mat out(sparse_r_img.rows, sparse_r_img.cols, CV_32FC1);
    dcmt::MatView d = dcmt::view_of(out);
    if (sparse_r_img.type() == CV_16UC1) {
        dcmt::img_completion_u16(dcmt::view_of(sparse_r_img), d, blur_type);
    } else {
        CV_Assert(sparse_r_img.type() == CV_32FC1);
        const cv::Mat in = dcmt::continuous(sparse_r_img);
        dcmt::img_completion(dcmt::view_of(in), d, extr, blur_type);
    }
    dense_r_img = out;
}

// img_completion_lc.cpp:34-38.  Slic is the reference's class (slic.h:30-71): public `clusters` ([col][row]) and `centers`.
// A CV_16UC1 input (the KITTI PNG as main_lc.cpp reads it) stands for its convertTo(CV_32F, 1.0 / 256.0) as well.
template <class SlicT>
inline void interpolate_with_superpixels(SlicT& slic, const cv::Mat& sparse_r_img, cv::Mat& dense_r_img, const std::string& blur_type,
                                         int use_superpixel) {
    cv::Mat out(sparse_r_img.rows, sparse_r_img.cols, CV_32FC1);
    dcmt::MatView d = dcmt::view_of(out);
    if (sparse_r_img.type() == CV_16UC1) {
        dcmt::interpolate_with_superpixels_u16(slic.clusters, slic.centers.size(), dcmt::view_of(sparse_r_img), d, use_superpixel);
    } else {
        CV_Assert(sparse_r_img.type() == CV_32FC1);
        const cv::Mat in = dcmt::continuous(sparse_r_img);
        dcmt::interpolate_with_superpixels(slic.clusters, slic.centers.size(), dcmt::view_of(in), d, blur_type, use_superpixel);
    }
    dense_r_img = out;
}

namespace dcmt {
// KITTI PNG in, KITTI PNG payload out: img_completion on a CV_16UC1 matrix (metres * 256) whose result comes back as a fresh
// continuous CV_16UC1 matrix -- what dense.convertTo(png, CV_16U, 256) in front of cv::imwrite gives, with half the
// device-to-host copy.
inline void img_completion_to_u16(const cv::Mat& sparse_u16, cv::Mat& dense_u16, const std::string& blur_type) {
    CV_Assert(sparse_u16.type() == CV_16UC1);
    cv::Mat out(sparse_u16.rows, sparse_u16.cols, CV_16UC1);
    MatView d = view_of(out);
    img_completion_u16_u16(view_of(sparse_u16), d, blur_type);
    dense_u16 = out;
}

// the same for interpolate_with_superpixels (main_lc.cpp:159-220)
template <class SlicT>
inline void interpolate_with_superpixels_to_u16(SlicT& slic, const cv::Mat& sparse_u16, cv::Mat& dense_u16, int use_superpixel) {
    CV_Assert(sparse_u16.type() == CV_16UC1);
    cv::Mat out(sparse_u16.rows, sparse_u16.cols, CV_16UC1);
    MatView d = view_of(out);
    interpolate_with_superpixels_u16_u16(slic.clusters, slic.centers.size(), view_of(sparse_u16), d, use_superpixel);
    dense_u16 = out;
}

// main_lc.cpp:182-220 in one call on the Mats as read: a CV_8UC3 BGR image (an ROI too) and a CV_16UC1 depth PNG payload;
// the result is a fresh continuous CV_32FC1 (metres) or CV_16UC1 (KITTI uint16) matrix.  Any other type throws.
inline void interpolate_with_superpixels_bgr(const cv::Mat& bgr, const cv::Mat& sparse_u16, cv::Mat& dense, int step, int nc,
                                             int use_superpixel = 1) {
    CV_Assert(bgr.type() == CV_8UC3 && sparse_u16.type() == CV_16UC1);
    cv::Mat out(sparse_u16.rows, sparse_u16.cols, CV_32FC1);
    MatView d = view_of(out);
    interpolate_with_superpixels_bgr(view_of(bgr), view_of(sparse_u16), d, step, nc, use_superpixel);
    dense = out;
}

inline void interpolate_with_superpixels_bgr_to_u16(const cv::Mat& bgr, const cv::Mat& sparse_u16, cv::Mat& dense_u16, int step, int nc,
                                                    int use_superpixel = 1) {
    CV_Assert(bgr.type() == CV_8UC3 && sparse_u16.type() == CV_16UC1);
    cv::Mat out(sparse_u16.rows, sparse_u16.cols, CV_16UC1);
    MatView d = view_of(out);
    interpolate_with_superpixels_bgr_to_u16(view_of(bgr), view_of(sparse_u16), d, step, nc, use_superpixel);
    dense_u16 = out;
}

// withSuperPixels + main_sl.cpp:1162-1253 on the Mats as read: CV_8UC3 left and right images (ROIs too) with equal steps; the
// depth and the disparity (when asked for) come back as fresh continuous CV_32FC1 matrices.  Other types or steps throw.
inline void stereo_chain(const float* points, int n_points, const float* T_row_major, const float* P_row_major, const cv::Mat& left_bgr,
                         const cv::Mat& right_bgr, cv::Mat& depth, int step, int nc = 40, cv::Mat* disparity = nullptr,
                         const dcmt_stereo_params* params = nullptr, int use_superpixel = 1) {
    CV_Assert(left_bgr.type() == CV_8UC3 && right_bgr.type() == CV_8UC3 && view_of(left_bgr).step == view_of(right_bgr).step);
    cv::Mat out(left_bgr.rows, left_bgr.cols, CV_32FC1), disp;
    if (disparity) disp.create(left_bgr.rows, left_bgr.cols, CV_32FC1);
    MatView d = view_of(out), v = view_of(disp);
    stereo_chain(points, n_points, T_row_major, P_row_major, view_of(left_bgr), view_of(right_bgr), d, step, nc, disparity ? &v : nullptr,
                 params, use_superpixel);
    depth = out;
    if (disparity) *disparity = disp;
}
}  // namespace dcmt

// main_sl.cpp:715.  `img` is an EntryType matrix: cv::Mat(rows, cols, CV_32FC(sizeof(EntryType))) (:1165, :1169)
inline void calculateMeasuementDerivatives(cv::Mat& img) {
    CV_Assert(img.elemSize() >= dcmt::kEntryBytes);
    dcmt::MatView v = dcmt::view_of(img);
    dcmt::calculateMeasuementDerivatives(v);
}
// main_sl.cpp:846
inline void get_initial_disparity(cv::Mat& initial_guess, cv::Mat& disparity_IG) {
    CV_Assert(initial_guess.type() == CV_32FC1 && disparity_IG.type() == CV_32FC1);
    dcmt::MatView d = dcmt::view_of(disparity_IG);
    dcmt::get_initial_disparity(dcmt::view_of(initial_guess), d);
}
// main_sl.cpp:804
inline void optimize_IG(cv::Mat& entryMatrix_left, cv::Mat& entryMatrix_right, cv::Mat& disparity_map_IG) {
    CV_Assert(entryMatrix_left.elemSize() >= dcmt::kEntryBytes && entryMatrix_right.elemSize() >= dcmt::kEntryBytes &&
              disparity_map_IG.type() == CV_32FC1);
    dcmt::MatView d = dcmt::view_of(disparity_map_IG);
    dcmt::optimize_IG(dcmt::view_of(entryMatrix_left), dcmt::view_of(entryMatrix_right), d);
}
// main_sl_OFFICIAL.cpp:832: the caller supplies the iteration count; damp 1370 (:836), error clip 221 (:848-855)
inline void optimize_IG(cv::Mat& entryMatrix_left, cv::Mat& entryMatrix_right, cv::Mat& disparity_map_IG, int& num_iterations) {
    dcmt::MatView d = dcmt::view_of(disparity_map_IG);
    dcmt::optimize_IG(dcmt::view_of(entryMatrix_left), dcmt::view_of(entryMatrix_right), d, num_iterations, 1370.0f, 221.0f);
}
// main_sl.cpp:863
inline void retrieve_optimized_depth(cv::Mat& disparity_refined, cv::Mat& optimized_depth) {
    CV_Assert(disparity_refined.type() == CV_32FC1 && optimized_depth.type() == CV_32FC1);
    dcmt::MatView d = dcmt::view_of(optimized_depth);
    dcmt::retrieve_optimized_depth(dcmt::view_of(disparity_refined), d);
}
// main_sl.cpp:747.  Vec2 is Eigen::Vector2f (anything with operator[] / operator() on two floats); img_point = (row, column)
template <class Vec2>
inline bool calculateObservationDerivatives(const cv::Mat& target_img, const Vec2 img_point, float& value, Vec2& derivative) {
    float dx = 0.0f, dy = 0.0f;
    if (!dcmt::sample_entries(dcmt::view_of(target_img), img_point[0], img_point[1], value, dx, dy)) return false;
    derivative[0] = dx;
    derivative[1] = dy;
    return true;
}

// main_sl.cpp:1165-1253: the sequence entry fill -> calculateMeasuementDerivatives -> get_initial_disparity ->
// optimize_IG -> retrieve_optimized_depth -> GaussianBlur in ONE fused kernel, on the caller's gray (CV_8UC1) or colour
// (CV_8UC3, BGR) images and depth Mat
inline void stereo_refine(const cv::Mat& dense_range_img, const cv::Mat& left_gray, const cv::Mat& right_gray, cv::Mat& optimized_depth,
                          const dcmt_stereo_params* params = nullptr) {
    CV_Assert(dense_range_img.type() == CV_32FC1 && left_gray.type() == right_gray.type() && (left_gray.type() == CV_8UC1 || left_gray.type() == CV_8UC3));
    const cv::Mat ig = dcmt::continuous(dense_range_img);
    cv::Mat l = dcmt::continuous(left_gray), r = dcmt::continuous(right_gray);
    if (l.type() == CV_8UC3) {  // the colour images as read: cv::cvtColor(COLOR_BGR2GRAY) (main_sl.cpp:1167,1171) on the device as well
        cv::Mat lg(l.rows, l.cols, CV_8UC1), rg(r.rows, r.cols, CV_8UC1);
        dcmt::MatView vlg = dcmt::view_of(lg), vrg = dcmt::view_of(rg);
        dcmt::bgr2gray(dcmt::view_of(l), vlg);
        dcmt::bgr2gray(dcmt::view_of(r), vrg);
        l = lg;
        r = rg;
    }
    cv::Mat out(ig.rows, ig.cols, CV_32FC1);
    dcmt::MatView vo = dcmt::view_of(out);
    dcmt::stereo_refine(dcmt::view_of(ig), dcmt::view_of(l), dcmt::view_of(r), vo, params);
    optimized_depth = out;
}

namespace dcmt {
// GT and result Mats as the three programs hold them: a CV_32FC1 pair, or the KITTI GT as read (CV_16UC1, no convertTo) with a
// CV_32FC1 or CV_16UC1 result.  A float32 GT with a uint16 result, and every other combination, throws.
inline dcmt_eval_result evaluate_mats(const cv::Mat& GT_img, const cv::Mat& r_img, float tolerance, int mode) {
    if (GT_img.type() == CV_16UC1 && r_img.type() == CV_16UC1) return evaluate_u16_u16(view_of(GT_img), view_of(r_img), tolerance, mode);
    if (GT_img.type() == CV_16UC1 && r_img.type() == CV_32FC1) return evaluate_u16(view_of(GT_img), view_of(r_img), tolerance, mode);
    CV_Assert(GT_img.type() == CV_32FC1 && r_img.type() == CV_32FC1);
    const cv::Mat g = continuous(GT_img), r = continuous(r_img);
    return evaluate(view_of(g), view_of(r), tolerance, mode);
}
// The KITTI benchmark's figures on Mats: CV_16UC1 GT with a CV_32FC1 or CV_16UC1 prediction, or a CV_32FC1 pair; any other
// pair throws.
inline dcmt_kitti_metrics evaluate_kitti(const cv::Mat& gt, const cv::Mat& pred) {
    if (gt.type() == CV_16UC1 && pred.type() == CV_16UC1) return evaluate_kitti_u16_u16(view_of(gt), view_of(pred));
    if (gt.type() == CV_16UC1 && pred.type() == CV_32FC1) return evaluate_kitti_u16(view_of(gt), view_of(pred));
    CV_Assert(gt.type() == CV_32FC1 && pred.type() == CV_32FC1);
    return evaluate_kitti(view_of(gt), view_of(pred));
}
}  // namespace dcmt

// the evaluation functions of main.cpp:16 / main_lc.cpp:85 / main_sl.cpp:1031, with the tolerances and masks of the MatView
// forms above
inline void evaluate_performance(const cv::Mat& GT_img, const cv::Mat& r_img, float& mse) {
    mse = dcmt::evaluate_mats(GT_img, r_img, 0.0f, DCMT_EVAL_GT_VALID).mean_err;
}
inline void evaluate_performance(const cv::Mat& GT_img, const cv::Mat& r_img, float& mse, float& mae) {
    const dcmt_eval_result r = dcmt::evaluate_mats(GT_img, r_img, 0.0f, DCMT_EVAL_BOTH_VALID);
    mse = r.rmse;
    mae = r.mae;
}
inline void evaluate_performances(cv::Mat& GT_img, cv::Mat& r_img, float& mae, float& rmse) {
    const dcmt_eval_result r = dcmt::evaluate_mats(GT_img, r_img, 2.0f, DCMT_EVAL_BOTH_VALID);
    mae = r.mae;
    rmse = r.rmse;
}
#endif  // DCMT_HAVE_OPENCV

#endif  // DCMT_IMG_COMPLETION_H_
