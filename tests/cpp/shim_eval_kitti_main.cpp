// Test program for dcmt::evaluate_kitti on cv::Mat (include/img_completion.h): the KITTI depth-completion benchmark's
// figures of one prediction, with the GT as cv::imread gives it (CV_16UC1, metres * 256) or converted to float32, and a
// uint16 or float32 prediction.  Compiled against the stand-in OpenCV headers of oracle/refshim and linked against
// libdcmt.so (GPU box) or the CPU emulator build of the same sources.
//
//   shim_eval_kitti_main ROWS COLS gt.u16 pred.u16
//
// Prints one line per pairing, "<pairing>: n_gt n_pred n_unfilled sum_abs sum_sq sum_iabs sum_isq mae_mm rmse_mm
// imae_per_km irmse_per_km density" (doubles with 17 digits, floats with 9), and "throws" for the float32 GT with a
// uint16 prediction.
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>

#include <opencv2/opencv.hpp>

#include "img_completion.h"
#ifndef DCMT_HAVE_OPENCV
#error "the cv::Mat half of img_completion.h was not enabled"
#endif

static bool read_u16(const char* path, cv::Mat& m) {
    FILE* f = std::fopen(path, "rb");
    if (!f) return false;
    const size_t n = (size_t)m.rows * m.cols;
    const bool ok = std::fread(m.data, sizeof(uint16_t), n, f) == n;
    std::fclose(f);
    return ok;
}

// the float32 Mat a convertTo(CV_32F, 1.0 / 256.0) gives (the stand-in headers have no convertTo)
static cv::Mat decoded(const cv::Mat& u16) {
    cv::Mat out(u16.rows, u16.cols, CV_32FC1);
    for (int r = 0; r < u16.rows; ++r)
        for (int c = 0; c < u16.cols; ++c)
            reinterpret_cast<float*>(out.data + r * out.step)[c] = (float)reinterpret_cast<const uint16_t*>(u16.data + r * u16.step)[c] / 256.0f;
    return out;
}

static void score(const char* what, const cv::Mat& gt, const cv::Mat& pred) {
    const dcmt_kitti_metrics m = dcmt::evaluate_kitti(gt, pred);
    std::printf("%s: %.17g %.17g %.17g %.17g %.17g %.17g %.17g %.9g %.9g %.9g %.9g %.9g\n", what, m.n_gt, m.n_pred, m.n_unfilled, m.sum_abs,
                m.sum_sq, m.sum_iabs, m.sum_isq, m.mae_mm, m.rmse_mm, m.imae_per_km, m.irmse_per_km, m.density);
}

int main(int argc, char** argv) {
    if (argc != 5) return 2;
    const int rows = std::atoi(argv[1]), cols = std::atoi(argv[2]);
    cv::Mat gt(rows, cols, CV_16UC1), pred(rows, cols, CV_16UC1);
    if (!read_u16(argv[3], gt) || !read_u16(argv[4], pred)) return 3;
    try {
        const cv::Mat gt_f = decoded(gt), pred_f = decoded(pred);
        score("u16 gt, u16 pred", gt, pred);
        score("u16 gt, f32 pred", gt, pred_f);
        score("f32 gt, f32 pred", gt_f, pred_f);
        try {
            dcmt::evaluate_kitti(gt_f, pred);
            std::printf("f32 gt, u16 pred: accepted\n");
        } catch (const std::exception&) {
            std::printf("f32 gt, u16 pred: throws\n");
        }
    } catch (const std::exception& e) {
        std::fprintf(stderr, "%s\n", e.what());
        return 4;
    }
    return 0;
}
