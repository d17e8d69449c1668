// Test program for the evaluation functions of include/img_completion.h on KITTI ground truth as read: the calls of
// src/DC_lidar_only/main.cpp:93-101 and src/DC_lidar_camera/main_lc.cpp:219-224, written as the reference writes them but
// with the GT left as cv::imread gives it (CV_16UC1, metres * 256) -- no convertTo.  Compiled against the stand-in OpenCV
// headers of oracle/refshim and linked against libdcmt.so (GPU box) or the CPU emulator build of the same sources.
//
//   shim_eval_u16_main ROWS COLS sparse.u16 gt.u16
//
// Prints one line per pairing, "<pairing>: mse rmse mae mae2 rmse2" (evaluate_performance with 3 and 4 arguments, then
// evaluate_performances), and "throws" for the float32 GT with a uint16 result.
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

static void score(const char* what, cv::Mat& GT_img, cv::Mat& dense_r_img) {
    float mse = 0, rmse = 0, mae = 0, mae2 = 0, rmse2 = 0;
    evaluate_performance(GT_img, dense_r_img, mse);        // main.cpp:101
    evaluate_performance(GT_img, dense_r_img, rmse, mae);  // main_lc.cpp:224
    evaluate_performances(GT_img, dense_r_img, mae2, rmse2);  // main_sl.cpp:1232
    std::printf("%s: %.9g %.9g %.9g %.9g %.9g\n", what, mse, rmse, mae, mae2, rmse2);
}

int main(int argc, char** argv) {
    if (argc != 5) return 2;
    const int rows = std::atoi(argv[1]), cols = std::atoi(argv[2]);
    cv::Mat image_r(rows, cols, CV_16UC1), GT_img(rows, cols, CV_16UC1);  // cv::imread(..., IMREAD_ANYDEPTH), main.cpp:75 / :82
    if (!read_u16(argv[3], image_r) || !read_u16(argv[4], GT_img)) return 3;
    try {
        cv::Mat dense_r_img, dense_u16;
        img_completion(image_r, dense_r_img, false, "gaussian");            // main.cpp:93, float32 result
        dcmt::img_completion_to_u16(image_r, dense_u16, "gaussian");         // the KITTI uint16 result a caller stores
        cv::Mat GT_f = decoded(GT_img), dense_u16_f = decoded(dense_u16);
        score("u16 gt, f32 result", GT_img, dense_r_img);
        score("f32 gt, f32 result", GT_f, dense_r_img);
        score("u16 gt, u16 result", GT_img, dense_u16);
        score("f32 gt, f32 of u16 result", GT_f, dense_u16_f);
        try {
            float mse = 0;
            evaluate_performance(GT_f, dense_u16, mse);
            std::printf("f32 gt, u16 result: accepted\n");
        } catch (const std::exception&) {
            std::printf("f32 gt, u16 result: throws\n");
        }
    } catch (const std::exception& e) {
        std::fprintf(stderr, "%s\n", e.what());
        return 4;
    }
    return 0;
}
