// color.cuh -- host-side interface of color.cu (device pointers).
#pragma once
#include "common.cuh"

namespace dcmt {
// cv::cvtColor(COLOR_BGR2Lab), CV_8UC3 -> CV_8UC3 (main_lc.cpp:184, main_sl.cpp:438); pitches / frame strides in bytes
cudaError_t color_bgr2lab(const uint8_t* bgr, size_t bgr_pitch, size_t bgr_fstride, uint8_t* lab, size_t lab_pitch, size_t lab_fstride,
                          int rows, int cols, int n_frames, cudaStream_t st);
}  // namespace dcmt
