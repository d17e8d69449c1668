// evaluate.cuh -- masked error reductions of the reference's evaluation functions (SURVEY.md 8f #3).
#pragma once
#include "common.cuh"

namespace dcmt {

// per-frame result, device or host memory (mirrors dcmt_eval_result in include/dcmt.h)
struct EvalResult {
    double count, sum_err, sum_abs, sum_sq;  // pixels in the mask, sum of (gt - r), of |gt - r|, of (gt - r)^2
    float mean_err, mae, rmse;               // sum_err / count, sum_abs / count, sqrt(sum_sq / count); NaN when count == 0
    int32_t pad;
};

constexpr int kEvalMaxBlocks = 128;  // partial sums per frame
size_t eval_partial_doubles(int n_frames);
// mode 0: mask = gt > tol (DC_lidar_only/main.cpp:16-34); mode 1: mask = gt > tol && r > tol (main_lc.cpp:85-116, main_sl.cpp:1031-1061).
// G / R: float (metres) or uint16_t (KITTI, metres * 256, decoded to u * 2^-8); each plane has its own pitch and frame
// stride in elements.  Instantiated for <float, float>, <uint16_t, float> and <uint16_t, uint16_t>.  Pixels go to the same
// threads in the same order whatever the types, so a uint16 call gives the bytes of the float32 call on the decoded
// planes when those have the same pitch, frame stride and base alignment counted in elements.
template <class G, class R>
cudaError_t eval_run(const G* gt, size_t gpitch, size_t gfstride, const R* r, size_t rpitch, size_t rfstride, int rows, int cols,
                     int n_frames, float tol, int mode, double* partials, EvalResult* out, cudaStream_t st);

}  // namespace dcmt
