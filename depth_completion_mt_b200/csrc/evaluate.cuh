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

// per-frame figures of the KITTI depth-completion benchmark (mirrors dcmt_kitti_metrics in include/dcmt.h, which states
// the rule: the devkit's background interpolation of the prediction, then the error terms at every GT-valid pixel)
struct KittiMetrics {
    double n_gt, n_pred, n_unfilled;                // GT-valid pixels; of those, valid in the prediction; left unfilled (p = -1)
    double sum_abs, sum_sq, sum_iabs, sum_isq;      // sums of |g - p|, its square, |1/g - 1/p|, its square
    float mae_mm, rmse_mm, imae_per_km, irmse_per_km, density;  // NaN when n_gt == 0
    int32_t pad;
};

// Workspace of kitti_run: partial sums, the first / last rows holding a valid prediction (two int32 per frame), and --
// for rows too wide for the validity bits to fit in shared memory -- one bit row per block in device memory (0 words
// otherwise).
size_t kitti_partial_doubles(int n_frames);
size_t kitti_bits_words(int rows, int cols, int n_frames);
// Same block layout, pixel order and lane / warp / block reduction as eval_run, so that on a prediction with no invalid
// pixel n_gt, sum_abs and sum_sq are the bytes of eval_run's count, sum_abs and sum_sq in mode 0 with tolerance 0.
// Instantiated for <float, float>, <uint16_t, float> and <uint16_t, uint16_t>.
template <class G, class R>
cudaError_t kitti_run(const G* gt, size_t gpitch, size_t gfstride, const R* r, size_t rpitch, size_t rfstride, int rows, int cols,
                      int n_frames, double* partials, int32_t* first_last, unsigned* bits, KittiMetrics* out, cudaStream_t st);

}  // namespace dcmt
