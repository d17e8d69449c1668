// fused_q8.cuh -- host-side interface of the strict-q8 fast path (fused_q8.cu).
#pragma once
#include "common.cuh"

namespace dcmt {

// Workspace + geometry of one chunk of frames on the fused path.  Buffers are indexed by SLOT
// (position inside the chunk); the frame a slot maps to is slot (+ pointer offset applied by the caller).
struct Q8Plan {
    int rows, cols;
    int th, tw;          // tile core (tw % 8 == 0)
    int mid_pitch;       // uint16 per row of the intermediate plane (cols rounded up to 8)
    int max_frames;      // slots
    uint16_t* mid;       // max_frames * rows * mid_pitch
    uint32_t* col_first; // max_frames * mid_pitch   (row << 16 | e) of the first valid row per column
    uint32_t* col_last;  // max_frames * mid_pitch
    FrameCounters* ctr;  // max_frames
    float* w1;           // max_frames * rows * cols, fix-up scratch
    float* w2;
    long long* prof_front;  // optional debugging aid: 16 clock64() stamps per CTA of k_q8_front / k_q8_tail
    long long* prof_tail;
    // float32 frames through the dictionary of rank_f32.cu: the front reads CODES from its uint16 input, the tail decodes
    // with `lut` (max_frames x kRankMaxValid floats) and blurs in float32; counters were zeroed (and possibly flagged)
    // before the front runs
    int codes_in;
    int counters_ready;
    const float* lut;
};

// fused path applies to frames of at least this size (smaller ones use the generic pipeline)
constexpr int kQ8MinRows = 32, kQ8MinCols = 32, kQ8MaxRows = 65535;

void q8_choose_tile(int rows, int cols, int* th, int* tw);
size_t q8_front_smem(int th, int tw);
size_t q8_tail_smem(int th, int tw);
cudaError_t q8_configure();
// A1..A4 for n_frames slots: in (float32) or in16 (KITTI uint16 = metres * 256; exactly one is non-null) -> plan.mid
// (+ column keys, counters zeroed).  `validate` != 0: check strict q8-ness of every float pixel (frames that fail are
// flagged for the generic pipeline); uint16 input needs no check.  Pitches in elements of the input type.
cudaError_t q8_run_front(const Q8Plan& p, const float* in, const uint16_t* in16, size_t in_pitch, size_t in_fstride, int n_frames,
                         int validate, cudaStream_t st);
// The front of interpolate_with_superpixels (img_completion_lc.cpp:34-145) for strict-q8 input: labels are rows x cols
// int32 per frame (contiguous), values outside [0, n_clusters) mean "no superpixel"; needs n_clusters <= 65535.
size_t q8_guided_smem(int th, int tw);
cudaError_t q8_run_guided_front(const Q8Plan& p, const float* in, const uint16_t* in16, size_t in_pitch, size_t in_fstride,
                                const int32_t* labels, int n_clusters, int n_frames, int validate, int* tile_flags, cudaStream_t st);
// ints of `tile_flags` scratch the guided front needs for n_frames frames
size_t q8_guided_tile_flags(int rows, int cols, int th, int tw, int n_frames);
// uint16 -> float32 metres (main.cpp:79) into a contiguous buffer, for frames served by the generic pipeline
cudaError_t q8_convert_u16(const uint16_t* in, size_t in_pitch, size_t in_fstride, float* out, int rows, int cols, int n_frames,
                           cudaStream_t st);
// A5..A10: plan.mid -> out (float32) or -- out16 non-null, strict q8 only (plan.lut null) -- out16 (KITTI uint16, the rule of
// depth_to_u16); blur in {none, gaussian}.  Pitches in elements of the output type.
cudaError_t q8_run_tail(const Q8Plan& p, float* out, uint16_t* out16, size_t out_pitch, size_t out_fstride, int n_frames, int blur,
                        cudaStream_t st);
// float32 metres -> KITTI uint16 (cv::Mat::convertTo(CV_16U, 256.0): round half to even, clamp to [0, 65535], NaN -> 0),
// pitched and batched; pitches in elements
cudaError_t depth_to_u16(const float* in, size_t in_pitch, size_t in_fstride, uint16_t* out, size_t out_pitch, size_t out_fstride,
                         int rows, int cols, int n_frames, cudaStream_t st);
// zero the per-frame counters (what q8_run_front does itself unless plan.counters_ready)
cudaError_t q8_zero_counters(const Q8Plan& p, int n_frames, cudaStream_t st);
// counters -> stats[4*n] (optional) and flags[n] (1 = frame must be redone by the generic pipeline)
cudaError_t q8_write_stats(const Q8Plan& p, int32_t* stats, int32_t* flags, int n_frames, cudaStream_t st);
// test aid: decode a uint16 plane (inverted space) into float
cudaError_t q8_decode_plane(const uint16_t* mid, size_t mid_pitch, float* out, int rows, int cols, cudaStream_t st);

}  // namespace dcmt
